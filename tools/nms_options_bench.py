"""NMS with Ultralytics' multi_label / classes / agnostic options on one GPU, batch 64 at 640x640 (the YAML network,
init_synthetic(0), class bias calibrated as bench.py does, so that the single-label conf-0.25 configuration is the
benchmark's).  Records, with the card's name and power limit read in the same run:
  * per configuration: model.nms timed with CUDA events over --reps launches (after warm-up), candidates per image
    (anchors with best score > conf, or (anchor, class) pairs > conf under multi_label, after the class filter) and
    kept rows per image;
  * the same statements composed from torch + torchvision.ops.nms on the device, one image at a time (what
    Ultralytics' non_max_suppression runs in model.val on a CUDA device), timed with CUDA events, and whether its
    rows equal ours;
  * with --parent DIR (a build of another commit): bench.py (stages_ms.nms, nms_stress_1280) and tools/nms_probe.py
    of DIR and of this tree, alternated --rounds times, and whether the two bench runs returned the same detections.
Writes <out>/nms_options_bench.json.  Usage: python tools/nms_options_bench.py --out DIR [--parent DIR]"""
import argparse
import json
import re
import subprocess
import sys
import tempfile
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import unina_yolo_dla_b200 as uyd  # noqa: E402

B, S, IOU, MAX_DET, MAX_NMS, MAX_WH = 64, 640, 0.7, 300, 30000, 7680
CONFIGS = {
    "single_conf0.25 (bench)": dict(conf=0.25),
    "single_conf0.001": dict(conf=0.001),
    "multi_label_conf0.001 (model.val)": dict(conf=0.001, multi_label=True),
    "multi_label_conf0.001_classes[0]": dict(conf=0.001, multi_label=True, classes=[0]),
    "agnostic_conf0.25": dict(conf=0.25, agnostic=True),
}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi name, power.limit, clocks.sm, clocks.max.sm":
            q.stdout.strip() or q.stderr.strip()}


def events_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def torch_nms(y, conf, classes=None, agnostic=False, multi_label=False):
    """Ultralytics 8.3.x non_max_suppression on the device, statement by statement (stable argsort for the max_nms cut)."""
    import torchvision

    multi_label &= y.shape[1] > 5
    cls_t = torch.tensor(classes, device=y.device) if classes is not None else None
    xc = y[:, 4:].amax(1) > conf
    p = y.transpose(-1, -2)
    p = torch.cat((p[..., :2] - p[..., 2:4] / 2, p[..., :2] + p[..., 2:4] / 2, p[..., 4:]), -1)
    out = []
    for b in range(y.shape[0]):
        x = p[b][xc[b]]
        box, cls = x[:, :4], x[:, 4:]
        if multi_label:
            i, j = torch.where(cls > conf)
            x = torch.cat((box[i], x[i, 4 + j, None], j[:, None].float()), 1)
        else:
            c, j = cls.max(1, keepdim=True)
            x = torch.cat((box, c, j.float()), 1)[c.view(-1) > conf]
        if cls_t is not None:
            x = x[(x[:, 5:6] == cls_t).any(1)]
        if x.shape[0] > MAX_NMS:
            x = x[x[:, 4].argsort(descending=True, stable=True)[:MAX_NMS]]
        i = torchvision.ops.nms(x[:, :4] + x[:, 5:6] * (0 if agnostic else MAX_WH), x[:, 4], IOU)[:MAX_DET]
        out.append(x[i])
    return out


def candidates(y, conf, classes=None, agnostic=False, multi_label=False):
    sc = y[:, 4:]
    keep = torch.zeros(sc.shape[1], dtype=torch.bool, device=y.device)
    keep[[c for c in (classes if classes is not None else range(sc.shape[1])) if 0 <= c < sc.shape[1]]] = True
    if multi_label:
        return ((sc > conf) & keep[None, :, None]).sum((1, 2))
    best, j = sc.max(1)
    return ((best > conf) & keep[j]).sum(1)


def configs(reps):
    m = uyd.UninaYoloB200.from_yaml().init_synthetic(0).cuda()
    x = torch.rand(B, 3, S, S, device="cuda", generator=torch.Generator(device="cuda").manual_seed(100))
    m.calibrate_cls_bias(x[:8], 1500, 0.25)   # bench.py's CANDIDATES_PER_IMAGE and CONF
    y = m.forward(x, raw_heads=False)
    out = {}
    for name, kw in CONFIGS.items():
        kw = dict(kw)
        conf = kw.pop("conf")
        det, cnt = m.nms(y, conf, IOU, MAX_DET, MAX_NMS, **kw)
        ms = events_ms(lambda: m.nms(y, conf, IOU, MAX_DET, MAX_NMS, **kw), reps)
        ms_torch = events_ms(lambda: torch_nms(y, conf, **kw), max(3, reps // 20))
        rows = torch_nms(y, conf, **kw)
        equal = sum(int(torch.equal(rows[b], det[b, : int(cnt[b])])) for b in range(B))
        cand = candidates(y, conf, **kw).float()
        out[name] = {"conf": conf, **{k: v for k, v in kw.items()}, "iou": IOU, "max_det": MAX_DET, "max_nms": MAX_NMS,
                     "uyd_nms_ms": ms, "torch_torchvision_ms": ms_torch, "speedup_vs_torch": ms_torch / ms,
                     "candidates_per_image": {"mean": float(cand.mean()), "min": int(cand.min()), "max": int(cand.max())},
                     "kept_per_image": {"mean": float(cnt.float().mean()), "min": int(cnt.min()), "max": int(cnt.max())},
                     "images_with_rows_equal_to_torch": f"{equal}/{B}"}
        print(name, json.dumps(out[name]), flush=True)
    return out


def ab(parent: Path, rounds: int, steps: int):
    """bench.py and nms_probe.py of the parent build and of this tree, alternated."""
    runs = {"parent": [], "this": []}
    same = []
    with tempfile.TemporaryDirectory() as tmp:
        for r in range(rounds):
            dumps = {}
            for tag, tree in (("parent", parent), ("this", ROOT)):
                dump = Path(tmp) / f"{tag}{r}"
                b = subprocess.run([sys.executable, str(tree / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "5",
                                    "--cpu-sample", "0", "--int8", "0", "--custom", "0", "--c4-batch", "0", "--sustain", "0",
                                    "--dump-outputs", str(dump)], capture_output=True, text=True, cwd=tree)
                res = json.loads([ln for ln in b.stdout.splitlines() if ln.startswith("{")][-1])
                p = subprocess.run([sys.executable, str(tree / "tools" / "nms_probe.py")], capture_output=True, text=True, cwd=tree)
                probe = re.search(r"nms ms ([0-9.]+)", p.stdout)
                runs[tag].append({"bench_stages_ms_nms": res["stages_ms"]["nms"],
                                  "bench_nms_stress_1280_ms": res.get("nms_stress_1280", {}).get("ms_per_step"),
                                  "bench_value": res.get("value"), "nms_probe_ms": float(probe.group(1)) if probe else p.stderr[-400:]})
                dumps[tag] = dump
                print(tag, r, json.dumps(runs[tag][-1]), flush=True)
            same.append(all(np.load(dumps["parent"] / f).tobytes() == np.load(dumps["this"] / f).tobytes()
                            for f in ("detections.npy", "counts.npy")))
    summary = {}
    for tag, rs in runs.items():
        for k in ("bench_stages_ms_nms", "bench_nms_stress_1280_ms", "nms_probe_ms"):
            v = [r[k] for r in rs if isinstance(r[k], float)]
            if v:
                summary.setdefault(tag, {})[k] = {"min": min(v), "max": max(v), "spread": max(v) - min(v)}
    return {"rounds": runs, "summary": summary, "bench_detections_identical_per_round": same}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--parent", default="", help="tree of another build for the A/B of the default configuration")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    a = ap.parse_args()
    res = {"card": card(), "workload": f"YAML network init_synthetic(0), batch {B} at {S}x{S}, y[{B}, 8, 33600]",
           "configs": configs(a.reps)}
    if a.parent:
        res["ab_default"] = ab(Path(a.parent).resolve(), a.rounds, a.steps)
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "nms_options_bench.json").write_text(json.dumps(res, indent=1))
    print(json.dumps(res["card"]))


if __name__ == "__main__":
    main()
