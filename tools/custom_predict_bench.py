"""Post-processing cost of the model.py network (UninaCustomB200) on one GPU: the per-image composition predict used
before predict_batched (UninaCustomB200._predict_per_image: head export, per image 3 x uyd_decode_tlbr +
uyd_nms_detections + a host read of the count) against the batched path (one uyd_nms_tlbr launch on the plan's head
buffers).  Records, with the card's name and power limit read in the same run:
  * post-processing per step at batch 64: _predict_per_image minus plan.run (host clock over synchronised steps)
    against uyd_nms_tlbr alone (CUDA events over --nms-launches launches);
  * predict_batched step time against plan.run alone at batch 64 and 256 (CUDA events);
  * predict latency at batch 1, old (_predict_per_image) against new (predict, CUDA-graph replay): p50 and min.
Every shape is warmed up before it is timed; frames are seeded.  Writes <out>/custom_predict_bench.json.
Usage: python tools/custom_predict_bench.py --out DIR [--size 640] [--bc 32]"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import unina_yolo_dla_b200 as uyd  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def host_ms(fn, steps):
    """Per-call milliseconds of fn() on the host clock, each call ended by a device synchronise."""
    out = []
    for _ in range(steps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3)
    return sorted(out)


def event_ms(fn, steps):
    """Mean milliseconds of fn() over `steps` back-to-back calls between two CUDA events."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def med(v):
    return v[len(v) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--size", type=int, default=640)
    ap.add_argument("--bc", type=int, default=32)
    ap.add_argument("--conf", type=float, default=0.5)
    ap.add_argument("--iou", type=float, default=0.45)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--nms-launches", type=int, default=400)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("custom_predict_bench.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    S = a.size
    m = uyd.UninaCustomB200(4, a.bc).init_synthetic(seed=0).cuda()
    g = torch.Generator(device="cuda").manual_seed(700)
    res = {"card": card(), "network": f"UninaCustomB200(num_classes=4, base_channels={a.bc})", "size": S,
           "conf": a.conf, "iou": a.iou, "frames": "torch.rand seeded 700 on the device, fp32 NCHW"}

    # ---- batch 64: post-processing per step, old against new ----
    B = 64
    x = torch.rand(B, 3, S, S, device="cuda", generator=g)
    p = m.plan_for(x)
    det = torch.empty(B, 1024, 6, device="cuda")
    cnt = torch.empty(B, dtype=torch.int32, device="cuda")
    nms = lambda: m._nms_tlbr_into(p, B, det, cnt, a.conf, a.iou, 0.0, True, 1024, 0)
    old = lambda: m._predict_per_image(x, conf=a.conf, iou=a.iou)
    for _ in range(3):  # warm-up of every path timed below
        p.run(x)
        old()
        nms()
        m.predict_batched(x, conf=a.conf, iou=a.iou, graph=False)
    want = old()
    got_det, got_cnt = m.predict_batched(x, conf=a.conf, iou=a.iou, graph=False)
    same = all(int(got_cnt[b]) == len(want[b]) and torch.equal(got_det[b, :len(want[b])], want[b]) for b in range(B))
    run_host = host_ms(lambda: p.run(x), a.steps)
    old_host = host_ms(old, a.steps)
    nms_ms = event_ms(nms, a.nms_launches)
    res["batch64_postprocess"] = {
        "per_image_path_ms": med(old_host), "plan_run_ms": med(run_host),
        "per_image_postprocess_ms": med(old_host) - med(run_host),
        "per_image_postprocess_note": "_predict_per_image minus plan.run, medians of host-clock steps ended by a synchronise; "
                                      "includes the head export (Plan.read), 256 launches and 64 host reads of the count",
        "nms_tlbr_ms": nms_ms, "nms_tlbr_note": f"uyd_nms_tlbr alone, CUDA events over {a.nms_launches} launches",
        "speedup": (med(old_host) - med(run_host)) / nms_ms,
        "kept_per_image_mean": float(got_cnt.float().mean()), "outputs_byte_equal": bool(same)}

    # ---- predict_batched step against plan.run alone, batch 64 and 256 ----
    rows = {}
    for B in (64, 256):
        x = torch.rand(B, 3, S, S, device="cuda", generator=g)
        p = m.plan_for(x)
        step = lambda: m.predict_batched(x, conf=a.conf, iou=a.iou, graph=False)
        run = lambda: p.run(x)
        for _ in range(3):
            step()
            run()
        t_run, t_step = event_ms(run, a.steps), event_ms(step, a.steps)
        rows[str(B)] = {"plan_run_ms": t_run, "predict_batched_ms": t_step, "postprocess_share": (t_step - t_run) / t_step,
                        "images_per_s": B / (t_step * 1e-3)}
        del x
    res["predict_batched_step"] = rows
    res["predict_batched_step_note"] = "CUDA events over back-to-back steps (eager launches, no graph at these batches)"

    # ---- batch 1 predict latency: old against new (graph replay), alternated ----
    x1 = torch.rand(1, 3, S, S, device="cuda", generator=g)
    for _ in range(5):
        m._predict_per_image(x1, conf=a.conf, iou=a.iou)
        m.predict(x1, conf=a.conf, iou=a.iou)
    lo, ln = [], []
    for _ in range(100):
        lo += host_ms(lambda: m._predict_per_image(x1, conf=a.conf, iou=a.iou), 1)
        ln += host_ms(lambda: m.predict(x1, conf=a.conf, iou=a.iou), 1)
    lo.sort()
    ln.sort()
    res["predict_bs1_ms"] = {"old_per_image": {"p50": med(lo), "min": lo[0]}, "new_graph": {"p50": med(ln), "min": ln[0]},
                             "note": "host clock per call ended by a synchronise, 100 calls each, old and new alternated; "
                                     "both return per-image [N,6] rows (one host read of the counts)"}
    res["card_after"] = card()
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "custom_predict_bench.json").write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
