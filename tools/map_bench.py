"""mAP50 / mAP50-95 of a validation pass on one GPU: DetectionEvaluator(nc=80) over 5 000 seeded images x 300
detections x 20 labels (1.5 M detection rows), in batches of 64, against the restated Ultralytics numpy path
(oracle/mapref.py: match_predictions per image, then ap_per_class) on the same rows on this machine's host cores.
Records, with the card's name, power limit and SM clock read in the same run:
  * update per batch of 64: CUDA events around every update call of a pass, with nc=80 (uyd_eval_update +
    uyd_eval_match) and with nc=None (uyd_eval_update only), alternated over rounds;
  * map_metrics(): host clock around the call, ended by a synchronise (stable torch.sort of the records, one
    uyd_eval_ap launch, the read-back and the numpy tail); the sort alone with CUDA events;
  * the numpy path: host clock around the per-image matching and around ap_per_class + the results dict;
  * equal: the results dict and the per-class arrays of both paths compared exactly.
Writes <out>/map_bench.json.  Usage: python tools/map_bench.py --out DIR"""
import argparse
import json
import os
import platform
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from unina_yolo_dla_b200.evaluate import DetectionEvaluator  # noqa: E402
from oracle import mapref as er  # noqa: E402

N_IMG, N_DET, N_GT, BATCH, NC = 5000, 300, 20, 64, 80


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi name, power.limit, clocks.sm, clocks.max.sm":
            q.stdout.strip() or q.stderr.strip()}


def data(seed=0):
    """Batches (det [b, 300, 6], cnt, gt [b, 20, 5], gcnt) on the device: labels uniform in a 640 image, detections
    jittered label copies (80 % with the label's class) in confidence order."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for s in range(0, N_IMG, BATCH):
        b = min(BATCH, N_IMG - s)
        xy = torch.rand(b, N_GT, 2, generator=g) * 580
        wh = torch.rand(b, N_GT, 2, generator=g) * 55 + 5
        cls = torch.randint(0, NC, (b, N_GT, 1), generator=g).float()
        gt = torch.cat((cls, xy, xy + wh), 2)
        src = torch.randint(0, N_GT, (b, N_DET), generator=g)
        box = torch.gather(gt[..., 1:], 1, src[..., None].expand(b, N_DET, 4)) + torch.randn(b, N_DET, 4, generator=g) * 4
        dcls = torch.where(torch.rand(b, N_DET, generator=g) < 0.8, torch.gather(cls[..., 0], 1, src),
                           torch.randint(0, NC, (b, N_DET), generator=g).float())
        conf = torch.rand(b, N_DET, generator=g).sort(1, descending=True).values
        det = torch.cat((box, conf[..., None], dcls[..., None]), 2)
        out.append(tuple(t.cuda() for t in (det, torch.full((b,), N_DET, dtype=torch.int32), gt, torch.full((b,), N_GT, dtype=torch.int32))))
    return out


def update_pass(batches, nc):
    ev = DetectionEvaluator(nc=nc)
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in batches]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in batches]
    torch.cuda.synchronize()
    for a, b, x in zip(ev0, ev1, batches):
        a.record()
        ev.update(*x)
        b.record()
    torch.cuda.synchronize()
    return ev, [a.elapsed_time(b) for a, b in zip(ev0, ev1)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {"card": card(), "workload": f"{N_IMG} images x {N_DET} detections x {N_GT} labels, nc {NC}, batches of {BATCH}",
           "host": {"cpu_count": os.cpu_count(), "processor": platform.processor(), "torch_threads": torch.get_num_threads()}}
    batches = data()
    update_pass(batches, NC)[0].map_metrics()   # warm-up of every shape
    update_pass(batches, None)
    upd = {"nc80": [], "nc_none": []}
    for _ in range(args.rounds):
        ev, t = update_pass(batches, NC)
        upd["nc80"].append(float(np.mean(t)))
        upd["nc_none"].append(float(np.mean(update_pass(batches, None)[1])))
    res["update_ms_per_batch64_mean_per_round"] = upd
    mm = []
    for _ in range(args.rounds):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        got = ev.map_metrics()
        torch.cuda.synchronize()
        mm.append((time.perf_counter() - t0) * 1e3)
    res["map_metrics_ms"] = mm
    keys = torch.cat(ev._keys)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st = []
    for _ in range(args.rounds):
        s0.record()
        torch.sort(keys, stable=True)
        s1.record()
        torch.cuda.synchronize()
        st.append(s0.elapsed_time(s1))
    res["records"] = int(keys.numel())
    res["sort_ms"] = st

    dets, gts = [], []
    for det, cnt, gt, gcnt in batches:
        det, gt = det.cpu(), gt.cpu()
        for b in range(det.shape[0]):
            dets.append(det[b, : int(cnt[b])])
            gts.append(gt[b, : int(gcnt[b])])
    t0 = time.perf_counter()
    stats = er.map_stats(dets, gts)
    t1 = time.perf_counter()
    ref = er.det_metrics(*stats)
    t2 = time.perf_counter()
    res["numpy_match_s"], res["numpy_ap_per_class_s"] = t1 - t0, t2 - t1
    res["results"] = {k: float(got[k]) for k in er.RESULT_KEYS + ("fitness",)}
    res["equal"] = bool(all(got[k] == ref[k] for k in er.RESULT_KEYS + ("fitness",))
                        and all(np.array_equal(got[k], ref[k]) for k in ("ap50", "ap", "ap_class_index")))
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "map_bench.json").write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
