"""INT8 against bf16 for the model.py network (UninaCustomB200) on one GPU.  bc32, 640x640 model input, synthetic
weights; the INT8 model is max-calibrated on 8 seeded frames with the default float layers (stem, head_p2).  Records,
with the card's name, power limit and SM clock read in the same run:
  * step time at batch 64 and 256: plan.run, CUDA events over back-to-back steps, INT8 and bf16 alternated in rounds
    (at least 200 steps of each), and predict_batched (plan + one NMS launch) the same way;
  * batch 1: predict (CUDA-graph replay) host-clock p50 per call ended by a synchronise;
  * the per-op table of the INT8 plan at batch 64 (plan.profile, median of several passes): for every conv_s8 its
    TOP/s and the fraction of the measured kind::i8 peak (profiles/int8_peak.json); for every conv shape that runs on
    the streamed-weight route, its INT8 and bf16 times side by side; the quantize launches, counted and timed.
Every shape is warmed up before it is timed; frames are seeded.  Writes <out>/custom_int8_bench.json.
Usage: python tools/custom_int8_bench.py --out DIR"""
import argparse
import json
import re
import subprocess
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
import unina_yolo_dla_b200 as uyd  # noqa: E402
from oracle import init as oi  # noqa: E402

S = 640
SHAPE = re.compile(r"^conv(?:_s8)? (\d+->\d+ k\d s\d) (\d+x\d+)")


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi name, power.limit, clocks.max.sm, clocks.sm":
            q.stdout.strip() or q.stderr.strip()}


def event_ms(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def alternate(fns: dict, steps: int, rounds: int) -> dict:
    """Mean ms per step of each fn over `rounds` alternated windows of `steps` steps; also the per-round spread."""
    for f in fns.values():
        for _ in range(3):
            f()
    per = {k: [] for k in fns}
    for _ in range(rounds):
        for k, f in fns.items():
            per[k].append(event_ms(f, steps))
    return {k: {"mean_ms": sum(v) / len(v), "min_ms": min(v), "max_ms": max(v), "steps": steps * rounds} for k, v in per.items()}


def med(v):
    v = sorted(v)
    return v[len(v) // 2]


def profile(p, x, passes):
    for _ in range(2):
        p.profile(x)
    runs = [p.profile(x) for _ in range(passes)]
    return [med([r[i] for r in runs]) for i in range(p.launches)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--bc", type=int, default=32)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--passes", type=int, default=7)
    ap.add_argument("--bs1-calls", type=int, default=300)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("custom_int8_bench.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    peak = json.loads((ROOT / "profiles" / "int8_peak.json").read_text())["int8_tops_dense"]
    mf = uyd.UninaCustomB200(4, a.bc).init_synthetic(seed=0).cuda()
    mq = uyd.UninaCustomB200(4, a.bc).cuda()
    mq.load_state_dict(mf.state_dict())
    calib = oi.seeded_frames(8, S, seed=11).cuda()
    amax = mq.calibrate_int8(calib, method="max")
    res = {"card": card(), "network": f"UninaCustomB200(num_classes=4, base_channels={a.bc}), init_synthetic(seed=0)",
           "model_input": [S, S], "int8": {"calibration": "max over 8 seeded frames (oracle.init.seeded_frames seed 11)",
                                           "float_layers": list(mq.quant.float_layers),
                                           "quantised_convs": sum(1 for n in amax if mq.quant.covers(n))},
           "int8_peak_tops": peak, "steps": {}, "predict_batched": {}}
    for B in (64, 256):
        x = oi.seeded_frames(B, S, seed=B).cuda()
        pf, pq = mf.plan_for(x), mq.plan_for(x)
        r = alternate({"bf16": lambda: pf.run(x), "int8": lambda: pq.run(x)}, a.steps, a.rounds)
        r["int8_over_bf16"] = r["int8"]["mean_ms"] / r["bf16"]["mean_ms"]
        res["steps"][f"batch{B}"] = r
        r = alternate({"bf16": lambda: mf.predict_batched(x, graph=False), "int8": lambda: mq.predict_batched(x, graph=False)},
                      a.steps, a.rounds)
        r["int8_over_bf16"] = r["int8"]["mean_ms"] / r["bf16"]["mean_ms"]
        res["predict_batched"][f"batch{B}"] = r
        del pf, pq
        mf.refresh(), mq.refresh()
        torch.cuda.empty_cache()

    # ---- batch 1: predict through the captured graph ----
    x1 = oi.seeded_frames(1, S, seed=1).cuda()
    bs1 = {}
    for name, m in (("bf16", mf), ("int8", mq)):
        for _ in range(10):
            m.predict(x1)
        t = []
        for _ in range(a.bs1_calls):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m.predict(x1)
            torch.cuda.synchronize()
            t.append((time.perf_counter() - t0) * 1e3)
        bs1[name] = {"p50_ms": med(t), "min_ms": min(t), "calls": a.bs1_calls}
    res["predict_bs1_graph"] = bs1

    # ---- per-op table at batch 64 ----
    B = 64
    x = oi.seeded_frames(B, S, seed=B).cuda()
    pf, pq = mf.plan_for(x), mq.plan_for(x)
    tq, tf = profile(pq, x, a.passes), profile(pf, x, a.passes)
    ops, quant = [], {"launches": 0, "ms": 0.0}
    for i, ms in enumerate(tq):
        text, fl, by = pq.op_info(i)
        row = {"op": i, "text": text, "ms": ms}
        if text.startswith("conv_s8"):
            tops = fl * B / (ms * 1e-3) / 1e12
            row.update(tops=tops, fraction_of_int8_peak=tops / peak, hbm_tb_s=by * B / (ms * 1e-3) / 1e12)
        if text.startswith("quantize"):
            quant["launches"] += 1
            quant["ms"] += ms
        ops.append(row)
    bf_ops = {}
    for i, ms in enumerate(tf):
        text = pf.op_info(i)[0]
        mt = SHAPE.match(text)
        if mt:
            bf_ops.setdefault(mt.groups(), []).append((text, ms))
    big, seen = [], {}
    for row in ops:
        mt = SHAPE.match(row["text"])
        if not (mt and row["text"].startswith("conv_s8") and "tc:big-" in row["text"]):
            continue
        k = mt.groups()
        j = seen.get(k, 0)
        seen[k] = j + 1
        bf = bf_ops.get(k, [])
        big.append({"shape": " ".join(k), "int8": row["text"], "int8_ms": row["ms"],
                    "bf16": bf[j][0] if j < len(bf) else None, "bf16_ms": bf[j][1] if j < len(bf) else None})
    res["per_op_batch64"] = {"int8_plan_ms_sum": sum(tq), "bf16_plan_ms_sum": sum(tf), "quantize": quant,
                             "conv_s8_ms_sum": sum(r["ms"] for r in ops if r["text"].startswith("conv_s8")),
                             "big_route_side_by_side": big, "int8_ops": ops}
    res["card_after"] = card()
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "custom_int8_bench.json").write_text(json.dumps(res, indent=1))
    print(json.dumps({k: res[k] for k in ("card", "steps", "predict_batched", "predict_bs1_graph")}, indent=1))
    print(json.dumps({k: v for k, v in res["per_op_batch64"].items() if k != "int8_ops"}, indent=1))


if __name__ == "__main__":
    main()
