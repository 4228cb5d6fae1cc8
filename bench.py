#!/usr/bin/env python
"""bench.py -- images/sec of the UNINA-YOLO-DLA inference hot path on B200.

Contract (driver): python bench.py --gpus N --steps K --warmup W [--impl reference]
prints ONE JSON line on rank 0.

Workload (BASELINE.json configs[1]): unina-yolo-dla-m, bf16 forward + DFL decode + NMS,
640x640, batch 64 per GPU, seeded synthetic weights (UninaYoloB200.init_synthetic) and frames.
A step = one pass of the hot path over one batch.
  value : images/s, frames already resident in HBM as NCHW fp32 (the reference forward signature)
  e2e   : images/s through the public streaming predict call with HOST frames: K pinned uint8
          NCHW batches fed to UninaYoloB200.predict_stream -> per step H2D (on a copy stream,
          overlapping the previous step's compute) -> forward(+/255 fused in the stem) -> decode
          -> NMS -> D2H of [B,300,6]+counts (+ NCCL all_gather of the detections when N > 1: the
          batched-eval gather).  e2e.single_call_ms is the same step as ONE blocking
          predict_batched call (copy and compute serialised).
  roofline    : the dominant kernel, timed live with CUDA events inside the timed steps
  cpu_baseline: the oracle (restated reference path) on the host cores, bounded sample
Multi-GPU: frames shard data-parallel, no collective on the forward path ("weak" scaling).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "images/sec @640x640 (forward + DFL decode + NMS)"
UNIT = "images/s"
CONF, IOU, MAX_DET = 0.25, 0.7, 300
CANDIDATES_PER_IMAGE = 1500


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="frames per GPU per step")
    ap.add_argument("--size", type=int, default=640)
    ap.add_argument("--cpu-sample", type=int, default=32, help="frames of the bounded CPU sample")
    ap.add_argument("--profile-out", default="", help="write the per-op table (markdown) here")
    ap.add_argument("--stress", type=int, default=32, metavar="BATCH",
                    help="N = 1: also time decode-free NMS on a synthetic dense 1280x1280 scene (134 400 anchors, ~100k candidates "
                         "per image, BASELINE config 5) at this batch (0 = skip)")
    ap.add_argument("--int8", type=int, default=256, metavar="BATCH",
                    help="N = 1: also time the INT8 graph (static max-calibrated scales, BASELINE config 3) at this batch (0 = skip)")
    ap.add_argument("--custom", type=int, default=64, metavar="BATCH",
                    help="N = 1: also time the model.py variant (UninaCustomB200, the pinned-oracle network) at this batch (0 = skip)")
    ap.add_argument("--c4-batch", type=int, default=256, metavar="BATCH",
                    help="every N: also time BASELINE config 4's per-GPU batch (resident and e2e), 0 = skip")
    ap.add_argument("--host-mem", default="pinned", choices=["pinned", "wc"],
                    help="host staging buffers of the e2e run: torch pinned memory, or write-combined pinned memory (uyd_host_alloc)")
    ap.add_argument("--sustain", type=float, default=2.0, metavar="SECONDS",
                    help="also run the resident step back to back for at least this long, with clocks (0 = skip)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step returned (rank 0: detections and counts) as DIR/<name>.npy, "
                         "so that two builds can be compared output for output on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs applies to the GPU path only")
    return a


DUMP_BYTES = 64_000_000   # --dump-outputs writes at most this much data


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """One float32 / float64 .npy file per returned array (float32 data as is, integer data widened to float64,
    which holds every int32 exactly).  The arrays share their leading (image) dimension; where all images would take
    more than DUMP_BYTES, a fixed seeded sample of them is written, with their indices as image_index.npy."""
    import numpy as np

    out = {k: t.detach().cpu() for k, t in arrays.items()}
    out = {k: t if t.dtype == torch.float32 else t.double() for k, t in out.items()}
    n = next(iter(out.values())).shape[0]
    per_image = sum(t[0].numel() * t.element_size() for t in out.values())
    if n * per_image > DUMP_BYTES:
        keep = torch.randperm(n, generator=torch.Generator().manual_seed(0))[: DUMP_BYTES // (per_image + 8)].sort().values
        out = {k: t[keep] for k, t in out.items()}
        out["image_index"] = keep.double()
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in out.items():
        np.save(d / f"{name}.npy", t.numpy())


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "tflops_burst": d["bf16_tflops"],
                "src": "measured"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "tflops_burst": 1600.0, "src": "fallback"}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = next((int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()), None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def build_models(size: int, need_oracle: bool):
    import unina_yolo_dla_b200 as uyd

    model = uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0)
    return model


def oracle_from(model):
    """The CPU oracle carrying the product's weights (cpu_baseline / --impl reference only)."""
    from oracle import yolo_graph as yg

    ref = yg.DetectionModel(yg.default_yaml_path())
    ref.load_state_dict({k: v.detach().cpu() for k, v in model.state_dict().items()}, strict=True)
    return ref.eval()


def cpu_pass(ref, frames: torch.Tensor):
    """Reference path on the host: fp32 forward + DFL decode + Ultralytics-style NMS."""
    from oracle import postproc as pp

    with torch.no_grad():
        y, _ = ref(frames)
    return pp.non_max_suppression(y.numpy(), CONF, IOU, MAX_DET)


def cpu_baseline(model, size: int, sample: int, chunk: int = 8):
    torch.set_num_threads(os.cpu_count() or 1)
    ref = oracle_from(model)
    g = torch.Generator().manual_seed(1)
    frames = torch.rand(chunk, 3, size, size, generator=g)
    cpu_pass(ref, frames[:2])  # warm-up
    t0 = time.perf_counter()
    done = 0
    while done < sample:
        cpu_pass(ref, frames)
        done += chunk
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{done} frames of the same workload in chunks of {chunk} (oracle fp32 forward + DFL decode + NMS)"}


def bench_int8(model, batch: int, size: int, dev, steps: int):
    """BASELINE config 3: the INT8 graph (model.0-2 float, every other conv int8 with static scales calibrated on
    8 frames, DFL projection quantised) at `batch` frames, forward + decode + NMS, frames resident in HBM."""
    g = torch.Generator(device=dev).manual_seed(300)
    x = torch.rand(batch, 3, size, size, device=dev, generator=g)
    model.calibrate_int8(x[:8])
    plan = model.plan_for(x)
    for _ in range(2):
        model.predict_batched(x, CONF, IOU, MAX_DET)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        model.predict_batched(x, CONF, IOU, MAX_DET)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    n_blk = sum(1 for i in range(plan.launches) if plan.op_info(i)[0].startswith("c3k_fused_s8"))
    n_fold = sum(1 for i in range(plan.launches) if plan.op_info(i)[0].startswith("conv_s8") and "+up(partial)" in plan.op_info(i)[0])
    n_s8 = sum(1 for i in range(plan.launches) if plan.op_info(i)[0].startswith("conv_s8")) - n_fold + 7 * n_blk
    s8_ops = sum(plan.op_info(i)[1] for i in range(plan.launches) if plan.op_info(i)[0].startswith("conv_s8"))
    prof = plan.profile(x, None)
    s8_ms = sum(t for i, t in enumerate(prof) if plan.op_info(i)[0].startswith("conv_s8"))
    q_ms = sum(t for i, t in enumerate(prof) if plan.op_info(i)[0].startswith("quantize"))
    pk8 = ROOT / "profiles" / "int8_peak.json"
    peak8 = json.loads(pk8.read_text())["int8_tops_dense"] if pk8.exists() else 4500.0
    tops = s8_ops * batch / (s8_ms * 1e-3) / 1e12
    out = {"value": batch / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "batch": batch, "steps": steps, "dtype": "s8 x s8 -> s32",
           "plan_launches": plan.launches, "int8_convs": n_s8, "activation_bytes": plan.bytes,
           "roofline": {"bound": "tensor", "achieved": tops, "peak": peak8, "unit": "TOP/s", "frac": tops / peak8,
                        "peak_source": "measured kind::i8 probe at the maximum SM clock (profiles/int8_peak.json)" if pk8.exists() else "nominal",
                        "int8_conv_ms": s8_ms, "quantize_ms": q_ms,
                        "note": "achieved = int8 conv ops of the plan x batch / the summed CUDA-event time of the conv_s8 launches"},
           "fused_c3k_blocks": n_blk,
           "note": "C3k blocks run as one launch each (seven int8 convs + their input quantisers, uyd_plan_add_c3k_s8; their time "
                   "is not in roofline.int8_conv_ms); the remaining quantize ops are separate launches (one int8 copy per activation "
                   "slice and scale)"}
    model.set_quantization(None)
    return out


def bench_nms_stress(model, batch: int, dev, steps: int):
    """BASELINE config 5: class-aware NMS on a dense 1280x1280 scene: 134 400 anchors per image, ~75 % of them
    above conf (top-30000 truncation active), boxes clustered around 64 centres per image."""
    A = 102400 + 25600 + 6400
    g = torch.Generator(device=dev).manual_seed(500)
    centres = torch.rand(batch, 2, 64, device=dev, generator=g) * 1200 + 40
    pick = torch.randint(0, 64, (batch, 1, A), device=dev, generator=g).expand(batch, 2, A)
    y = torch.empty(batch, 8, A, device=dev)
    y[:, 0:2] = torch.gather(centres, 2, pick) + torch.randn(batch, 2, A, device=dev, generator=g) * 6
    y[:, 2:4] = torch.rand(batch, 2, A, device=dev, generator=g) * 88 + 8
    sc = torch.rand(batch, 4, A, device=dev, generator=g)
    lift = torch.rand(batch, 1, A, device=dev, generator=g) < 0.75
    y[:, 4:] = torch.where(lift, 0.25 + 0.75 * sc, 0.2 * sc)
    cand = int((y[:, 4:].amax(1) > CONF).sum(1).float().mean())
    for _ in range(2):
        det, cnt = model.nms(y, CONF, IOU, MAX_DET)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        det, cnt = model.nms(y, CONF, IOU, MAX_DET)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"ms_per_step": ms, "images_per_s": batch / (ms * 1e-3), "batch": batch, "anchors": A, "candidates_per_image": cand,
            "kept_per_image": float(cnt.float().mean()), "steps": steps}


FAMILIES = (("stem", "stem"), ("c3k", "c3k"), ("chain", "chain"), ("conv_tc", " tc"), ("sppf", "sppf"))


def family_of(text: str) -> str:
    for name, key in FAMILIES:
        if key in text:
            return name
    return "other"


def family_table(plan, ms, batch, pk, nms_ms=None):
    """Per-kernel-family share of the step and both roofline fractions (algorithmic flops / bytes of the ops in the
    family over the family's summed CUDA-event time)."""
    fam = {}
    for i, t in enumerate(ms):
        text, fl, by = plan.op_info(i)
        f = fam.setdefault(family_of(text), {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
        f["launches"] += 1; f["ms"] += t; f["flops"] += fl * batch; f["bytes"] += by * batch
    total = sum(ms) + (nms_ms or 0.0)
    out = {}
    for name, f in fam.items():
        tf, gb = f["flops"] / (f["ms"] * 1e-3) / 1e12, f["bytes"] / (f["ms"] * 1e-3) / 1e9
        out[name] = {"launches": f["launches"], "ms": f["ms"], "share": f["ms"] / total, "tflops": tf, "frac_tensor": tf / pk["tflops_burst"],
                     "gbs": gb, "frac_hbm": gb / pk["hbm_gbs"]}
    if nms_ms:
        out["nms"] = {"launches": 1, "ms": nms_ms, "share": nms_ms / total}
    return out


def bench_custom(batch: int, size: int, dev, steps: int, pk, profile_out: str = ""):
    """The model.py variant (UninaCustomB200, base_channels 32: 35.7 GFLOP per 640x640 frame, every 3x3 conv with
    C >= 32): conv stack at `batch` resident frames + one-frame predict (forward + TLBR decode + postprocess.hpp NMS)."""
    import unina_yolo_dla_b200 as uyd

    m = uyd.UninaCustomB200(4, 32).init_synthetic(seed=0).to(dev)
    g = torch.Generator(device=dev).manual_seed(700)
    x = torch.rand(batch, 3, size, size, device=dev, generator=g)
    plan = m.plan_for(x)
    for _ in range(3):
        plan.run(x)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        plan.run(x)
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / steps
    ms = plan.profile(x, None)
    flops = sum(plan.op_info(i)[1] for i in range(plan.launches))
    x1 = x[:1].contiguous()
    for _ in range(3):
        m.predict(x1, conf=0.5, iou=0.45)
    lat = []
    for _ in range(20):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.predict(x1, conf=0.5, iou=0.45)
        torch.cuda.synchronize()
        lat.append((time.perf_counter() - t0) * 1e3)
    lat.sort()
    tf = flops * batch / (ms_step * 1e-3) / 1e12
    if profile_out:
        rows = ["| # | op | ms | share | TFLOP/s | frac of burst peak | GB/s |", "|---|---|---|---|---|---|---|"]
        for i in sorted(range(len(ms)), key=lambda i: -ms[i]):
            t, fl, by = plan.op_info(i)
            tfi = fl * batch / (ms[i] * 1e-3) / 1e12
            rows.append(f"| {i} | {t} | {ms[i]:.4f} | {100 * ms[i] / sum(ms):.1f}% | {tfi:.1f} | {tfi / pk['tflops_burst']:.2f} | {by * batch / (ms[i] * 1e-3) / 1e9:.0f} |")
        Path(profile_out).write_text(f"model.py variant (UninaCustomB200 bc32): per-op CUDA-event times, batch {batch}, {size}x{size}\n\n" + "\n".join(rows) + "\n")
    return {"workload": f"model.py network (base_channels 32) conv stack, {size}x{size}, batch {batch}, bf16, resident frames",
            "value": batch / (ms_step * 1e-3), "unit": UNIT, "ms_per_step": ms_step, "plan_launches": plan.launches,
            "conv_gflop_per_image": flops / 1e9, "tflops": tf, "frac_of_tensor_peak_burst": tf / pk["tflops_burst"],
            "frac_of_tensor_peak_sustained": tf / pk["tflops"], "families": family_table(plan, ms, batch, pk),
            "predict_bs1_ms": {"p50": lat[len(lat) // 2], "min": lat[0],
                               "note": "forward + TLBR decode x3 + record NMS + D2H of the kept count, one frame, host wall clock"}}


def cpu_calibrate_cls_bias(ref, frames: torch.Tensor, per_image: int, conf: float) -> float:
    """UninaYoloB200.calibrate_cls_bias restated on the CPU oracle (the reference arm must not touch libuyd.so):
    shifts the class biases so that about `per_image` anchors per image clear `conf`."""
    import math

    det = ref.model[-1]
    with torch.no_grad():
        _, xs = ref(frames)
        best = torch.cat([t[:, 4 * det.reg_max:].amax(1).flatten(1) for t in xs], 1)
        k = max(1, min(best.shape[1] - 1, per_image))
        kth = best.topk(k, dim=1).values[:, -1].mean().item()
        shift = math.log(conf / (1 - conf)) - kth
        for cls in det.cv3:
            cls[-1].bias.add_(shift)
    return shift


def run_reference(a):
    """--impl reference: the reference's CPU implementation of the path on the host cores.
    ultralytics is not installable here (no network, unpinned, not vendored) and model.py is a
    different network, so this is the oracle port (kind = "port", see DESIGN.md)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    torch.set_num_threads(os.cpu_count() or 1)
    model = build_models(a.size, True)          # CPU module only: same seeded weights as the GPU arm, libuyd.so is never loaded
    ref = oracle_from(model)
    chunk = 8
    g = torch.Generator().manual_seed(0)
    cpu_calibrate_cls_bias(ref, torch.rand(chunk, 3, a.size, a.size, generator=g), CANDIDATES_PER_IMAGE, CONF)  # same NMS load as the GPU arm
    frames = torch.rand(chunk, 3, a.size, a.size, generator=torch.Generator().manual_seed(1))
    per_step = max(chunk, a.batch // chunk * chunk)   # the same batch-64 step as the GPU arm, walked in chunks of 8 frames

    def one_step():
        for _ in range(per_step // chunk):
            cpu_pass(ref, frames)

    cpu_pass(ref, frames)
    for _ in range(max(0, a.warmup - 1)):
        one_step()
    steps = max(1, a.steps)
    t0 = time.perf_counter()
    for _ in range(steps):
        one_step()
    dt = time.perf_counter() - t0
    v = steps * per_step / dt
    chunk = per_step
    cores = torch.get_num_threads()
    sample = f"{chunk} frames per step in chunks of 8 ({steps} timed steps of the batch-{a.batch} workload)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": steps, "warmup": a.warmup,
        "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"unina-yolo-dla-m bf16 forward + DFL decode + NMS, {a.size}x{a.size}, batch {a.batch} per GPU",
                   "reference_arm": f"oracle port, fp32 on the host cores, {chunk} frames per step (chunks of 8 frames), class biases calibrated on the CPU oracle"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)

    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    B, S = a.batch, a.size

    model = build_models(S, False).to(dev)
    gen = torch.Generator(device=dev).manual_seed(100 + rank)
    x_dev = torch.rand(B, 3, S, S, device=dev, generator=gen)                       # resident fp32 frames
    x_host = (torch.rand(B, 3, S, S, generator=torch.Generator().manual_seed(200 + rank)) * 255).to(torch.uint8)
    if a.host_mem == "wc":
        from unina_yolo_dla_b200.hostmem import pinned_frames

        wc = pinned_frames(x_host.shape, torch.uint8, write_combined=True)
        wc.copy_(x_host)
        x_host = wc
    else:
        x_host = x_host.pin_memory()
    x_u8 = torch.empty_like(x_host, device=dev)
    model.calibrate_cls_bias(x_dev[: min(B, 8)], CANDIDATES_PER_IMAGE, CONF)
    plan = model.plan_for(x_dev, fused=True)   # the plan predict runs: head kernels decode in their epilogue
    y_prof = torch.empty(B, 4 + model.nc, model.num_anchors(S, S), device=dev)
    det_host = torch.empty(B, MAX_DET, 6).pin_memory()
    cnt_host = torch.empty(B, dtype=torch.int32).pin_memory()

    last = []   # what the most recent resident step returned (det, cnt): --dump-outputs writes the last timed one

    def step_resident():
        last[:] = model.predict_batched(x_dev, CONF, IOU, MAX_DET)

    def step_e2e():  # one blocking call: H2D, compute, D2H serialised
        x_u8.copy_(x_host, non_blocking=True)
        det, cnt = model.predict_batched(x_u8, CONF, IOU, MAX_DET)
        if world > 1:  # batched-eval gather of the detections (the only collective of the path)
            det, cnt = gatherer.start(det, cnt).wait()
            det, cnt = det[rank * B:(rank + 1) * B], cnt[rank * B:(rank + 1) * B]
        det_host.copy_(det, non_blocking=True)
        cnt_host.copy_(cnt, non_blocking=True)

    gatherer = None
    if world > 1:
        from unina_yolo_dla_b200.dp import DetectionGather

        gatherer = DetectionGather()

    def run_stream(steps, xh=None, gather=True, h2d=True):
        """The streaming API: H2D of step i+1 overlaps the compute of step i; with N > 1 every step's detections go
        through ONE fixed-shape NCCL all_gather on a side stream (no host sync) and the rank's rows come back to the
        host.  gather / h2d = False switch one stage off (e2e.bound_probe)."""
        xh = x_host if xh is None else xh
        dh = det_host if xh is x_host else torch.empty(xh.shape[0], MAX_DET, 6).pin_memory()
        ch = cnt_host if xh is x_host else torch.empty(xh.shape[0], dtype=torch.int32).pin_memory()
        nb = xh.shape[0]
        src = (xh for _ in range(steps))
        if not h2d:  # frames already on the device: the generator only slices them
            xd = xh.to(dev)
            for _ in range(steps):
                det, cnt = model.predict_batched(xd, CONF, IOU, MAX_DET)
                if world > 1 and gather:
                    det, cnt = gatherer.start(det, cnt).wait()
                    det, cnt = det[rank * nb:(rank + 1) * nb], cnt[rank * nb:(rank + 1) * nb]
                dh.copy_(det, non_blocking=True)
                ch.copy_(cnt, non_blocking=True)
            return
        if world == 1 or not gather:
            for det_h, cnt_h in model.predict_stream(src, CONF, IOU, MAX_DET, to_host=True):
                pass
            dh.copy_(det_h)
            ch.copy_(cnt_h)
        else:
            pending = None
            for det, cnt in model.predict_stream(src, CONF, IOU, MAX_DET, to_host=False):
                h = gatherer.start(det, cnt)
                if pending is not None:  # consume step i - 1 while step i's exchange is in flight
                    gd, gc = pending.wait()
                    dh.copy_(gd[rank * nb:(rank + 1) * nb], non_blocking=True)
                    ch.copy_(gc[rank * nb:(rank + 1) * nb], non_blocking=True)
                pending = h
            gd, gc = pending.wait()
            dh.copy_(gd[rank * nb:(rank + 1) * nb], non_blocking=True)
            ch.copy_(gc[rank * nb:(rank + 1) * nb], non_blocking=True)

    warm = max(3, a.warmup)
    for _ in range(warm):
        step_resident()
    torch.cuda.synchronize()
    # per-op profile (outside the timed region) -> dominant kernel
    ms = plan.profile(x_dev, y_prof)
    top = max(range(len(ms)), key=lambda i: ms[i])
    top_text, top_flops, top_bytes = plan.op_info(top)
    plan.set_timed_op(top, min(a.steps, 4096))   # the library keeps at most 4096 event pairs: longer runs sample the first ones

    def timed(fn, steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_total = timed(step_resident, a.steps)
    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=10)   # an nvidia-smi query still in flight stalls work submission for tens of ms
    top_ms_total, top_n = plan.timed_op_read()
    plan.set_timed_op(-1, 0)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"detections": last[0], "counts": last[1]})

    def run_resident_stream(steps):  # the streaming API on resident frames: NMS of step i on a second stream under step i + 1
        for _det, _cnt in model.predict_stream((x_dev for _ in range(steps)), CONF, IOU, MAX_DET, to_host=False):
            pass

    run_resident_stream(3)
    ms_pipe = min(timed(lambda: run_resident_stream(a.steps), 1) for _ in range(2))
    for _ in range(2):
        step_e2e()
    ms_e2e_single = timed(step_e2e, a.steps)
    run_stream(2)
    # the streamed run is one host-driven pipeline of K steps: a single hiccup of the host (page faults of the pinned
    # staging buffers, a neighbour on the PCIe switch) lands entirely in it, so it is repeated and the best of three kept
    ms_e2e = min(timed(lambda: run_stream(a.steps), 1) for _ in range(3))
    n_det = int(cnt_host.sum().item())
    # which stage bounds e2e: the same streamed run with one stage switched off
    probe = {}
    if world > 1:
        probe["no_gather_ms_per_step"] = min(timed(lambda: run_stream(a.steps, gather=False), 1) for _ in range(2)) / a.steps
    probe["no_h2d_ms_per_step"] = min(timed(lambda: run_stream(a.steps, h2d=False), 1) for _ in range(2)) / a.steps

    def h2d_only():  # the pinned host -> device copies of the streamed run alone, all ranks at once: the platform's H2D rate
        for _ in range(a.steps):
            x_u8.copy_(x_host, non_blocking=True)

    h2d_only()
    h2d_ms = min(timed(h2d_only, 1) for _ in range(2)) / a.steps
    probe["h2d_only_ms_per_step"] = h2d_ms
    probe["h2d_only_gbs_per_gpu"] = x_host.numel() / (h2d_ms * 1e-3) / 1e9
    # ceiling the host-to-device path of the box puts on e2e with 3-byte pixels (all ranks copying at once;
    # tools/h2d_probe.py: pinned, write-combined, two streams and chunked copies all give the same figure)
    probe["h2d_cap_images_per_s"] = world * B / (h2d_ms * 1e-3)
    # the same streamed run fed with NV12 camera frames (1.5 bytes per pixel over PCIe; the stem converts on load)
    nv_host = torch.randint(0, 256, (B, S * 3 // 2, S), dtype=torch.uint8, generator=torch.Generator().manual_seed(600 + rank)).pin_memory()

    def run_stream_nv12(steps):
        pending = None
        for det, cnt in model.predict_stream((nv_host for _ in range(steps)), CONF, IOU, MAX_DET, to_host=world == 1, camera="nv12"):
            if world > 1:
                h = gatherer.start(det, cnt)
                if pending is not None:
                    gd, gc = pending.wait()
                    det_host.copy_(gd[rank * B:(rank + 1) * B], non_blocking=True)
                    cnt_host.copy_(gc[rank * B:(rank + 1) * B], non_blocking=True)
                pending = h
        if pending is not None:
            gd, gc = pending.wait()
            det_host.copy_(gd[rank * B:(rank + 1) * B], non_blocking=True)
            cnt_host.copy_(gc[rank * B:(rank + 1) * B], non_blocking=True)

    run_stream_nv12(2)
    ms_nv12 = min(timed(lambda: run_stream_nv12(a.steps), 1) for _ in range(2))
    # sustained: the resident step back to back for >= a.sustain seconds, clocks sampled throughout
    sustained = None
    if a.sustain > 0:
        n_sus = max(a.steps, int(a.sustain * 1e3 / (ms_total / a.steps)) + 1)
        smp = ClockSampler(local)
        if rank == 0:
            smp.start()
        ms_sus = timed(step_resident, n_sus)
        if rank == 0:
            smp.stop_flag = True
            smp.join(timeout=10)
        sustained = {"steps": n_sus, "seconds": ms_sus * 1e-3, "value": world * B * n_sus / (ms_sus * 1e-3), "unit": UNIT,
                     "ms_per_step": ms_sus / n_sus, "clocks": smp.summary() if rank == 0 else None}
    # BASELINE config 4: 256 frames per GPU
    c4 = None
    if a.c4_batch > 0 and a.c4_batch != B:
        B4 = a.c4_batch
        x4 = torch.rand(B4, 3, S, S, device=dev, generator=gen)
        x4_host = (torch.rand(B4, 3, S, S, generator=torch.Generator().manual_seed(400 + rank)) * 255).to(torch.uint8).pin_memory()
        k4 = max(3, a.steps // 4)
        for _ in range(2):
            model.predict_batched(x4, CONF, IOU, MAX_DET)
        ms4 = timed(lambda: model.predict_batched(x4, CONF, IOU, MAX_DET), k4)
        run_stream(2, x4_host)
        ms4_e2e = min(timed(lambda: run_stream(k4, x4_host), 1) for _ in range(2))
        c4 = {"batch_per_gpu": B4, "steps": k4, "value": world * B4 * k4 / (ms4 * 1e-3), "unit": UNIT, "ms_per_step": ms4 / k4,
              "e2e": {"value": world * B4 * k4 / (ms4_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms4_e2e / k4,
                      "h2d_bytes_per_step": x4_host.numel(), "d2h_bytes_per_step": B4 * (MAX_DET * 6 + 1) * 4}}
        del x4, x4_host
        model._stream_state.clear()
        torch.cuda.empty_cache()

    # stage split of one resident step and batch-1 latency (p50 over 50 synchronised calls)
    def span(fn, reps=5):
        fn()  # warm-up: the first call may grow the caching allocator
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    y_keep = model.forward(x_dev, raw_heads=False)
    ms_fwd_decode = span(lambda: model.forward(x_dev, raw_heads=False))
    ms_stack = span(lambda: plan.run(x_dev, y_prof if plan.fused else None))
    ms_nms = span(lambda: model.nms(y_keep, CONF, IOU, MAX_DET))
    x1 = x_dev[:1].contiguous()
    for _ in range(5):
        model.predict_batched(x1, CONF, IOU, MAX_DET)
    lat = []
    for _ in range(50):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.predict_batched(x1, CONF, IOU, MAX_DET)
        torch.cuda.synchronize()
        lat.append((time.perf_counter() - t0) * 1e3)
    lat.sort()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    top_ms = top_ms_total / max(top_n, 1)
    tensor_bound = top_flops / max(top_bytes, 1.0) > 100.0  # FLOP/B well above 1: judged on the tensor pipe
    if tensor_bound:
        achieved, peak, unit = top_flops * B / (top_ms * 1e-3) / 1e12, pk["tflops"], "TFLOP/s"
    else:
        achieved, peak, unit = top_bytes * B / (top_ms * 1e-3) / 1e9, pk["hbm_gbs"], "GB/s"
    traffic = None
    tj = ROOT / "profiles" / "roofline_traffic.json"
    if tj.exists():
        traffic = json.loads(tj.read_text()).get(top_text)
    # conv stack (+ DFL decode per level when the plan does not decode in its head kernels) + the fused NMS kernel
    kernels_per_step = plan.launches + (0 if plan.fused else len(plan.heads)) + 1
    conv_flops = sum(plan.op_info(i)[1] for i in range(plan.launches))
    out = {
        "metric": METRIC, "value": world * B * a.steps / (ms_total * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
        "warmup": warm, "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"unina-yolo-dla-m bf16 forward + DFL decode + NMS, {S}x{S}, batch {B} per GPU",
                   "global_batch": world * B, "parallelism": f"dp{world}", "conf": CONF, "iou": IOU, "max_det": MAX_DET,
                   "candidates_per_image_target": CANDIDATES_PER_IMAGE, "detections_last_step": n_det,
                   "weights": "seeded synthetic (init_synthetic seed 0)",
                   "l2": f"inputs larger than L2 ({x_dev.numel() * 4 / 1e6:.0f} MB fp32 frames + {plan.bytes / 1e6:.0f} MB activations per step)",
                   "conv_gflop_per_image": conv_flops / 1e9},
        "e2e": {"value": world * B * a.steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": x_host.numel(),
                "d2h_bytes_per_step": det_host.numel() * 4 + cnt_host.numel() * 4, "ms_per_step": ms_e2e / a.steps,
                "single_call_ms": ms_e2e_single / a.steps,
                "frac_of_h2d_cap": (world * B * a.steps / (ms_e2e * 1e-3)) / probe["h2d_cap_images_per_s"],
                "api": "UninaYoloB200.predict_stream(pinned uint8 NCHW host batches): H2D of step i+1 overlaps step i (best of 3 runs of K steps); "
                       "N > 1: + one fixed-shape NCCL all_gather of the detections per step on a side stream; "
                       "single_call_ms = one blocking predict_batched(host frames) per step",
                "bound_probe": dict(probe, note="the same streamed run with the gather (N > 1) or the H2D copy switched off, and the H2D copies "
                                                "alone on all ranks at once: e2e ms_per_step ~ max(resident step, h2d_only) means the "
                                                "host-to-device path of the box bounds e2e")},
        "e2e_nv12": {"value": world * B * a.steps / (ms_nv12 * 1e-3), "unit": UNIT, "ms_per_step": ms_nv12 / a.steps,
                     "h2d_bytes_per_step": nv_host.numel(), "d2h_bytes_per_step": det_host.numel() * 4 + cnt_host.numel() * 4,
                     "api": "predict_stream(camera='nv12'): pinned host NV12 frames (Y rows + interleaved UV rows) -> H2D -> the stem reads the "
                            "planes itself (uyd_plan_run_camera) -> decode -> NMS -> D2H (+ gather at N > 1); an additional record, "
                            "the headline e2e stays on uint8 NCHW frames"},
        "resident_stream": {"value": world * B * a.steps / (ms_pipe * 1e-3), "unit": UNIT, "ms_per_step": ms_pipe / a.steps,
                            "api": "predict_stream on device-resident frames: the same K steps, the per-image NMS kernel (one SM per frame) of "
                                   "step i on a second stream under the forward of step i + 1"},
        "gpu_launches": kernels_per_step * a.steps,
        "roofline": {"kernel": top_text, "bound": "tensor" if tensor_bound else "hbm", "achieved": achieved, "peak": peak,
                     "unit": unit, "frac": achieved / peak, "traffic": traffic, "peak_source": pk["src"],
                     "avg_launch_ms": top_ms, "launches_timed": top_n,
                     "share_of_conv_stack": ms[top] / sum(ms),
                     "families": family_table(plan, ms, B, pk, ms_nms)},
        "conv_stack": {"ms_per_step_profiled": sum(ms), "tflops": conv_flops * B / (sum(ms) * 1e-3) / 1e12,
                       "frac_of_tensor_peak": conv_flops * B / (sum(ms) * 1e-3) / 1e12 / pk["tflops"]},
        "stages_ms": {"conv_stack": ms_stack, "dfl_decode": ms_fwd_decode - ms_stack, "nms": ms_nms,
                      "note": "fused plan: the DFL decode runs inside the head kernels (conv_stack includes it)" if plan.fused else ""},
        "latency_bs1_ms": {"p50": lat[len(lat) // 2], "min": lat[0], "p90": lat[int(len(lat) * 0.9)], "calls": len(lat),
                           "note": "predict_batched on one resident frame (CUDA-graph replay), host-synchronised wall clock"},
        "clocks": sampler.summary(),
    }
    if sustained:
        out["sustained"] = sustained
    if c4:
        out["c4_batch256"] = c4
    if world == 1:
        if a.stress > 0:
            out["nms_stress_1280"] = bench_nms_stress(model, a.stress, dev, max(3, a.steps // 2))
        if a.int8 > 0:
            out["int8"] = bench_int8(model, a.int8, S, dev, max(3, a.steps // 4))
        model._plans.clear() if hasattr(model, "_plans") else None
        torch.cuda.empty_cache()
        if a.custom > 0:
            out["custom_variant"] = bench_custom(a.custom, S, dev, max(3, a.steps // 2), pk,
                                                 a.profile_out.replace(".md", "_custom.md") if a.profile_out else "")
        if a.cpu_sample > 0:   # 0 only in the A/B tooling (tools/gpu_ab.sh); the driver's default run always carries it
            out["cpu_baseline"] = cpu_baseline(model, S, a.cpu_sample)
    if a.profile_out:
        rows = ["| # | op | ms | share | TFLOP/s | GB/s |", "|---|---|---|---|---|---|"]
        for i in sorted(range(len(ms)), key=lambda i: -ms[i]):
            t, fl, by = plan.op_info(i)
            rows.append(f"| {i} | {t} | {ms[i]:.4f} | {100 * ms[i] / sum(ms):.1f}% | {fl * B / (ms[i] * 1e-3) / 1e12:.1f} | {by * B / (ms[i] * 1e-3) / 1e9:.0f} |")
        Path(a.profile_out).write_text(f"per-op CUDA-event times, batch {B}, {S}x{S} (one pass, ops serialised)\n\n" + "\n".join(rows) + "\n")
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
