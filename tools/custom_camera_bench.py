"""Camera frames into the model.py network (UninaCustomB200) on one GPU: the two-step path (uyd_preprocess_* into a
reused fp32 NCHW tensor, then predict_batched) against predict_camera (the stem reads the camera bytes itself).  Three
formats: BGRA 640x640, BGRA 1280x720 resized to 640x640, NV12 640x640.  Records, with the card's name and power limit
read in the same run:
  * batch 64: step time of both paths (CUDA events over back-to-back steps, eager launches, old and new alternated
    over several rounds), and the pre-processing launches alone, which is the part of the saving that comes from the
    removed kernel; the rest is the stem reading bytes instead of fp32;
  * batch 1: host-clock p50 / min per call ended by a synchronise, CUDA-graph replay of the network + NMS on both sides
    (the two-step path launches its pre-processing kernel before the replay);
  * outputs_byte_equal for BGRA at the model's extent (detections and counts of both paths at batch 64).
Every shape is warmed up before it is timed; frames are seeded.  Writes <out>/custom_camera_bench.json.
Usage: python tools/custom_camera_bench.py --out DIR [--bc 32]"""
import argparse
import ctypes as C
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import unina_yolo_dla_b200 as uyd  # noqa: E402
from unina_yolo_dla_b200 import _lib, preprocess  # noqa: E402

S = 640
FORMATS = {"bgra_640": ("bgra", 640, 640), "bgra_1280x720": ("bgra", 720, 1280), "nv12_640": ("nv12", 640, 640)}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() or q.stderr.strip()}


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


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
    v = sorted(v)
    return v[len(v) // 2]


def inputs(fmt, B, gen):
    kind, h, w = FORMATS[fmt]
    if kind == "bgra":
        return torch.randint(0, 256, (B, h, w, 4), generator=gen, dtype=torch.uint8, device="cuda"), None
    y = torch.randint(0, 256, (B, h, w), generator=gen, dtype=torch.uint8, device="cuda")
    uv = torch.randint(0, 256, (B, h // 2, w), generator=gen, dtype=torch.uint8, device="cuda")
    return y, uv


def preprocess_into(fmt, frames, uv, out, norm):
    """The node's pre-processing kernels into the reused fp32 tensor `out` (one launch per batch, NV12: per frame)."""
    L = _lib.lib()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    kind, h, w = FORMATS[fmt]
    B = frames.shape[0]
    if kind == "bgra" and (h, w) == (S, S):
        _lib.check(L.uyd_preprocess_bgra_batch(C.c_void_p(frames.data_ptr()), C.c_void_p(out.data_ptr()), B, h * w * 4, w, h, w * 4,
                                               norm, st), "uyd_preprocess_bgra_batch")
    elif kind == "bgra":
        _lib.check(L.uyd_preprocess_bgra_resize_batch(C.c_void_p(frames.data_ptr()), C.c_void_p(out.data_ptr()), B, h * w * 4, w, h,
                                                      w * 4, S, S, norm, st), "uyd_preprocess_bgra_resize_batch")
    else:
        for b in range(B):
            _lib.check(L.uyd_preprocess_nv12(C.c_void_p(frames[b].data_ptr()), C.c_void_p(uv[b].data_ptr()),
                                             C.c_void_p(out[b].data_ptr()), w, h, w, w, norm, st), "uyd_preprocess_nv12")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--bc", type=int, default=32)
    ap.add_argument("--conf", type=float, default=0.5)
    ap.add_argument("--iou", type=float, default=0.45)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--bs1-calls", type=int, default=200)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("custom_camera_bench.py measures on a GPU; none is visible")
    torch.cuda.set_device(0)
    m = uyd.UninaCustomB200(4, a.bc).init_synthetic(seed=0).cuda()
    norm = preprocess.norm_params()
    gen = torch.Generator(device="cuda").manual_seed(900)
    res = {"card": card(), "network": f"UninaCustomB200(num_classes=4, base_channels={a.bc})", "model_input": [S, S],
           "conf": a.conf, "iou": a.iou, "norm": "ImageNet", "frames": "torch.randint seeded 900 on the device, uint8",
           "batch64": {}, "batch1": {}}
    kw = dict(conf=a.conf, iou=a.iou)
    for fmt in FORMATS:
        kind = FORMATS[fmt][0]
        size = None if kind == "nv12" else (S, S)
        # ---- batch 64: CUDA events over back-to-back steps, old and new alternated ----
        B = 64
        frames, uv = inputs(fmt, B, gen)
        x = torch.empty(B, 3, S, S, device="cuda")
        pre = lambda: preprocess_into(fmt, frames, uv, x, norm)
        old = lambda: (pre(), m.predict_batched(x, graph=False, **kw))
        new = lambda: m.predict_camera(frames, size=size, norm=norm, uv=uv, graph=False, **kw)
        for _ in range(3):
            old()
            new()
        row = {}
        if fmt == "bgra_640":
            pre()
            d0, c0 = m.predict_batched(x, graph=False, **kw)
            d1, c1 = new()
            row["outputs_byte_equal"] = bool(torch.equal(d0, d1) and torch.equal(c0, c1))
            row["kept_per_image_mean"] = float(c1.float().mean())
        to, tn, tp = [], [], []
        for _ in range(a.rounds):
            to.append(event_ms(old, a.steps))
            tn.append(event_ms(new, a.steps))
            tp.append(event_ms(pre, a.steps))
        row.update({"two_step_ms": med(to), "predict_camera_ms": med(tn), "saving_ms": med(to) - med(tn),
                    "preprocess_alone_ms": med(tp), "stem_share_of_saving_ms": med(to) - med(tn) - med(tp),
                    "two_step_rounds_ms": to, "predict_camera_rounds_ms": tn})
        res["batch64"][fmt] = row
        del frames, uv, x
        # ---- batch 1: host clock, graph replay on both sides, alternated ----
        frames, uv = inputs(fmt, 1, gen)
        x = torch.empty(1, 3, S, S, device="cuda")
        old1 = lambda: (preprocess_into(fmt, frames, uv, x, norm), m.predict_batched(x, graph=True, **kw))
        new1 = lambda: m.predict_camera(frames, size=size, norm=norm, uv=uv, graph=True, **kw)
        for _ in range(10):
            old1()
            new1()
        lo, ln = [], []
        for _ in range(a.bs1_calls):
            lo.append(host_ms(old1))
            ln.append(host_ms(new1))
        lo.sort()
        ln.sort()
        res["batch1"][fmt] = {"two_step": {"p50": med(lo), "min": lo[0]}, "predict_camera": {"p50": med(ln), "min": ln[0]}}
    res["batch64_note"] = (f"CUDA events over {a.steps} back-to-back steps, median of {a.rounds} alternated rounds; two_step = "
                           "uyd_preprocess_* into a reused fp32 tensor + predict_batched(graph=False); NV12 pre-processing is one "
                           "launch per frame (uyd_preprocess_nv12 takes one frame)")
    res["batch1_note"] = (f"host clock per call ended by a synchronise, {a.bs1_calls} calls each, alternated; both return "
                          "(det, count) on the device")
    res["card_after"] = card()
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "custom_camera_bench.json").write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
