"""Letterboxed camera frames on one GPU, both networks: predict_camera(letterbox=True) against the stretch path at the
same plan extent (predict_camera without letterbox: the same convs, only the loader differs) and against the path a
user takes without this feature (cv2 letterbox on the host, H2D copy, predict_batched, boxes still in model-input
pixels).  Batch 64 of seeded 1280 x 720 BGRA frames resident on the device (236 MB: larger than L2), plan extents
384 x 640 (the predictor's rectangular choice) and 640 x 640.  Records, with the card's name, power limit and SM clock
read in the same run:
  * predict_camera step times, CUDA events over back-to-back eager steps, letterbox and stretch alternated over rounds;
  * the user path split into host CPU time (cv2.resize + copyMakeBorder of 64 frames into pinned memory, host clock)
    and the device part (H2D of the letterboxed bytes, the network's input conversion, predict_batched; host clock
    ended by a synchronise);
  * outputs_byte_equal: predict_camera(letterbox=True) rows against the user path's rows mapped back with the torch
    scale_boxes statements;
  * uyd_letterbox_boxes alone on [64, max_det, 6] with every row counted: CUDA events over many launches, replayed from
    a CUDA graph (the kernel) and issued one by one from Python (what a Python caller pays per call).
Writes <out>/letterbox_bench.json.  Usage: python tools/letterbox_bench.py --out DIR"""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import unina_yolo_dla_b200 as uyd  # noqa: E402
from unina_yolo_dla_b200 import preprocess  # noqa: E402

W0, H0, B = 1280, 720, 64
PLANS = [(384, 640), (640, 640)]


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi name, power.limit, clocks.sm, clocks.max.sm":
            q.stdout.strip() or q.stderr.strip()}


def host_ms(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def event_ms(fn, steps):
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


def scale_boxes_torch(det, cnt, h0, w0, H, W):
    """Ultralytics scale_boxes + clip_boxes on each image's first count rows, with torch on the device."""
    out = det.clone()
    gain = min(H / h0, W / w0)
    pad = (round((W - w0 * gain) / 2 - 0.1), round((H - h0 * gain) / 2 - 0.1))
    for b, n in enumerate(cnt.tolist()):
        bx = out[b, :n]
        bx[..., 0] -= pad[0]
        bx[..., 1] -= pad[1]
        bx[..., 2] -= pad[0]
        bx[..., 3] -= pad[1]
        bx[..., :4] /= gain
        bx[..., 0].clamp_(0, w0)
        bx[..., 1].clamp_(0, h0)
        bx[..., 2].clamp_(0, w0)
        bx[..., 3].clamp_(0, h0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--box-launches", type=int, default=2000)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("letterbox_bench.py measures on a GPU; none is visible")
    import cv2

    torch.cuda.set_device(0)
    g = torch.Generator().manual_seed(1234)
    low = torch.rand(B, 4, H0 // 32, W0 // 32, generator=g)
    img = 0.7 * torch.nn.functional.interpolate(low, size=(H0, W0), mode="bilinear", align_corners=False)
    frames_h = ((img + 0.3 * torch.rand(B, 4, H0, W0, generator=g)) * 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    frames = frames_h.cuda()
    frames_np = frames_h.numpy()
    res = {"card": card(), "batch": B, "frame": [H0, W0], "frames": "smooth + noise BGRA, seeded 1234, resident on the device",
           "cv2": cv2.__version__, "networks": {}}
    nets = {"yaml": (uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0).cuda(), dict(conf=0.25, iou=0.7)),
            "custom_bc32": (uyd.UninaCustomB200(4, 32).init_synthetic(seed=0).cuda(), dict(conf=0.5, iou=0.45, graph=False))}
    for name, (m, kw) in nets.items():
        rows = {}
        for H, W in PLANS:
            nw, nh, left, top, _ = preprocess.letterbox_geometry(H0, W0, H, W)
            staged = torch.empty(B, H, W, 4, dtype=torch.uint8).pin_memory()
            staged_np = staged.numpy()
            dev = torch.empty(B, H, W, 4, dtype=torch.uint8, device="cuda")

            def host_letterbox():
                for i in range(B):
                    r = cv2.resize(frames_np[i], (nw, nh), interpolation=cv2.INTER_LINEAR)
                    staged_np[i] = cv2.copyMakeBorder(r, top, H - nh - top, left, W - nw - left, cv2.BORDER_CONSTANT,
                                                      value=(114, 114, 114, 114))

            def device_part():
                dev.copy_(staged, non_blocking=True)
                if name == "yaml":
                    x = dev[..., [2, 1, 0]].permute(0, 3, 1, 2).contiguous()   # RGB NCHW uint8, the network's u8 input
                else:
                    x = preprocess.bgra(dev, preprocess.norm_params())           # ImageNet fp32, as predict_camera's default
                return m.predict_batched(x, **kw)

            lbox = lambda: m.predict_camera(frames, size=(H, W), letterbox=True, **kw)
            stretch = lambda: m.predict_camera(frames, size=(H, W), **kw)
            for _ in range(3):
                lbox()
                stretch()
                host_letterbox()
                device_part()
            d0, c0 = device_part()
            want = scale_boxes_torch(d0, c0, H0, W0, H, W)
            d1, c1 = lbox()
            row = {"outputs_byte_equal": bool(torch.equal(c0, c1) and torch.equal(want, d1)),
                   "kept_per_image_mean": float(c1.float().mean())}
            tl, ts, th, td = [], [], [], []
            for _ in range(a.rounds):
                tl.append(event_ms(lbox, a.steps))
                ts.append(event_ms(stretch, a.steps))
                t0 = time.perf_counter()
                host_letterbox()
                th.append((time.perf_counter() - t0) * 1e3)
                td.append(host_ms(device_part))
            row.update({"predict_camera_letterbox_ms": med(tl), "predict_camera_stretch_ms": med(ts),
                        "letterbox_minus_stretch_ms": med(tl) - med(ts),
                        "user_path_host_cpu_cv2_letterbox_ms": med(th), "user_path_device_h2d_predict_batched_ms": med(td),
                        "user_path_total_ms": med(th) + med(td),
                        "letterbox_rounds_ms": tl, "stretch_rounds_ms": ts, "host_cv2_rounds_ms": th, "device_part_rounds_ms": td})
            rows[f"{H}x{W}"] = row
            del staged, dev
        res["networks"][name] = rows
    boxes = {}
    for max_det in (300, 1024):
        det = torch.rand(B, max_det, 6, device="cuda") * 640
        cnt = torch.full((B,), max_det, dtype=torch.int32, device="cuda")
        call = lambda: preprocess.letterbox_boxes(det, cnt, H0, W0, 384, 640)
        for _ in range(10):
            call()
        # device time: 100 launches captured in one CUDA graph (a launch from Python costs more host time than the kernel)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for _ in range(100):
                call()
        graph.replay()
        boxes[f"64x{max_det}"] = {
            "us_per_launch_graph": med([event_ms(graph.replay, a.box_launches // 100) for _ in range(3)]) * 1e3 / 100,
            "us_per_call_from_python": med([event_ms(call, a.box_launches) for _ in range(3)]) * 1e3}
    res["uyd_letterbox_boxes"] = boxes
    res["note"] = (f"predict_camera: CUDA events over {a.steps} back-to-back eager steps, median of {a.rounds} rounds with "
                   "letterbox and stretch alternated; user path: host clock, median of the same rounds, host CPU part = cv2 "
                   "letterbox of all 64 frames into pinned memory, device part = H2D + input conversion + predict_batched "
                   "ended by a synchronise (its rows are still in model-input pixels); uyd_letterbox_boxes: CUDA events over "
                   f"{a.box_launches} launches replayed from CUDA graphs of 100 (device time) and issued one by one from "
                   "Python (host-bound), median of 3")
    res["card_after"] = card()
    out = Path(a.out)
    out.mkdir(parents=True, exist_ok=True)
    (out / "letterbox_bench.json").write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps({k: v for k, v in res.items()}, indent=1))


if __name__ == "__main__":
    main()
