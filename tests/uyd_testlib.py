"""Helpers shared by the GPU parity tests and tools/gpu_probe.py."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

import unina_yolo_dla_b200 as uyd
from unina_yolo_dla_b200 import _lib
from unina_yolo_dla_b200._lib import IMPL_AUTO, IMPL_DIRECT, IMPL_TC, UYD_BF16, UYD_F32  # noqa: F401

_DT = {UYD_BF16: torch.bfloat16, UYD_F32: torch.float32}


def bf16_round(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).float()


class Canary:
    """Fills every buffer of a finalized plan (all max_batch images, all channels, bf16 and fp32 alike) with seeded
    finite values, |v| <= 8, so that a kernel reading outside its input slice reads real-looking data, not zeros.
    ``snapshot()`` after the inputs are written, ``check(outputs, batch)`` after the run: every element outside
    the output slices (other channels, images >= batch, other buffers) must still hold its value."""

    def __init__(self, plan, seed=1234):
        self.plan = plan
        g = torch.Generator().manual_seed(seed)
        for buf, (h, w, c, dtype) in plan.shapes.items():
            v = ((torch.rand(plan.max_batch, h, w, c, generator=g) * 16 - 8)).to(_DT[dtype])
            self._copy(buf, v.cuda(plan.device), to_plan=True)
        torch.cuda.synchronize()
        self.before = None

    def _copy(self, buf, t, to_plan):
        ptr = C.c_void_p()
        _lib.check(_lib.lib().uyd_plan_buffer_ptr(self.plan.handle, buf, C.byref(ptr)), "uyd_plan_buffer_ptr")
        src, dst = (C.c_void_p(t.data_ptr()), ptr) if to_plan else (ptr, C.c_void_p(t.data_ptr()))
        _lib.check(_lib.lib().uyd_memcpy_d2d(dst, src, t.numel() * t.element_size(), self.plan._stream()), "uyd_memcpy_d2d")

    def raw(self, buf):
        h, w, c, dtype = self.plan.shapes[buf]
        t = torch.empty(self.plan.max_batch, h, w, c, dtype=_DT[dtype], device=f"cuda:{self.plan.device}")
        self._copy(buf, t, to_plan=False)
        torch.cuda.synchronize()
        return t.cpu()

    def snapshot(self):
        self.before = {b: self.raw(b) for b in self.plan.shapes}

    def check(self, outputs, batch):
        for b, old in self.before.items():
            new = self.raw(b)
            keep = torch.ones(old.shape, dtype=torch.bool)
            for s in outputs:
                if s.buf == b:
                    keep[:batch, :, :, s.coff:s.coff + s.c] = False
            changed = (new != old) & keep
            assert not bool(changed.any()), f"buffer {b}: {int(changed.sum())} elements outside the output slices " \
                f"changed, first at (n, y, x, c) = {tuple(int(i) for i in changed.nonzero()[0])}"


def launched(fn):
    """Runs fn once under torch.profiler and returns the ids (fp64ref.kernel_id) of the CUDA kernels it launched, plus
    "grid:<id>:<x>,<y>,<z>" for each launch's grid (runtime variants such as a tile height show only there)."""
    import json
    import tempfile

    from torch.profiler import ProfilerActivity, profile

    import fp64ref

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        prof.export_chrome_trace(f"{d}/trace.json")
        with open(f"{d}/trace.json") as f:
            events = json.load(f)["traceEvents"]
    out = set()
    for e in events:
        if e.get("cat") == "kernel":
            k = fp64ref.kernel_id(e["name"])
            out |= {k, f"grid:{k}:" + ",".join(str(v) for v in e.get("args", {}).get("grid", []))}
    return out


def run_canaried(p, writes, outputs, batch, run=None, kernels=None):
    """Runs a finalized plan on canary-filled buffers: ``writes`` = [(slice, NCHW tensor)], ``run`` defaults to
    run_no_input(batch).  Checks that only ``outputs`` changed; returns them read back as NCHW fp32."""
    can = Canary(p)
    for s, t in writes:
        p.write(s, t)
    can.snapshot()
    names = launched(run or (lambda: p.run_no_input(batch)))
    if kernels is not None:
        kernels |= names
    can.check(outputs, batch)
    return [p.read(s, batch).cpu() for s in outputs]


def run_single_conv(cin, cout, k, stride, H, W, batch=2, impl=IMPL_AUTO, relu=True, residual=False, depthwise=False,
                    in_total=None, in_coff=0, out_total=None, out_coff=0, out_f32=False, seed=0, max_batch=None,
                    kernels=None):
    """Builds a one-conv plan on canary-filled buffers, runs it, checks that nothing outside the output slice
    changed and returns (got NCHW fp32, fp64 reference, per-element slack) on the same bf16-rounded operands.
    ``kernels``: a set that receives the ids of the kernels the run launched and "op_info:<the op's text>"."""
    import fp64ref

    g = torch.Generator().manual_seed(seed)
    in_total = in_total or cin
    out_total = out_total or cout
    x = torch.randn(batch, cin, H, W, generator=g)
    wshape = (cout, 1, k, k) if depthwise else (cout, cin, k, k)
    w = torch.randn(*wshape, generator=g) / (wshape[1] * k * k) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    oh, ow = (H + 2 * (k // 2) - k) // stride + 1, (W + 2 * (k // 2) - k) // stride + 1
    r = torch.randn(batch, cout, oh, ow, generator=g) if residual else None

    p = uyd.Plan(0, max_batch or batch)
    src = p.buffer(H, W, in_total)
    dst = p.buffer(oh, ow, out_total, UYD_F32 if out_f32 else UYD_BF16)
    rs = p.buffer(oh, ow, cout) if residual else None
    s_in, s_out = src.sub(in_coff, cin), dst.sub(out_coff, cout)
    p.conv(s_in, s_out, w.numpy(), b.numpy(), k, stride, relu=relu, depthwise=depthwise, res=rs, impl=impl)
    p.finalize()
    got, = run_canaried(p, [(s_in, x)] + ([(rs, r)] if residual else []), [s_out], batch, kernels=kernels)
    if kernels is not None:
        kernels.add("op_info:" + p.op_info(0)[0])
    # the fp64 reference runs on the device: the same exact arithmetic, minutes less CPU time for the large cases
    dev = lambda t: None if t is None else t.to("cuda", torch.float64)
    ref, slack = fp64ref.conv(dev(bf16_round(x)), dev(bf16_round(w)), dev(b), stride=stride, groups=cin if depthwise else 1,
                              relu=relu, res=dev(bf16_round(r)) if residual else None, bf16_out=not out_f32)
    return got, ref.cpu(), slack.cpu()


def rel_err(got: torch.Tensor, ref: torch.Tensor) -> float:
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-12))


def synth_predictions(B, nc, A, seed=0, frac_conf=0.2, img=640.0, cluster=False):
    """Synthetic y[B,4+nc,A] with overlapping boxes and a controllable share above conf."""
    rng = np.random.default_rng(seed)
    y = np.zeros((B, 4 + nc, A), np.float32)
    if cluster:
        centers = rng.uniform(40, img - 40, (B, 2, 64))
        pick = rng.integers(0, 64, (B, A))
        cxy = np.take_along_axis(centers, pick[:, None, :].repeat(2, 1), 2) + rng.normal(0, 6, (B, 2, A))
    else:
        cxy = rng.uniform(0, img, (B, 2, A))
    y[:, 0:2] = cxy
    y[:, 2:4] = rng.uniform(8, 96, (B, 2, A))
    sc = rng.uniform(0, 1, (B, nc, A)).astype(np.float32)
    lift = rng.uniform(0, 1, (B, 1, A)) < frac_conf
    y[:, 4:] = np.where(lift, 0.25 + 0.75 * sc, 0.2 * sc)
    return y
