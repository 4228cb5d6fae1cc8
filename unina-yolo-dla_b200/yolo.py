"""``UninaYoloB200``: the YAML-built detector (reference: ``DetectionModel(cfg, nc)`` after
``apply_dla_patches`` + ``replace_silu_with_relu``, trainer.py:31-136,146-158) as a drop-in
``nn.Module`` whose forward runs entirely through libuyd's CUDA plan.

Same construction from ``unina-yolo-dla-m.yaml`` (unina-yolo-dla-m.yaml:14-62), same
``state_dict`` keys/shapes (925 entries), same eval output ``(y[B,4+nc,A], [x_l])`` and
``predict`` -> per-image ``[N,6]`` rows ``(x1,y1,x2,y2,conf,cls)`` (train.py:396-423,
trainer.py:237-240).  The modules below only *hold* parameters under the reference's names and
know how to emit themselves into a plan; they never compute with torch.
"""
from __future__ import annotations

import ast
import ctypes as C
import math
import operator
import os
from math import gcd
from pathlib import Path

import numpy as np
import torch
import torch.nn as nn
import yaml

from . import _lib
from ._lib import CHAIN_DFL, CHAIN_PW3, CHAIN_STORE, UYD_BF16, UYD_F32, UYD_S8, check
from . import preprocess as P
from . import quant as Q
from .plan import NETWORK_INPUT, Plan, Slice, fold_bn

DEFAULT_YAML = Path(__file__).resolve().parent / "unina-yolo-dla-m.yaml"


class _NoFuse(Exception):
    """The decode cannot be folded into the head kernels for this graph / shape."""


def _make_divisible(x, d):
    return int(math.ceil(x / d) * d)


class Conv(nn.Module):
    """Conv2d(bias=False) + BatchNorm2d(eps 1e-3) + ReLU, parameters under ``conv.*`` / ``bn.*``."""

    def __init__(self, c1, c2, k=1, s=1, g=1):
        super().__init__()
        self.conv = nn.Conv2d(c1, c2, k, s, k // 2, groups=g, bias=False)
        self.bn = nn.BatchNorm2d(c2, eps=1e-3, momentum=0.03)
        self.act = nn.ReLU(inplace=True)
        self.k, self.s, self.g, self.c1, self.c2 = k, s, g, c1, c2

    def emit(self, p: Plan, src: Slice, dst: Slice | None = None, res: Slice | None = None, feeds: nn.Conv2d | None = None,
             feeds_f32: bool = False) -> Slice:
        """``feeds``: the conv that is the ONLY consumer of this output (the caller owns that knowledge).  In the INT8
        graph such an output is written directly as the consumer's int8 input (no bf16 tensor, no quantize launch);
        ``feeds_f32``: that consumer writes into an fp32 head buffer (its tensor-core eligibility rule differs)."""
        oh, ow = (p.in_hw[0] // self.s, p.in_hw[1] // self.s) if src.buf < 0 else (
            (src.h + 2 * (self.k // 2) - self.k) // self.s + 1, (src.w + 2 * (self.k // 2) - self.k) // self.s + 1)
        dst_was_none = dst is None
        name = getattr(self.conv, "_uyd_name", "")
        private_s8 = (dst_was_none and feeds is not None and src.buf >= 0 and _quantized(p, name)
                      and _quantized(p, getattr(feeds, "_uyd_name", "")) and os.environ.get("UYD_INT8_NO_DIRECT", "0") != "1")
        if dst is None and not private_s8:
            dst = p.buffer(oh, ow, self.c2)
        dw = self.g > 1
        assert not dw or self.g == self.c1 == self.c2, "only depth-wise grouped convs occur in this graph"
        _record_input(p, name, src)
        if _quantized(p, name) and src.buf >= 0:
            return emit_quant_conv(p, name, self.conv, self.bn, src, dst, relu=True, res=res, feeds=feeds if private_s8 else None,
                                   feeds_f32=feeds_f32)
        w, b = fold_bn(self.conv, self.bn)
        return p.conv(src, dst, w, b, self.k, self.s, relu=True, depthwise=dw, res=res)


def DWConv(c1, c2, k=1, s=1):
    return Conv(c1, c2, k, s, g=gcd(c1, c2))


def _quantized(p, name: str) -> bool:
    q = getattr(p, "quant", None)
    return q is not None and q.covers(name)


def _record_input(p, name: str, src: Slice) -> None:
    rec = getattr(p, "conv_inputs", None)
    if rec is not None and name:
        rec[name] = src


def _tc_rows(cout: int, dst_f32: bool) -> bool:
    """Output rows the tcgen05 int8 kernel can store (a power-of-two number of 16-byte lanes)."""
    return (cout >= 8 and cout & (cout - 1) == 0) or (cout == 4 and dst_f32)


def _s8_width(c: int, tc_rows: bool) -> int:
    """Channels of the int8 copy a quantised conv reads: padded with zero channels to a multiple of 32 for tcgen05."""
    if tc_rows and os.environ.get("UYD_INT8_NO_PAD", "0") != "1":
        return (c + 31) // 32 * 32
    return c


def _s8_copy(p: Plan, src: Slice, scale: float, cpad: int) -> Slice:
    """The int8 copy of a bf16 activation slice for input scale ``scale``, ``cpad`` channels wide (zero pad channels):
    one copy per (slice, scale, width), shared by the convs that agree on them."""
    cache = p.__dict__.setdefault("_qcache", {})
    key = (src.buf, src.coff, src.c, scale, cpad)
    q = cache.get(key)
    if q is None:
        q = p.buffer(src.h, src.w, cpad, UYD_S8)          # zero-filled at finalize: the pad channels stay zero
        p.quantize(src, q.sub(0, src.c), scale)
        cache[key] = q
    return q


def emit_quant_conv(p: Plan, name: str, conv: nn.Conv2d, bn, src: Slice, dst: Slice | None, relu: bool, res: Slice | None = None,
                    feeds: nn.Conv2d | None = None, feeds_f32: bool = False) -> Slice:
    """QuantConv2d as an integer convolution (quant.py): input quantiser -> int8 conv -> requant epilogue.
    ``src`` in a UYD_S8 buffer = the producer already wrote this conv's int8 input (see ``feeds``).
    ``feeds`` (with ``dst`` None): this conv's output is consumed by that quantised conv only; it is written as ITS int8
    input -- y rounded to bf16 (the activation the graph defines), times its input scale, rounded, clamped: the very
    bytes ``quantize`` would produce from the bf16 tensor, which is never materialised."""
    ax, aw = p.quant.amax[name]
    scale = float(Q.scale_of(ax))
    qw = Q.quantize_weights(conv.weight, aw)
    mult, bias = Q.requant_params(ax, aw, bn, conv.bias)
    cout, dw = qw.shape[0], conv.groups > 1
    # tensor-core (tcgen05 kind::i8) eligibility is a matter of layout, not of arithmetic (the int32 sums are
    # exact either way): the int8 copy of the input is ours, so it is padded with zero channels to a multiple
    # of 32, and a depth-wise conv runs as a dense conv with diagonal weights.
    dst_f32 = dst is not None and p.shapes[dst.buf][3] == UYD_F32
    tc_rows = _tc_rows(cout, dst_f32)
    cpad = _s8_width(src.c, tc_rows)
    s8_in = p.shapes[src.buf][3] == UYD_S8
    if s8_in:
        pscale, pwidth = p._s8_direct[src.buf]
        assert pscale == scale and pwidth == cpad and src.coff == 0, "direct int8 input: producer / consumer disagree"
    if tc_rows and os.environ.get("UYD_INT8_NO_PAD", "0") != "1":
        if dw:
            dense = np.zeros((cout, cpad, qw.shape[2], qw.shape[3]), np.int8)
            dense[np.arange(cout), np.arange(cout)] = qw[:, 0]
            qw, dw = dense, False
        elif cpad != src.c:
            qw = np.concatenate((qw, np.zeros((cout, cpad - src.c, qw.shape[2], qw.shape[3]), np.int8)), 1)
    if s8_in:
        qsrc = Slice(src.buf, 0, cpad, src.h, src.w)
    else:
        qsrc = _s8_copy(p, src, scale, cpad)
    k, st = conv.kernel_size[0], conv.stride[0]
    if feeds is not None and dst is None:
        fname = feeds._uyd_name
        fscale = float(Q.scale_of(p.quant.amax[fname][0]))
        fwidth = _s8_width(cout, _tc_rows(feeds.out_channels, feeds_f32))
        oh, ow = (src.h + 2 * (k // 2) - k) // st + 1, (src.w + 2 * (k // 2) - k) // st + 1
        obuf = p.buffer(oh, ow, fwidth, UYD_S8)
        p.__dict__.setdefault("_s8_direct", {})[obuf.buf] = (fscale, fwidth)
        wout = cout
        if tc_rows and cout < 16 <= fwidth and not dw:  # 16-byte output rows for the tcgen05 store path: zero output channels
            wout = 16
            qw = np.concatenate((qw, np.zeros((wout - cout, *qw.shape[1:]), np.int8)), 0)
            mult = np.concatenate((mult, np.zeros(wout - cout, np.float32)))
            bias = np.concatenate((bias, np.zeros(wout - cout, np.float32)))
        p.conv_s8(qsrc, obuf.sub(0, wout), qw, mult, bias, k, st, relu=relu, depthwise=dw, res=res, out_scale=fscale, out_round_bf16=True)
        return Slice(obuf.buf, 0, cout, oh, ow)
    return p.conv_s8(qsrc, dst, qw, mult, bias, k, st, relu=relu, depthwise=dw, res=res)


def emit_plain_conv(p: Plan, conv: nn.Conv2d, src: Slice, dst: Slice) -> Slice:
    """Final biased 1x1 convs of the heads (no BN, no activation)."""
    name = getattr(conv, "_uyd_name", "")
    _record_input(p, name, src)
    if _quantized(p, name):
        return emit_quant_conv(p, name, conv, None, src, dst, relu=False)
    w = conv.weight.detach().float().cpu().numpy()
    b = conv.bias.detach().float().cpu().numpy()
    return p.conv(src, dst, w, b, conv.kernel_size[0], conv.stride[0], relu=False)


class Bottleneck(nn.Module):
    def __init__(self, c1, c2, shortcut=True, g=1, k=(3, 3), e=0.5):
        super().__init__()
        c_ = int(c2 * e)
        self.cv1 = Conv(c1, c_, k[0], 1)
        self.cv2 = Conv(c_, c2, k[1], 1, g=g)
        self.add = shortcut and c1 == c2

    def emit(self, p, src, dst=None):
        t = self.cv1.emit(p, src, feeds=self.cv2.conv)   # t has one consumer: in the INT8 graph it is written as cv2's int8 input
        return self.cv2.emit(p, t, dst, res=src if self.add else None)


class C3k(nn.Module):
    """cv3(cat(m(cv1(x)), cv2(x))) -- the cat buffer is written in place by both branches."""

    def __init__(self, c1, c2, n=1, shortcut=True, g=1, e=0.5, k=3):
        super().__init__()
        c_ = int(c2 * e)
        self.c_ = c_
        self.cv1 = Conv(c1, c_, 1, 1)
        self.cv2 = Conv(c1, c_, 1, 1)
        self.cv3 = Conv(2 * c_, c2, 1)
        self.m = nn.Sequential(*(Bottleneck(c_, c_, shortcut, g, k=(k, k), e=1.0) for _ in range(n)))

    def emit(self, p, src, dst=None):
        fusable = (len(self.m) == 2 and all(b.add and b.cv1.k == 3 and b.cv2.k == 3 for b in self.m)
                   and self.cv3.c2 == src.c and 2 * self.c_ == src.c and os.environ.get("UYD_NO_C3K_FUSION", "0") != "1"
                   and getattr(p, "fusion", True) and not _quantized(p, getattr(self.cv1.conv, "_uyd_name", "")))
        if fusable:
            dst = dst or p.buffer(src.h, src.w, self.cv3.c2)
            if p.c3k_supported(src, dst) and p.shapes[src.buf][2] % 8 == 0 and p.shapes[dst.buf][2] % 8 == 0:
                folded = [fold_bn(m.conv, m.bn) for m in (self.cv1, self.cv2, self.m[0].cv1, self.m[0].cv2,
                                                          self.m[1].cv1, self.m[1].cv2, self.cv3)]
                return p.c3k(src, dst, [w for w, _ in folded], [b for _, b in folded])
        convs = (self.cv1, self.cv2, self.m[0].cv1, self.m[0].cv2, self.m[1].cv1, self.m[1].cv2, self.cv3) if len(self.m) == 2 else ()
        names = [getattr(m.conv, "_uyd_name", "") for m in convs]
        fusable_q = (len(convs) == 7 and all(b.add and b.cv1.k == 3 and b.cv2.k == 3 for b in self.m) and self.cv3.c2 == src.c
                     and 2 * self.c_ == src.c and getattr(p, "fusion", True) and os.environ.get("UYD_INT8_NO_C3K_FUSION", "0") != "1"
                     and all(_quantized(p, n) for n in names) and getattr(p, "conv_inputs", None) is None)
        if fusable_q:
            # INT8 graph: the whole block in one launch (uyd_plan_add_c3k_s8) -- the seven QuantConv2d with their input
            # quantisers inside the kernel, bit-identical to the quantize + conv_s8 ops emitted below
            dst = dst or p.buffer(src.h, src.w, self.cv3.c2)
            if p.c3k_supported(src, dst) and p.shapes[src.buf][2] % 8 == 0 and p.shapes[dst.buf][2] % 8 == 0:
                wq, mu, bi, sc = [], [], [], []
                for m, n in zip(convs, names):
                    ax, aw = p.quant.amax[n]
                    wq.append(Q.quantize_weights(m.conv.weight, aw))
                    mm, bb = Q.requant_params(ax, aw, m.bn, m.conv.bias)
                    mu.append(mm)
                    bi.append(bb)
                    sc.append(float(Q.scale_of(ax)))
                for m, n in zip(convs, names):
                    _record_input(p, n, src)
                return p.c3k_s8(src, dst, wq, mu, bi, sc)
        cat = p.buffer(src.h, src.w, 2 * self.c_)
        t = self.cv1.emit(p, src)
        for i, b in enumerate(self.m):
            t = b.emit(p, t, cat.sub(0, self.c_) if i == len(self.m) - 1 else None)
        self.cv2.emit(p, src, cat.sub(self.c_, self.c_))
        return self.cv3.emit(p, cat, dst)


class UpCat:
    """Upsample(x2, nearest) + Concat that is never materialised: ``low`` (half extent) is the tensor the graph
    upsamples, ``skip`` (full extent) the one it is concatenated with, in that channel order."""

    def __init__(self, low: Slice, skip: Slice):
        self.low, self.skip = low, skip
        self.h, self.w, self.c = skip.h, skip.w, low.c + skip.c


class StemOut:
    """Output of the fused stem when its only consumer is a C3k2 whose 1x1 cv1 joins the stem's launch
    (uyd_plan_add_stem2_pw): the 32-channel tensor is never written."""

    def __init__(self, h, w, c, folded):
        self.h, self.w, self.c, self.folded = h, w, c, folded


class C3k2(nn.Module):
    """C2f: cv1 -> chunk(2) -> n blocks chained on the last chunk -> cat -> cv2.  cv1 writes
    straight into the first 2c channels of the cat buffer; each block appends its c channels."""

    def __init__(self, c1, c2, n=1, c3k=False, e=0.5, g=1, shortcut=True):
        super().__init__()
        self.c = int(c2 * e)
        self.cv1 = Conv(c1, 2 * self.c, 1, 1)
        self.cv2 = Conv((2 + n) * self.c, c2, 1)
        self.m = nn.ModuleList(
            C3k(self.c, self.c, 2, shortcut, g) if c3k else Bottleneck(self.c, self.c, shortcut, g) for _ in range(n))

    def emit(self, p, src, dst=None, feeds=None):
        c, n = self.c, len(self.m)
        cat = p.buffer(src.h, src.w, (2 + n) * c)
        if isinstance(src, UpCat) and _quantized(p, getattr(self.cv1.conv, "_uyd_name", "")):
            # INT8 graph: the input quantiser is element-wise, so q(cat(up(a), b)) = cat(up(q(a)), q(b)), and the integer
            # sums split the same way: acc = up(W_a q(a)) + W_b q(b).  W_a q(a) is computed at HALF resolution into an fp32
            # buffer (exact: |sum| < 2^24) and added to the accumulator of the skip conv before its requant epilogue --
            # bit-identical to upsample -> concat -> quantize -> conv, without the upsampled tensor and its int8 copy.
            name = self.cv1.conv._uyd_name
            ax, aw = p.quant.amax[name]
            scale = float(Q.scale_of(ax))
            qw = Q.quantize_weights(self.cv1.conv.weight, aw)
            mult, bias = Q.requant_params(ax, aw, self.cv1.bn, self.cv1.conv.bias)
            ca, cb = src.low.c, src.skip.c
            pad32 = lambda n: (n + 31) // 32 * 32
            qa, qb = _s8_copy(p, src.low, scale, pad32(ca)), _s8_copy(p, src.skip, scale, pad32(cb))
            wpad = lambda w, n: np.concatenate((w, np.zeros((w.shape[0], n - w.shape[1], 1, 1), np.int8)), 1) if n != w.shape[1] else w
            part = p.buffer(src.low.h, src.low.w, 2 * c, UYD_F32)
            p.conv_s8(qa, part, wpad(qw[:, :ca], pad32(ca)), np.ones(2 * c, np.float32), np.zeros(2 * c, np.float32), 1, 1, relu=False)
            p.conv_s8(qb, cat.sub(0, 2 * c), wpad(qw[:, ca:], pad32(cb)), mult, bias, 1, 1, relu=True, pre=part)
        elif isinstance(src, UpCat):
            # cv1 is linear and 1x1, nearest upsampling commutes with it:
            #   cv1(cat(up(a), b)) = relu(up(W_a a) + W_b b + bias)
            # W_a a is computed at HALF resolution into an fp32 buffer and added inside cv1's epilogue, so
            # neither the upsampled tensor nor the concatenation is ever written (SURVEY.md a-5 / a-6).
            w, b = fold_bn(self.cv1.conv, self.cv1.bn)
            ca = src.low.c
            part = p.buffer(src.low.h, src.low.w, 2 * c, UYD_F32)
            p.conv(src.low, part, w[:, :ca], b * 0, 1, 1, relu=False)
            p.conv(src.skip, cat.sub(0, 2 * c), w[:, ca:], b, 1, 1, relu=True, pre=part)
        elif isinstance(src, StemOut):
            w, b = fold_bn(self.cv1.conv, self.cv1.bn)
            p.stem2(cat.sub(0, 2 * c), *src.folded, w, b)
        else:
            self.cv1.emit(p, src, cat.sub(0, 2 * c))
        for i, m in enumerate(self.m):
            m.emit(p, cat.sub((1 + i) * c, c), cat.sub((2 + i) * c, c))
        return self.cv2.emit(p, cat, dst, feeds=feeds)


class SPPF_DLA(nn.Module):
    """trainer.py:108-124 (incl. the (c1, 5) argument repair)."""

    def __init__(self, c1, c2, k=5):
        super().__init__()
        if c2 == k and c2 < 16:
            c2 = c1
        c_ = c1 // 2
        self.c_ = c_
        self.cv1 = Conv(c1, c_, 1, 1)
        self.cv2 = Conv(c_ * 4, c2, 1, 1)
        self.m = nn.MaxPool2d(kernel_size=k, stride=1, padding=k // 2)
        self.k = k

    def emit(self, p, src, dst=None):
        assert self.k == 5, "the pool cascade kernel is built for k = 5"
        cat = p.buffer(src.h, src.w, 4 * self.c_)
        self.cv1.emit(p, src, cat.sub(0, self.c_))
        p.sppf_pool(cat, self.c_)
        return self.cv2.emit(p, cat, dst)


class Concat(nn.Module):
    def __init__(self, dimension=1):
        super().__init__()
        self.d = dimension


class DFL(nn.Module):
    def __init__(self, c1=16):
        super().__init__()
        self.conv = nn.Conv2d(c1, 1, 1, bias=False).requires_grad_(False)
        self.conv.weight.data[:] = torch.arange(c1, dtype=torch.float).view(1, c1, 1, 1)
        self.c1 = c1


class Detect(nn.Module):
    """Attribute contract used by the reference (mine_data.py:110-161): nl, nc, reg_max, stride,
    cv2[i] (box branch), cv3[i] (cls branch), dfl."""

    def __init__(self, nc=80, ch=()):
        super().__init__()
        self.nc, self.nl, self.reg_max = nc, len(ch), 16
        self.no = nc + self.reg_max * 4
        self.stride = torch.zeros(self.nl)
        c2 = max(16, ch[0] // 4, self.reg_max * 4)
        c3 = max(ch[0], min(nc, 100))
        self.cv2 = nn.ModuleList(
            nn.Sequential(Conv(x, c2, 3), Conv(c2, c2, 3), nn.Conv2d(c2, 4 * self.reg_max, 1)) for x in ch)
        self.cv3 = nn.ModuleList(
            nn.Sequential(nn.Sequential(DWConv(x, x, 3), Conv(x, c3, 1)),
                          nn.Sequential(DWConv(c3, c3, 3), Conv(c3, c3, 1)),
                          nn.Conv2d(c3, nc, 1)) for x in ch)
        self.dfl = DFL(self.reg_max)

    def bias_init(self):
        for a, b, s in zip(self.cv2, self.cv3, self.stride):
            a[-1].bias.data[:] = 1.0
            b[-1].bias.data[: self.nc] = math.log(5 / self.nc / (640 / float(s)) ** 2)

    def emit(self, p, feats, fused: bool = False):
        """Box branch: Conv3x3 -> [Conv3x3 -> Conv2d 1x1 -> DFL] (one chained tcgen05 launch).
        Class branch: [DWConv3x3 -> Conv1x1] -> [DWConv3x3 -> Conv1x1 -> Conv2d 1x1 (-> sigmoid)].
        ``fused``: the chained kernels write the decoded prediction y directly and no raw head
        tensor exists; otherwise they write the raw logits into fp32 head buffers."""
        use_chain = (os.environ.get("UYD_NO_CHAIN", "0") != "1" and getattr(p, "fusion", True)
                     and not _quantized(p, getattr(self.cv2[0][0].conv, "_uyd_name", "")))
        a_total = sum(f.h * f.w for f in feats)
        heads, a_off = [], 0
        wb = lambda conv: (conv.weight.detach().float().cpu().numpy(), conv.bias.detach().float().cpu().numpy())
        for i, f in enumerate(feats):
            geo = dict(a_total=a_total, a_off=a_off, no=4 + self.nc, stride=float(self.stride[i]))
            head = None if fused else p.buffer(f.h, f.w, self.no, UYD_F32)
            # ---- box branch ----
            mid_conv, last = self.cv2[i][1], self.cv2[i][2]
            t = self.cv2[i][0].emit(p, f, feeds=mid_conv.conv)
            if (use_chain and mid_conv.k == 3 and mid_conv.s == 1 and mid_conv.g == 1 and 4 * self.reg_max == 64
                    and p.chain_supported(t, mid_conv.c2, 64) and p.shapes[t.buf][2] % 8 == 0):
                w1, b1 = fold_bn(mid_conv.conv, mid_conv.bn)
                w2, b2 = wb(last)
                p.chain(t, w1, b1, w2, b2, final=CHAIN_DFL if fused else CHAIN_STORE,
                        out=None if fused else head.sub(0, 4 * self.reg_max), y_ch0=0, **geo)
            elif fused:
                raise _NoFuse
            else:
                emit_plain_conv(p, last, mid_conv.emit(p, t, feeds=last, feeds_f32=True), head.sub(0, 4 * self.reg_max))
            # ---- class branch ----
            b0, b1_, last = self.cv3[i][0], self.cv3[i][1], self.cv3[i][2]
            mid = b0[1].c2
            dw_ok = lambda blk, c: blk[0].g == c and blk[0].k == 3 and blk[0].s == 1 and blk[1].k == 1
            if use_chain and dw_ok(b0, f.c) and p.chain_supported(f, f.c, mid) and mid % 16 == 0 and p.shapes[f.buf][2] % 8 == 0:
                w1, b1 = fold_bn(b0[0].conv, b0[0].bn)
                w2, b2 = fold_bn(b0[1].conv, b0[1].bn)
                z1 = p.chain(f, w1, b1, w2, b2, dw1=True, relu2=True, final=CHAIN_STORE, out=p.buffer(f.h, f.w, mid))
            else:
                z1 = b0[1].emit(p, b0[0].emit(p, f, feeds=b0[1].conv), feeds=b1_[0].conv)
            if use_chain and dw_ok(b1_, mid) and b1_[1].c2 == mid and p.chain_supported(z1, mid, mid) and self.nc <= 8:
                w1, b1 = fold_bn(b1_[0].conv, b1_[0].bn)
                w2, b2 = fold_bn(b1_[1].conv, b1_[1].bn)
                w3, b3 = wb(last)
                p.chain(z1, w1, b1, w2, b2, dw1=True, relu2=True, final=CHAIN_PW3, w3=w3, b3=b3,
                        out=None if fused else head.sub(4 * self.reg_max, self.nc), y_ch0=4, **geo)
            elif fused:
                raise _NoFuse
            else:
                emit_plain_conv(p, last, b1_[1].emit(p, b1_[0].emit(p, z1, feeds=b1_[1].conv), feeds=last, feeds_f32=True),
                                head.sub(4 * self.reg_max, self.nc))
            heads.append(head if head is not None else Slice(-1, 0, self.no, f.h, f.w))
            a_off += f.h * f.w
        return heads


def _class_ids(classes):
    """Ultralytics' ``classes`` (None, an int or an iterable of ints) as a tuple of ints, or None."""
    if classes is None:
        return None
    return tuple(operator.index(c) for c in ([classes] if isinstance(classes, int) else classes))


def _nms_options(classes, multi_label: bool):
    """``uyd_nms_options`` for Ultralytics' ``classes`` / ``multi_label``, or None at their defaults (plain ``uyd_nms``).
    ``[]`` keeps nothing; ids outside [0, nc) match nothing."""
    if classes is None and not multi_label:
        return None
    opt = _lib.NmsOptions(multi_label=1 if multi_label else 0)
    if classes is not None:
        # every id outside [0, 256] matches nothing: clamping keeps that and fits a C int
        ids = [min(max(c, -1), 1 << 30) for c in _class_ids(classes)]
        opt.num_filter_classes = len(ids)
        opt.filter_classes = (C.c_int * max(1, len(ids)))(*ids)   # the struct keeps the array alive
    return opt


def _literal(a):
    if isinstance(a, str):
        try:
            return ast.literal_eval(a)
        except (ValueError, SyntaxError):
            return a
    return a


def parse_model(d: dict, ch: int = 3):
    """YAML -> holder modules (parse_model semantics restated in SURVEY.md appendix A.1,
    with the scale/scales defaults injected by trainer.py:85-94)."""
    nc = d["nc"]
    scale = d.get("scale", "m")
    depth, width, max_ch = d.get("scales", {scale: [1.0, 1.0, 1024]})[scale]
    chs, layers, save = [ch], [], []
    for i, (f, n, m, args) in enumerate(d["backbone"] + d["head"]):
        args = [nc if a == "nc" else _literal(a) for a in args]
        n = max(round(n * depth), 1) if n > 1 else n
        if m in ("Conv", "C3k2"):
            c1, c2 = chs[f], args[0]
            if c2 != nc:
                c2 = _make_divisible(min(c2, max_ch) * width, 8)
            args = [c1, c2, *args[1:]]
            if m == "C3k2":
                args.insert(2, n)
                if scale in "mlx":
                    args[3] = True
            mod = Conv(*args) if m == "Conv" else C3k2(*args)
        elif m == "SPPF_DLA":
            c2 = chs[f]
            mod = SPPF_DLA(*args)
        elif m == "nn.Upsample":
            c2 = chs[f]
            mod = nn.Upsample(*args)
            if not (mod.scale_factor == 2 and mod.mode == "nearest"):
                raise NotImplementedError("only nearest x2 upsampling is on the hot path")
        elif m == "Concat":
            c2 = sum(chs[x] for x in f)
            mod = Concat(*args)
        elif m == "Detect":
            c2 = None
            mod = Detect(args[0], [chs[x] for x in f])
        else:
            raise NotImplementedError(f"module {m} is not part of the UNINA-YOLO-DLA graph")
        mod.i, mod.f, mod.c_out = i, f, c2
        save.extend(x % i for x in ([f] if isinstance(f, int) else f) if x != -1)
        layers.append(mod)
        if i == 0:
            chs = []
        chs.append(c2)
    return nn.Sequential(*layers), sorted(save)


class UninaYoloB200(nn.Module):
    def __init__(self, cfg=DEFAULT_YAML, ch: int = 3, nc: int | None = None, verbose: bool = False):
        super().__init__()
        self.yaml = dict(cfg) if isinstance(cfg, dict) else yaml.safe_load(Path(cfg).read_text())
        if nc is not None:
            self.yaml["nc"] = nc
        self.model, self.save = parse_model(self.yaml, ch)
        self.nc = self.yaml["nc"]
        self.names = {i: str(i) for i in range(self.nc)}
        det = self.model[-1]
        # strides of the detect inputs: product of the conv strides on the path (dry-run result)
        det.stride = torch.tensor([float(s) for s in self._level_strides()])
        self.stride = det.stride
        det.bias_init()
        for name, mod in self.named_modules():
            if isinstance(mod, nn.Conv2d):
                mod._uyd_name = name            # the key of the pytorch-quantization ``_amax`` buffers
        self._plans = {}
        self._nms_ws = {}
        self._graphs = {}
        self.quant = None                       # quant.QuantSpec when the INT8 path is active
        self.eval()

    @classmethod
    def from_yaml(cls, path=DEFAULT_YAML, nc: int | None = None) -> "UninaYoloB200":
        return cls(path, nc=nc)

    # ---- graph bookkeeping -------------------------------------------------------------
    def _level_strides(self):
        st = []
        for m in self.model:
            fi = m.f if isinstance(m.f, int) else m.f[0]
            s_in = 1 if (m.i == 0) else st[fi if fi != -1 else m.i - 1]
            if isinstance(m, Conv):
                st.append(s_in * m.s)
            elif isinstance(m, nn.Upsample):
                st.append(s_in // 2)
            elif isinstance(m, Detect):
                st.append(0)
                return [st[j] for j in m.f]
            else:
                st.append(s_in)
        raise ValueError("graph has no Detect layer")

    def num_anchors(self, H: int, W: int) -> int:
        return sum((H // int(s)) * (W // int(s)) for s in self.stride.tolist())

    def refresh(self) -> None:
        """Drop compiled plans (call after mutating parameters in place)."""
        self._graphs.clear()
        self._plans.clear()

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """Accepts the reference schema (925 entries) plus, for QAT checkpoints, the pytorch-quantization
        ``<conv>._input_quantizer._amax`` / ``<conv>._weight_quantizer._amax`` buffers, which switch the
        INT8 path on (qat.py:109-124)."""
        plain, amax = Q.split_state_dict(state_dict)
        out = super().load_state_dict(plain, strict=strict, assign=assign)
        if amax:
            self.set_quantization(amax)
        self.refresh()
        return out

    def set_quantization(self, amax: dict | None, float_layers=(0, 1, 2)) -> "UninaYoloB200":
        """Switches the INT8 path on (``amax``: conv module name -> (input amax, weight amax)) or off (None).
        Convs of ``model.{i}`` for i in ``float_layers`` stay bf16 (the reference's precision carve-out,
        qat.py:700-753); convs without an entry stay bf16 too."""
        self.quant = Q.QuantSpec(dict(amax), tuple(float_layers)) if amax else None
        self.refresh()
        return self

    def quant_state_dict(self) -> dict:
        """The ``_amax`` buffers of the active quantisation in pytorch-quantization's naming."""
        return Q.amax_state_dict(self.quant)

    def _apply(self, fn, recurse=True):
        self._graphs.clear()
        self._plans.clear()
        return super()._apply(fn, recurse)

    # ---- plan construction -------------------------------------------------------------
    def _build_plan(self, device: int, max_batch: int, H: int, W: int, fused: bool = False, fusion: bool = True,
                    record_inputs: bool = False) -> Plan:
        """``fusion=False`` emits one op per conv (calibration needs every conv input in HBM);
        ``record_inputs`` keeps the input slice of every conv in ``plan.conv_inputs``."""
        p = Plan(device, max_batch)
        p.in_hw = (H, W)
        p.fused = fused
        p.fusion = fusion
        p.quant = self.quant
        if record_inputs:
            p.conv_inputs = {}
        layers = list(self.model)
        # pass 1: extents of every layer output
        shape = []
        for m in layers:
            src = None if m.i == 0 else (m.f if isinstance(m.f, int) else m.f[0])
            ih, iw = (H, W) if m.i == 0 else shape[src if src != -1 else m.i - 1][1:]
            if isinstance(m, Conv):
                shape.append((m.c2, ih // m.s, iw // m.s))
            elif isinstance(m, nn.Upsample):
                shape.append((m.c_out, ih * 2, iw * 2))
            elif isinstance(m, Detect):
                shape.append(None)
            else:
                shape.append((m.c_out, ih, iw))
        # pass 2a: Upsample -> Concat([-1, j]) -> C3k2 with no other consumer: folded into the C3k2's first conv
        folded = {}   # concat layer index -> (upsample layer index, skip layer index)
        if fusion and os.environ.get("UYD_NO_UPSAMPLE_FOLD", "0") != "1":
            for u, c, k in zip(layers, layers[1:], layers[2:]):
                if (isinstance(u, nn.Upsample) and isinstance(c, Concat) and isinstance(k, C3k2) and isinstance(c.f, list)
                        and len(c.f) == 2 and c.f[0] == -1 and c.f[1] != -1 and k.f == -1 and u.i not in self.save
                        and c.i not in self.save and (2 * k.c) % 16 == 0 and shape[u.i][0] % 16 == 0
                        and shape[c.f[1] % c.i][0] % 16 == 0
                        and (not _quantized(p, getattr(k.cv1.conv, "_uyd_name", "")) or os.environ.get("UYD_INT8_NO_UPFOLD", "0") != "1")):
                    folded[c.i] = (u.i, c.f[1] % c.i)
        # pass 2: every tensor consumed by a Concat lives inside that Concat's buffer
        home = {}
        for m in layers:
            if isinstance(m, Concat) and m.i not in folded:
                c, h, w = shape[m.i]
                cat = p.buffer(h, w, c)
                home[m.i] = cat
                off = 0
                for j in m.f:
                    j = m.i - 1 if j == -1 else j
                    assert j not in home, "a tensor feeding two Concat layers would need a copy"
                    home[j] = cat.sub(off, shape[j][0])
                    off += shape[j][0]
        # pass 3: emit
        outs = []
        l0, l1 = layers[0], layers[1]
        stem2 = (os.environ.get("UYD_NO_STEM_FUSION", "0") != "1" and fusion and not _quantized(p, "model.1.conv") and isinstance(l0, Conv) and isinstance(l1, Conv)
                 and (l0.c1, l0.c2, l0.k, l0.s, l0.g) == (3, 16, 3, 2, 1) and (l1.c1, l1.c2, l1.k, l1.s, l1.g) == (16, 32, 3, 2, 1)
                 and l1.f == -1 and 0 not in self.save and 0 not in home and H % 4 == 0 and W % 4 == 0)
        l2 = layers[2] if len(layers) > 2 else None
        # model.1 feeds only model.2 (a C3k2 with a 32 -> 16 cv1): that 1x1 joins the stem's launch
        stem_pw = (stem2 and os.environ.get("UYD_NO_STEM_PW", "0") != "1" and isinstance(l2, C3k2) and l2.f == -1 and l2.c == 8
                   and 1 not in self.save and 1 not in home and getattr(p, "conv_inputs", None) is None
                   and not _quantized(p, getattr(l2.cv1.conv, "_uyd_name", "")))
        for m in layers:
            def src_of(j):
                return outs[m.i - 1] if j == -1 else outs[j]
            dst = home.get(m.i)
            if stem2 and m.i == 0:
                outs.append(None)      # lives only in shared memory of the fused stem kernel
            elif stem_pw and m.i == 1:
                outs.append(StemOut(H // 4, W // 4, l1.c2, fold_bn(l0.conv, l0.bn) + fold_bn(l1.conv, l1.bn)))
            elif stem2 and m.i == 1:
                dst = dst or p.buffer(H // 4, W // 4, l1.c2)
                if p.shapes[dst.buf][2] % 8 or dst.coff % 8:
                    raise ValueError("fused stem needs a 16-byte aligned output slice")
                (w0, b0), (w1, b1) = fold_bn(l0.conv, l0.bn), fold_bn(l1.conv, l1.bn)
                outs.append(p.stem2(dst, w0, b0, w1, b1))
            elif m.i == 0:
                assert isinstance(m, Conv), "the first layer must be a Conv reading the frame"
                outs.append(m.emit(p, NETWORK_INPUT, dst))
            elif isinstance(m, (Conv, C3k2, SPPF_DLA)):
                # INT8 graph: a layer whose output is read by the next layer only (not saved for a Concat / Detect) writes it
                # directly as the int8 input of that layer's first conv -- no bf16 tensor, no quantize launch
                feeds = None
                nxt = layers[m.i + 1] if m.i + 1 < len(layers) else None
                if (self.quant is not None and fusion and not record_inputs and dst is None and m.i not in self.save
                        and isinstance(m, (Conv, C3k2)) and isinstance(nxt, (Conv, C3k2, SPPF_DLA)) and nxt.f == -1
                        and os.environ.get("UYD_INT8_NO_LAYER_FEEDS", "0") != "1"):
                    first = nxt.conv if isinstance(nxt, Conv) else nxt.cv1.conv
                    last = m.conv if isinstance(m, Conv) else m.cv2.conv
                    if _quantized(p, getattr(first, "_uyd_name", "")) and _quantized(p, getattr(last, "_uyd_name", "")):
                        feeds = first
                outs.append(m.emit(p, src_of(m.f), dst, feeds=feeds) if feeds is not None else m.emit(p, src_of(m.f), dst))
            elif isinstance(m, nn.Upsample):
                s = src_of(m.f)
                if any(u == m.i for u, _ in folded.values()):
                    outs.append(s)      # stays at half resolution: its consumer is a folded Concat
                    continue
                dst = dst or p.buffer(s.h * 2, s.w * 2, s.c)
                outs.append(p.upsample2x(s, dst))
            elif isinstance(m, Concat):
                if m.i in folded:
                    u, j = folded[m.i]
                    outs.append(UpCat(outs[u], outs[j]))
                    continue
                outs.append(home[m.i])
            elif isinstance(m, Detect):
                feats = [src_of(j) for j in m.f]
                heads = m.emit(p, feats, fused)
                if fused:
                    p.heads = heads  # extents only: the decoded output is written by the head kernels
                else:
                    p.set_heads(heads, [int(s) for s in m.stride.tolist()], m.reg_max, m.nc)
                    dfl_name = getattr(m.dfl.conv, "_uyd_name", "")
                    _record_input(p, dfl_name, Slice(-2, 0, m.reg_max, 0, 0))
                    if _quantized(p, dfl_name):
                        check(_lib.lib().uyd_plan_set_dfl_quant(p.handle, float(self.quant.amax[dfl_name][0])), "uyd_plan_set_dfl_quant")
                outs.append(None)
        hidden = set(folded) | {u for u, _ in folded.values()}   # layers whose output tensor is never written
        p.layer_outputs = [None if (i in hidden or not isinstance(o, Slice)) else o for i, o in enumerate(outs)]
        return p.finalize()

    def plan_for(self, x: torch.Tensor, fused: bool = False) -> Plan:
        """The compiled plan for frames shaped like ``x``.  ``fused``: the variant whose head kernels
        write the decoded prediction directly (no raw head tensors); falls back to the raw-head
        variant when the graph / shape does not allow it."""
        B, _, H, W = x.shape
        dev = x.device.index if x.device.index is not None else torch.cuda.current_device()
        key = (dev, H, W, bool(fused))
        p = self._plans.get(key)
        if p is None or p.max_batch < B:
            if H % 32 or W % 32:
                raise ValueError("frame height/width must be multiples of 32")
            if fused:
                try:
                    p = self._build_plan(dev, B, H, W, True)
                except _NoFuse:
                    p = self.plan_for(x, False)
            else:
                p = self._build_plan(dev, B, H, W, False)
            self._plans[key] = p
        return p

    def _decoded_into(self, x: torch.Tensor, y: torch.Tensor) -> Plan:
        """x -> y[B,4+nc,A] through the fused plan (C calls only: usable under graph capture)."""
        p = self.plan_for(x, fused=os.environ.get("UYD_NO_FUSED_DECODE", "0") != "1")
        if p.fused:
            p.run(x, y)
        else:
            p.run(x)
            p.decode(y, x.shape[0])
        return p

    # ---- execution ---------------------------------------------------------------------
    def _prep(self, x: torch.Tensor) -> torch.Tensor:
        if self.training:
            raise RuntimeError("UninaYoloB200 implements the inference path only: call .eval()")
        if not torch.cuda.is_available():
            raise _lib.UydError("no CUDA device: the B200 path has no CPU fallback")
        if not x.is_cuda:
            x = x.to(next(self.parameters()).device if next(self.parameters()).is_cuda else "cuda", non_blocking=True)
        # uint8 frames go to the GPU as they are: the stem conv divides by 255 on load
        return x.contiguous() if x.dtype == torch.uint8 else x.float().contiguous()

    @torch.no_grad()
    def init_synthetic(self, seed: int = 0, cls_bias: float = -1.1, gain: float = 1.0) -> "UninaYoloB200":
        """Seeded, data-free initialisation for parity runs and benchmarks: normal conv weights
        with variance gain/fan_in and non-trivial BN statistics, so BN folding is exercised and
        every layer output still depends on the frame (torch's default init decays ~10x per
        stage and makes every score equal to the head bias, SURVEY.md header fact 3).
        gain = 1 (LeCun) gives a contractive, well-conditioned network: 2^-9 bf16 rounding noise
        is not amplified with depth.  gain = 2 (He) amplifies it ~4x, and BN statistics
        calibrated on random data make the net chaotic (>50 % deviation even in fp16) --
        DESIGN.md "Numerics" has the measurements."""
        from .synth import synthetic_init_

        synthetic_init_(self, seed, gain)
        det = self.model[-1]
        for box, cls in zip(det.cv2, det.cv3):
            box[-1].bias.fill_(1.0)
            cls[-1].bias.fill_(cls_bias)
        self.refresh()
        return self

    @torch.no_grad()
    def calibrate_cls_bias(self, x: torch.Tensor, per_image: int, conf: float = 0.25) -> float:
        """Shifts the class-branch biases so that about ``per_image`` anchors per frame clear
        ``conf`` on the frames ``x`` (synthetic-weight benchmarks need a realistic NMS load).
        Runs the CUDA forward once; returns the applied shift."""
        _, xs = self.forward(x)
        det = self.model[-1]
        best = torch.cat([t[:, 4 * det.reg_max:].amax(1).flatten(1) for t in xs], 1)  # [B, A] logits
        k = max(1, min(best.shape[1] - 1, per_image))
        kth = best.topk(k, dim=1).values[:, -1].mean().item()
        shift = math.log(conf / (1 - conf)) - kth
        for cls in det.cv3:
            cls[-1].bias.add_(shift)
        self.refresh()
        return shift

    @torch.no_grad()
    def calibrate_int8(self, frames: torch.Tensor, float_layers=(0, 1, 2), enable: bool = True, method: str = "max",
                       batch_size: int = 8, percentile: float = 99.99) -> dict:
        """Static INT8 scales from a calibration set (the reference's calibration pass, qat.py:129-220, never
        materialises them).  ``frames`` [N,3,H,W] is walked in chunks of ``batch_size`` through the bf16 forward.
          method "max"                     : amax = max |x| (one GPU reduction per conv input, uyd_plan_slice_absmax)
          method "histogram" / "entropy"   : the reference's default (qat.py:91-126, 676-697): |x| histogram with 2048
                                             bins per conv input on the GPU (uyd_plan_slice_histogram), KL-divergence
                                             threshold search on the host (quant.amax_entropy)
          method "percentile" / "mse"      : the other two amax rules of the same calibrator
        Weights use the same method on the host.  Returns ``{conv name: (amax_in, amax_w)}`` and, with ``enable``,
        switches the INT8 path on."""
        rule = Q.calibration_rule(method)
        saved, self.quant = self.quant, None
        try:
            x_all = self._prep(frames)
            _, _, H, W = x_all.shape
            B = min(batch_size, x_all.shape[0])
            dev = x_all.device.index if x_all.device.index is not None else torch.cuda.current_device()
            p = self._build_plan(dev, B, H, W, fused=False, fusion=False, record_inputs=True)
            names = [n for n, s in p.conv_inputs.items() if s.buf >= 0]
            det = self.model[-1]
            dfl_name = getattr(det.dfl.conv, "_uyd_name", "")
            dfl_cal, dfl_max = (Q.HistogramCalibrator() if rule != "max" else None), 0.0

            def dfl_batch(x, nb):
                nonlocal dfl_max
                if dfl_name in p.conv_inputs:  # input of the DFL projection: the softmax probabilities of the box logits
                    for lvl, hd in enumerate(p.heads):
                        t = torch.empty(nb, hd.c, hd.h, hd.w, dtype=torch.float32, device=x.device)
                        p.export_head(lvl, t, nb)
                        pr = t[:, :4 * det.reg_max].reshape(nb, 4, det.reg_max, -1).softmax(2)
                        dfl_max = max(dfl_max, float(pr.max()))
                        if dfl_cal is not None:
                            dfl_cal.collect_host(pr.cpu().numpy())

            a_in = Q.collect_input_amax(p, x_all, B, names, rule, percentile, per_batch=dfl_batch)
            convs = {n: m for n, m in self.named_modules() if isinstance(m, nn.Conv2d)}
            amax = {n: (max(a, 1e-6), Q.weight_amax(convs[n].weight, rule, percentile)) for n, a in zip(names, a_in)}
            if dfl_name in p.conv_inputs:
                amax[dfl_name] = (dfl_max if rule == "max" else dfl_cal.compute_amax(rule, percentile), float(det.reg_max - 1))
        finally:
            self.quant = saved
        if enable:
            self.set_quantization(amax, float_layers)
        return amax

    @torch.no_grad()
    def forward(self, x: torch.Tensor, raw_heads: bool = True):
        """Eval forward of DetectionModel: ``(y[B,4+nc,A], [x_l[B,no,H_l,W_l]])``."""
        x = self._prep(x)
        B = x.shape[0]
        A = self.num_anchors(x.shape[2], x.shape[3])
        y = torch.empty(B, 4 + self.nc, A, dtype=torch.float32, device=x.device)
        if not raw_heads:
            self._decoded_into(x, y)
            return y
        p = self.plan_for(x)
        p.run(x)
        p.decode(y, B)
        xs = []
        for lvl, h in enumerate(p.heads):
            t = torch.empty(B, h.c, h.h, h.w, dtype=torch.float32, device=x.device)
            p.export_head(lvl, t, B)
            xs.append(t)
        return y, xs

    @torch.no_grad()
    def forward_camera(self, frames: torch.Tensor, size=None, norm=None, uv: torch.Tensor | None = None,
                       letterbox: bool = False) -> torch.Tensor:
        """Camera bytes straight into the stem (SURVEY 8f-1; replaces preprocess_bgra_resize / preprocess_nv12 +
        the CHW fp32 tensor, perception_node.cpp:604-612): ``frames`` uint8 device ``[B,H,W,4]`` packed BGRA, resampled
        bilinearly to ``size=(H',W')`` when given, or -- with ``uv`` ``[B,H/2,W]`` -- the Y planes ``[B,H,W]`` of NV12
        frames.  ``norm``: ``_lib.NormParams`` (default: plain x / 255, what the YAML model is fed).
        ``letterbox``: BGRA frames of any extent are letterboxed as the Ultralytics predictor does (aspect-kept
        cv2 INTER_LINEAR resize, grey 114 around it) into ``size``, by default ``preprocess.letterbox_shape(H, W)``
        (1280 x 720 -> 384 x 640).  Returns the decoded prediction ``y[B,4+nc,A]`` in model-input pixels."""
        import types

        if self.training:
            raise RuntimeError("UninaYoloB200 implements the inference path only: call .eval()")
        assert frames.is_cuda and frames.dtype == torch.uint8 and frames.stride(-1) == 1
        nv12 = uv is not None
        if nv12 and letterbox:
            raise ValueError("letterbox reads packed BGRA frames; NV12 frames are not letterboxed")
        B, H, W = frames.shape[:3]
        oh, ow = (H, W) if nv12 else P.camera_extent(H, W, size, letterbox)
        p = self.plan_for(types.SimpleNamespace(shape=(B, 3, oh, ow), device=frames.device),
                          fused=os.environ.get("UYD_NO_FUSED_DECODE", "0") != "1")
        f = _lib.CameraFrames()
        f.format = _lib.CAM_NV12 if nv12 else (_lib.CAM_BGRA_LETTERBOX if letterbox else _lib.CAM_BGRA)
        f.width, f.height = W, H
        f.pitch = frames.stride(1)
        f.frame_stride = frames.stride(0)
        f.data = frames.data_ptr()
        if nv12:
            assert uv.is_cuda and uv.dtype == torch.uint8 and uv.stride(-1) == 1 and uv.shape[0] == B
            f.uv, f.uv_pitch, f.uv_frame_stride = uv.data_ptr(), uv.stride(1), uv.stride(0)
        f.norm = norm if norm is not None else _lib.NormParams(0.0, 0.0, 0.0, 1.0, 1.0, 1.0)
        y = torch.empty(B, 4 + self.nc, self.num_anchors(oh, ow), dtype=torch.float32, device=frames.device)
        if p.fused:
            p.run_camera(f, B, y)
        else:
            p.run_camera(f, B)
            p.decode(y, B)
        return y

    @torch.no_grad()
    def predict_camera(self, frames: torch.Tensor, size=None, norm=None, uv=None, conf: float = 0.25, iou: float = 0.7,
                       max_det: int = 300, max_nms: int = 30000, letterbox: bool = False, *, classes=None,
                       agnostic: bool = False, multi_label: bool = False):
        """``forward_camera`` + NMS: (det[B,max_det,6], count[B]) on the device.  With ``letterbox`` the rows are in
        frame pixels (``scale_boxes`` + ``clip_boxes`` of the Ultralytics predictor, one launch).  ``classes``,
        ``agnostic``, ``multi_label``: as in ``nms``."""
        det, cnt = self.nms(self.forward_camera(frames, size, norm, uv, letterbox), conf, iou, max_det, max_nms,
                            classes=classes, agnostic=agnostic, multi_label=multi_label)
        if letterbox:
            H, W = frames.shape[1:3]
            P.letterbox_boxes(det, cnt, H, W, *P.camera_extent(H, W, size, True))
        return det, cnt

    def _nms_workspace(self, dev: int, B: int, A: int, device) -> torch.Tensor:
        need = int(_lib.lib().uyd_nms_workspace_bytes(B, A))
        ws = self._nms_ws.get(dev)
        if ws is None or ws.numel() < need:
            ws = torch.empty(need, dtype=torch.uint8, device=device)
            self._nms_ws[dev] = ws
        return ws

    def _nms_into(self, y, det, idx, cnt, ws, conf, iou, max_det, max_nms, max_wh, opt=None) -> None:
        """C call only (no allocation): safe inside CUDA-graph capture.  ``opt``: ``_nms_options`` (None: uyd_nms)."""
        B, no, A = y.shape
        dev = y.device.index if y.device.index is not None else torch.cuda.current_device()
        if opt is not None:
            check(_lib.lib().uyd_nms_ex(_lib.context(dev), C.c_void_p(y.data_ptr()), B, no - 4, A, conf, iou, max_nms, max_det,
                                        max_wh, C.byref(opt), C.c_void_p(det.data_ptr()),
                                        C.c_void_p(idx.data_ptr()) if idx is not None else None, C.c_void_p(cnt.data_ptr()),
                                        C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "uyd_nms_ex")
            return
        check(_lib.lib().uyd_nms(_lib.context(dev), C.c_void_p(y.data_ptr()), B, no - 4, A, conf, iou, max_nms, max_det,
                                 max_wh, C.c_void_p(ws.data_ptr()), ws.numel(), C.c_void_p(det.data_ptr()),
                                 C.c_void_p(idx.data_ptr()) if idx is not None else None, C.c_void_p(cnt.data_ptr()),
                                 C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "uyd_nms")

    @torch.no_grad()
    def nms(self, y: torch.Tensor, conf: float = 0.25, iou: float = 0.7, max_det: int = 300, max_nms: int = 30000,
            max_wh: float = 7680.0, return_index: bool = False, *, classes=None, agnostic: bool = False,
            multi_label: bool = False):
        """Ultralytics ``non_max_suppression`` on ``y[B,4+nc,A]`` -> (det[B,max_det,6], count[B]).
        ``classes``: keep only these class ids (an int or a list; ``[]`` keeps nothing), filtered before the
        ``max_nms`` truncation and the NMS.  ``agnostic``: NMS across classes (``max_wh`` 0).  ``multi_label``: every
        (anchor, class) pair with a score above ``conf`` is a candidate (what ``model.val`` runs), not only the best
        class of each anchor; ``return_index`` then gives the anchor of each row."""
        assert y.is_cuda and y.dtype == torch.float32 and y.is_contiguous()
        B, no, A = y.shape
        dev = y.device.index if y.device.index is not None else torch.cuda.current_device()
        ws = self._nms_workspace(dev, B, A, y.device)
        # uyd_nms defines every output element (zeros / -1 past the count): no fill launches
        det = torch.empty(B, max_det, 6, dtype=torch.float32, device=y.device)
        idx = torch.empty((B, max_det), dtype=torch.int32, device=y.device) if return_index else None
        cnt = torch.empty(B, dtype=torch.int32, device=y.device)
        self._nms_into(y, det, idx, cnt, ws, conf, iou, max_det, max_nms, 0.0 if agnostic else max_wh,
                       _nms_options(classes, multi_label))
        return (det, cnt, idx) if return_index else (det, cnt)

    # batches up to this size replay a captured CUDA graph (the ~70 launches of a step are
    # launch-latency-bound below it); larger batches are launched directly.
    GRAPH_MAX_BATCH = 8

    def _graph_for(self, x: torch.Tensor, conf, iou, max_det, max_nms, classes=None, agnostic=False, multi_label=False):
        B, _, H, W = x.shape
        dev = x.device.index if x.device.index is not None else torch.cuda.current_device()
        key = (dev, B, H, W, x.dtype, float(conf), float(iou), int(max_det), int(max_nms), _class_ids(classes), bool(agnostic), bool(multi_label))
        g = self._graphs.get(key)
        if g is not None:
            return g
        A = self.num_anchors(H, W)
        xs = torch.empty_like(x)
        y = torch.empty(B, 4 + self.nc, A, dtype=torch.float32, device=x.device)
        det = torch.zeros(B, max_det, 6, dtype=torch.float32, device=x.device)
        cnt = torch.zeros(B, dtype=torch.int32, device=x.device)
        ws = torch.empty(int(_lib.lib().uyd_nms_workspace_bytes(B, A)), dtype=torch.uint8, device=x.device)
        opt = _nms_options(classes, multi_label)   # read at launch: the captured kernel holds the class mask by value

        def body():
            det.zero_()
            self._decoded_into(xs, y)
            self._nms_into(y, det, None, cnt, ws, conf, iou, max_det, max_nms, 0.0 if agnostic else 7680.0, opt)

        xs.copy_(x)
        side = torch.cuda.Stream(device=x.device)
        side.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(side):  # warm-up outside capture: one-time kernel attribute calls happen here
            body()
        torch.cuda.current_stream(x.device).wait_stream(side)
        torch.cuda.synchronize(x.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body()
        g = (graph, xs, det, cnt, (self.plan_for(xs, True), y, ws))  # the graph writes y / ws on every replay: keep them alive
        self._graphs[key] = g
        return g

    @torch.no_grad()
    def predict_batched(self, x: torch.Tensor, conf: float = 0.25, iou: float = 0.7, max_det: int = 300,
                        max_nms: int = 30000, graph: bool | None = None, *, classes=None, agnostic: bool = False,
                        multi_label: bool = False):
        """Forward + decode + NMS, everything left on the device: (det[B,max_det,6], count[B]).
        ``graph`` (default: batch <= GRAPH_MAX_BATCH) replays the whole step as one CUDA graph.  ``classes``,
        ``agnostic``, ``multi_label``: as in ``nms``; ``model.val``'s NMS is ``conf=0.001, iou=0.7, multi_label=True``."""
        x = self._prep(x)
        if graph is None:
            graph = x.shape[0] <= self.GRAPH_MAX_BATCH and os.environ.get("UYD_NO_GRAPH", "0") != "1"
        if graph:
            with torch.cuda.device(x.device):   # capture and replay on the frames' device, whatever the caller's current one is
                g, xs, det, cnt, _ = self._graph_for(x, conf, iou, max_det, max_nms, classes, agnostic, multi_label)
                xs.copy_(x)
                g.replay()
                return det.clone(), cnt.clone()
        y = self.forward(x, raw_heads=False)
        return self.nms(y, conf, iou, max_det, max_nms, classes=classes, agnostic=agnostic, multi_label=multi_label)

    @torch.no_grad()
    def predict(self, x: torch.Tensor, conf: float = 0.25, iou: float = 0.7, max_det: int = 300, max_nms: int = 30000, *,
                classes=None, agnostic: bool = False, multi_label: bool = False):
        """Per-image ``[N_i, 6]`` tensors ``(x1,y1,x2,y2,conf,cls)`` like ``result.boxes.data``; ``classes`` and
        ``agnostic`` are ``YOLO.predict``'s ``classes=`` / ``agnostic_nms=`` (see ``nms``)."""
        det, cnt = self.predict_batched(x, conf, iou, max_det, max_nms, classes=classes, agnostic=agnostic,
                                        multi_label=multi_label)
        counts = cnt.tolist()
        return [det[b, :n] for b, n in enumerate(counts)]

    @torch.no_grad()
    def predict_stream(self, batches, conf: float = 0.25, iou: float = 0.7, max_det: int = 300, max_nms: int = 30000,
                       to_host: bool = True, camera: str | None = None, size=None, norm=None, letterbox: bool = False, *,
                       classes=None, agnostic: bool = False, multi_label: bool = False):
        """Generator form of ``predict`` (the reference consumes ``YOLO.predict(..., stream=True)``,
        train.py:396-423): ``batches`` yields host frame batches ``[B,3,H,W]`` (uint8 or float, ideally
        pinned).  Batch i+1 is copied host->device on a copy stream while batch i computes, so a
        steady-state step costs max(copy, compute) instead of their sum.  Yields, in order,
        ``(det[B,max_det,6], count[B])`` -- pinned host tensors (``to_host``) or device tensors;
        either stays valid while the generator is advanced twice more (the pinned result buffers rotate
        through a ring of four, separate from the two input staging slots).
        NMS (and the result copy) of step i run on a second stream: the per-image NMS kernel occupies one SM per frame, so
        at batch 64 it leaves 84 of the 148 SMs idle -- the next step's forward fills them.  Batches that are already
        device tensors are used in place (no staging copy).
        ``camera``: the batches are camera frames read by the stem itself (``forward_camera``): ``"nv12"`` = uint8
        ``[B, 3H/2, W]`` (the Y rows followed by the interleaved UV rows: 1.5 bytes per pixel over PCIe instead of 3),
        ``"bgra"`` = uint8 ``[B, H, W, 4]`` (resampled to ``size`` when given); ``norm`` as in ``forward_camera``.
        ``letterbox`` (``camera="bgra"`` only): the frames are letterboxed as in ``forward_camera`` and the rows come
        back in frame pixels.  ``classes``, ``agnostic``, ``multi_label``: as in ``nms``."""
        if camera not in (None, "nv12", "bgra"):
            raise ValueError("camera must be None, 'nv12' or 'bgra'")
        if letterbox and camera != "bgra":
            raise ValueError("letterbox needs camera='bgra'")
        if not torch.cuda.is_available():
            raise _lib.UydError("no CUDA device: the B200 path has no CPU fallback")
        prm = next(self.parameters())
        device = prm.device if prm.is_cuda else torch.device("cuda", torch.cuda.current_device())
        it = iter(batches)
        try:
            first = next(it)
        except StopIteration:
            return
        Bmax = first.shape[0]
        main_s = torch.cuda.current_stream(device)
        # staging slots, pinned result buffers, copy stream and events are allocated once per
        # (frame shape, dtype, max_det) and reused by later calls: cudaHostAlloc alone costs milliseconds
        skey = (device, tuple(first.shape), first.dtype, max_det, to_host, camera)
        state = self.__dict__.setdefault("_stream_state", {}).get(skey)
        if state is None:

            class Slot:
                pass

            slots = []
            for _ in range(2):
                s = Slot()
                s.x = torch.empty(first.shape, dtype=first.dtype if first.dtype == torch.uint8 else torch.float32, device=device)
                s.ready, s.free = torch.cuda.Event(), torch.cuda.Event()
                s.n_in = 0
                slots.append(s)
            # result ring: step i writes entry i % 4 and the result of step k is handed out during step k + 1, so the
            # entry is next written by step k + 4 -- after the consumer advanced the generator three more times
            outs = []
            for _ in range(4):
                r = Slot()
                r.out, r.fwd = torch.cuda.Event(), torch.cuda.Event()
                r.det = r.cnt = r.det_h = r.cnt_h = None
                r.n = 0
                if to_host:
                    r.det_h = torch.empty(Bmax, max_det, 6, dtype=torch.float32).pin_memory()
                    r.cnt_h = torch.empty(Bmax, dtype=torch.int32).pin_memory()
                outs.append(r)
            state = self._stream_state[skey] = (torch.cuda.Stream(device=device), slots, outs, torch.cuda.Stream(device=device))
        copy_s, slots, outs, post_s = state
        copy_s.wait_stream(main_s)   # a previous generator's last step may still read the slots
        post_s.wait_stream(main_s)
        for s in slots:
            s.free.record(main_s)

        def stage(s, xb):
            if xb.shape[0] > Bmax or xb.shape[1:] != first.shape[1:]:
                raise ValueError("predict_stream: later batches must not exceed the first batch's shape")
            s.n_in = xb.shape[0]
            s.direct = xb if xb.is_cuda else None
            if xb.is_cuda:   # already resident: no staging copy
                s.ready.record(main_s)
                return
            with torch.cuda.stream(copy_s):
                copy_s.wait_event(s.free)  # the step that last read this slot has finished
                s.x[: s.n_in].copy_(xb, non_blocking=True)
                s.ready.record(copy_s)

        stage(slots[0], first)
        i, pending = 0, None
        while True:
            s = slots[i % 2]
            try:
                nxt = next(it)
            except StopIteration:
                nxt = None
            if nxt is not None:
                stage(slots[(i + 1) % 2], nxt)
            r = outs[i % 4]
            main_s.wait_event(s.ready)
            r.n = s.n_in
            xin = s.direct if s.direct is not None else s.x[: r.n]
            if camera == "nv12":
                hh = xin.shape[1] * 2 // 3
                y = self.forward_camera(xin[:, :hh], None, norm, xin[:, hh:])
            elif camera == "bgra":
                y = self.forward_camera(xin, size, norm, None, letterbox)
            elif r.n <= self.GRAPH_MAX_BATCH and os.environ.get("UYD_NO_GRAPH", "0") != "1":
                y = None   # small batches replay the whole step as one CUDA graph
                r.det, r.cnt = self.predict_batched(xin, conf, iou, max_det, max_nms, classes=classes, agnostic=agnostic,
                                                    multi_label=multi_label)
            else:
                y = self.forward(xin, raw_heads=False)
            s.free.record(main_s)
            r.fwd.record(main_s)
            with torch.cuda.stream(post_s):
                post_s.wait_event(r.fwd)
                if y is not None:
                    y.record_stream(post_s)
                    r.det, r.cnt = self.nms(y, conf, iou, max_det, max_nms, classes=classes, agnostic=agnostic,
                                            multi_label=multi_label)
                    if letterbox:
                        h0, w0 = xin.shape[1:3]
                        P.letterbox_boxes(r.det, r.cnt, h0, w0, *P.camera_extent(h0, w0, size, True))
                if to_host:
                    r.det_h[: r.n].copy_(r.det, non_blocking=True)
                    r.cnt_h[: r.n].copy_(r.cnt, non_blocking=True)
                r.out.record(post_s)
            del y
            if pending is not None:
                yield self._stream_result(pending, to_host, main_s)
            pending = r
            i += 1
            if nxt is None:
                break
        yield self._stream_result(pending, to_host, main_s)

    @staticmethod
    def _stream_result(s, to_host, main_s):
        if to_host:
            s.out.synchronize()
            return s.det_h[: s.n], s.cnt_h[: s.n]
        main_s.wait_event(s.out)   # device results were produced on the post-processing stream
        s.det.record_stream(main_s)
        s.cnt.record_stream(main_s)
        return s.det, s.cnt
