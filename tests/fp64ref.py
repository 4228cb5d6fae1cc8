"""fp64 references of the bf16 kernels' ops with a derived per-element error bound (CPU, torch).

Every function returns ``(ref, slack)`` as fp64 tensors.  ``ref`` is the exact result on the operands the kernel
sees (bf16-rounded activations and weights, fp32 biases); ``slack`` bounds |kernel - ref| element by element for a
correct kernel.  For one conv over K = cin/groups * k * k terms:

    slack = 2 K 2^-24 (|x| * |w| + |b|)      fp32 accumulation in any order (FMA products are exact)
          + |slack_in| * |w|                 error carried in from a fused predecessor
          + 2^-24 |ref|                      one fp32 add of a residual or of upsampled partial sums

(* is the same convolution.)  ReLU is 1-Lipschitz and does not widen the bound.  An output rounded to bf16 is
bounded by rounding both ends of [ref - slack, ref + slack] (bf16_interval): the result is one bf16 value where
both ends round alike, and spans at most the two neighbours (< 2^-8 |ref| + slack) where they do not.  A fused
block carries this interval from stage to stage, so the next stage inherits slack only from elements whose
rounding the fp32 error could flip; bounding every intermediate by 2^-8 |ref| instead grows by sum|w| (~10 for
these 3x3 convs) per stage and says nothing after four.  Even so, flipped roundings spread through the four 3x3
stages of a C3k block in proportion to their sum|w|: with unit-gain weights the median slack / |ref| at the output
reaches 1.0 (c = 32, 80 x 40) and the bound passes truncated weights.  The C3k bound cases therefore draw their 3x3
weights at gain 0.4 (c3k_operands; median <= 0.012, max slack <= 0.006 max|ref| at every GPU case's shape), and
the unit-gain C3k tests keep their whole-tensor check beside the bound.  The measured worst |err| / slack of every
kernel instance is in profiles/r04_kernel_bounds.md.  Frame inputs carry their own representation error:
hi + lo bf16 planes (conv_stem_mma_kernel) are exact to 2^-17 relative, tf32 rounding (stem_v2_kernel) to 2^-11.

The bound is never scaled by a per-case constant; the same formula serves the CUDA-core and the tensor-core kernels.
"""
from __future__ import annotations

import json
import os
import re

import torch
import torch.nn.functional as F

U32 = 2.0 ** -24          # fp32 unit roundoff
FRAME_HILO = 2.0 ** -17   # fp32 frame split into hi + lo bf16 planes
FRAME_TF32 = 2.0 ** -11   # fp32 frame rounded to tf32
FRAME_BF16 = 2.0 ** -9    # fp32 frame rounded to bf16 (the hi plane alone)

__all__ = ["bf16", "bf16_interval", "conv", "upsample2x", "chain", "c3k", "c3k_operands", "cls_branch", "stem2", "max_pool_cascade",
           "kernel_id", "assert_within"]


def bf16(t: torch.Tensor) -> torch.Tensor:
    """The fp64 value of t rounded to bf16 (round to nearest even)."""
    return t.float().to(torch.bfloat16).double()


def _d(t):
    return None if t is None else torch.as_tensor(t).double()


def upsample2x(t: torch.Tensor) -> torch.Tensor:
    return t.repeat_interleave(2, 2).repeat_interleave(2, 3)


def conv(x, w, b, *, stride=1, groups=1, relu=True, res=None, res_slack=None, bf16_out=False, slack_in=None,
         pre=None, pre_slack=None):
    """Conv(k x k, padding k // 2) + bias [+ upsampled partial sums ``pre``] [ReLU] [+ residual] [-> bf16].

    ``x`` and ``w`` must already hold the values the kernel reads (bf16-rounded); ``w`` is [cout, cin/groups, k, k].
    ``pre`` is [n, cout, h/2, w/2], added before the activation (the Upsample + Concat + 1x1 fold)."""
    x, w, b = _d(x), _d(w), _d(b)
    k = w.shape[-1]
    kw = dict(stride=stride, padding=k // 2, groups=groups)
    K = w.shape[1] * k * k
    ref = F.conv2d(x, w, None, **kw) + b.view(1, -1, 1, 1)
    mag = F.conv2d(x.abs(), w.abs(), None, **kw) + b.abs().view(1, -1, 1, 1)
    slack = 2 * K * U32 * mag
    if slack_in is not None:
        slack = slack + F.conv2d(_d(slack_in), w.abs(), None, **kw)
    if pre is not None:
        up = upsample2x(_d(pre))
        ref = ref + up
        slack = slack + U32 * (mag + up.abs())
        if pre_slack is not None:
            slack = slack + upsample2x(_d(pre_slack))
    if relu:
        ref = ref.clamp_min(0)
    if res is not None:
        ref = ref + _d(res)
        slack = slack + U32 * ref.abs()
        if res_slack is not None:
            slack = slack + _d(res_slack)
    if bf16_out:
        lo, hi = ref - slack, ref + slack
        if relu and res is None:
            lo = lo.clamp_min(0)
        return bf16_interval(lo, hi)
    return ref, slack


def bf16_interval(lo, hi):
    """(centre, half-width) of the bf16 values an fp32 number in [lo, hi] rounds to (round to nearest even).

    fp32 and bf16 rounding are both monotone, so the kernel's bf16 value lies in [bf16(lo), bf16(hi)].  Where both
    ends round alike the output is known exactly and carries no slack into the next stage; where they differ the
    interval spans the neighbours, at most 2^-8 |value| wide for the slacks of these ops."""
    lo, hi = bf16(lo), bf16(hi)
    return (lo + hi) / 2, (hi - lo) / 2


def chain(x, w1, b1, w2, b2, *, dw1=False, relu2=False, bf16_2=False, w3=None, b3=None):
    """conv_chain: 3x3 conv (dense or depth-wise) + ReLU -> bf16 -> 1x1 conv [+ ReLU] [-> bf16 -> 1x1 conv]."""
    w2 = _d(w2).reshape(w2.shape[0], -1, 1, 1)
    t, st = conv(x, w1, b1, groups=x.shape[1] if dw1 else 1, bf16_out=True)
    u, su = conv(t, w2, b2, relu=relu2, bf16_out=bf16_2 or w3 is not None, slack_in=st)
    if w3 is None:
        return u, su
    return conv(u, _d(w3).reshape(w3.shape[0], -1, 1, 1), b3, relu=False, slack_in=su)


def c3k(x, ws, bs):
    """C3k block, ws / bs = [cv1, cv2, m0.cv1, m0.cv2, m1.cv1, m1.cv2, cv3]; every stage writes bf16."""
    cb = lambda t, s, i, **kw: conv(t, ws[i], bs[i], bf16_out=True, slack_in=s, **kw)
    a, sa = cb(x, None, 0)
    b, sb = cb(x, None, 1)
    t, st = cb(a, sa, 2)
    u, su = cb(t, st, 3, res=a, res_slack=sa)
    t, st = cb(u, su, 4)
    v, sv = cb(t, st, 5, res=u, res_slack=su)
    return cb(torch.cat((v, b), 1), torch.cat((sv, sb), 1), 6)


C3K_GAIN3 = 0.4   # gain of the 3x3 weights in the C3k bound cases (c3k_operands)


def c3k_operands(c, H, W, B, seed=None, gain3=C3K_GAIN3):
    """Seeded C3k operands (fp32, not rounded): x, ws, bs for c3k().  The worst-case carry through the four 3x3
    stages grows with sum|w| of each; at unit gain (sum|w| ~ 10) it passes truncated weights or a missing bias, at
    gain 0.4 every such fault breaks the bound in thousands of elements (test_fp64ref_host.py)."""
    g = torch.Generator().manual_seed(c + H + W + B if seed is None else seed)
    h = c // 2
    shapes = [(h, c, 1), (h, c, 1), (h, h, 3), (h, h, 3), (h, h, 3), (h, h, 3), (c, c, 1)]
    ws = [torch.randn(co, ci, k, k, generator=g) / (ci * k * k) ** 0.5 * (gain3 if k == 3 else 1.0) for co, ci, k in shapes]
    bs = [torch.randn(co, generator=g) * 0.1 for co, _, _ in shapes]
    return torch.randn(B, c, H, W, generator=g), ws, bs


def cls_branch(x, ws, bs):
    """Detect class branch: dw3x3 -> 1x1 -> dw3x3 -> 1x1 (bf16 between stages, ReLU) -> 1x1 logits (fp32)."""
    t, s = conv(x, ws[0], bs[0], groups=x.shape[1], bf16_out=True)
    t, s = conv(t, ws[1], bs[1], bf16_out=True, slack_in=s)
    t, s = conv(t, ws[2], bs[2], groups=t.shape[1], bf16_out=True, slack_in=s)
    t, s = conv(t, ws[3], bs[3], bf16_out=True, slack_in=s)
    return conv(t, ws[4], bs[4], relu=False, slack_in=s)


def stem2(frame, w0, b0, w1, b1, w2=None, b2=None, frame_rel=FRAME_TF32):
    """Fused stem: Conv(3,16,3,2) -> Conv(16,32,3,2) [-> 1x1 Conv(32,16)], ReLU and bf16 after each."""
    frame = _d(frame)
    t, s = conv(frame, w0, b0, stride=2, bf16_out=True, slack_in=frame_rel * frame.abs())
    t, s = conv(t, w1, b1, stride=2, bf16_out=True, slack_in=s)
    if w2 is not None:
        t, s = conv(t, _d(w2).reshape(16, 32, 1, 1), b2, bf16_out=True, slack_in=s)
    return t, s


def max_pool_cascade(x):
    """SPPF: the input and three cascaded 5x5 stride-1 max pools, concatenated on channels."""
    y1 = F.max_pool2d(x, 5, 1, 2)
    y2 = F.max_pool2d(y1, 5, 1, 2)
    return torch.cat((x, y1, y2, F.max_pool2d(y2, 5, 1, 2)), 1)


def kernel_id(name: str) -> str:
    """A demangled kernel name (cu++filt or the CUDA profiler) as 'name<arg,...>': no namespaces, casts, spaces or
    parameter list; true / false as 1 / 0."""
    s = name.strip().replace("(anonymous namespace)::", "").replace("<unnamed>::", "")
    s = s[5:] if s.startswith("void ") else s
    depth = 0
    for i, ch in enumerate(s):
        depth += (ch == "<") - (ch == ">")
        if ch == "(" and depth == 0:
            s = s[:i]
            break
    s = re.sub(r"\((?:int|bool|unsigned int)\)", "", s)
    s = re.sub(r"\b\w+::", "", s).replace(" ", "")
    s = re.sub(r"\btrue\b", "1", re.sub(r"\bfalse\b", "0", s))
    return s.replace("unsignedchar", "uint8")


def assert_within(got, ref, slack, what=""):
    """Fails unless |got - ref| <= slack everywhere (NaN fails).  Returns the tightness: the median of slack / |ref|
    over the elements with |ref| > 1e-3 max|ref|.  With UYD_BOUNDS_LOG set, appends one JSON line per call there."""
    got, ref, slack = got.double(), _d(ref), _d(slack)
    assert got.shape == ref.shape == slack.shape, (what, got.shape, ref.shape, slack.shape)
    err = (got - ref).abs()
    bad = ~(err <= slack)
    ratio = torch.where(slack > 0, err / slack, torch.where(err > 0, torch.inf, 0.0)).nan_to_num(nan=torch.inf)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    big = ref.abs() > 1e-3 * float(ref.abs().max())
    tight = float((slack[big] / ref.abs()[big]).median()) if bool(big.any()) else 0.0
    if os.environ.get("UYD_BOUNDS_LOG"):
        with open(os.environ["UYD_BOUNDS_LOG"], "a") as f:
            f.write(json.dumps(dict(what=what, worst=worst, tightness=tight, n=int(ref.numel()))) + "\n")
    if bool(bad.any()):
        i = int(ratio.flatten().argmax())
        idx = tuple(int(v) for v in torch.unravel_index(torch.tensor(i), ratio.shape))
        raise AssertionError(f"{what}: {int(bad.sum())} of {ref.numel()} elements outside the bound; worst at (n, c, y, x) = "
                             f"{idx}: got {float(got[idx]):.9g}, ref {float(ref[idx]):.9g}, |err|/slack = {worst:.3g}")
    return tight
