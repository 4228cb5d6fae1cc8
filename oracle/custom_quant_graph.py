"""Oracle: integer reference of the INT8 (QAT fake-quant) model.py network, ``oracle/custom_graph.CustomNet``.
TEST INFRASTRUCTURE.

PARITY UNPINNED (see oracle/quant.py): the fake-quant arithmetic is the published one as the reference configures it
(qat.py:109-124: 8 bit, narrow range, per-tensor input and weight scales).  Same fixed conventions as
``oracle/quant_graph.Int8Graph``, which the CUDA path implements exactly (raw heads are compared byte for byte):
  * activations between layers are bf16 values; every quantised Conv + BN + ReLU computes
    y = relu(float32(acc) * m_c + b_c) [+ residual, fp32] and rounds y once to bf16;
  * the final biased 1x1 convs of the heads produce fp32 (no rounding);
  * max-pool / upsample / concat act on the bf16 values;
  * the integer sums are formed in fp64 (exact): |acc| reaches 2304 * 127^2 > 2^24 in the 256 -> 256 3x3 heads.
Every conv after the stem is quantised; the stem is not restated: ``forward_from`` starts from the tensor it
produces (the GPU plan's ``feature_slices["stem"]``).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import custom_graph as cg
from .quant_graph import Int8Graph, bf16


class CustomInt8Graph(Int8Graph):
    def __init__(self, model: cg.CustomNet, amax: dict):
        self.model, self.amax = model, amax

    def cbr(self, m: cg.CBR, name: str, x, res=None):
        return self.qconv(m.conv, m.bn, name + ".conv", x, True, res)

    def csp(self, m: cg.CSP, name: str, x):
        a = self.cbr(m.cv1, name + ".cv1", x)
        for j, b in enumerate(m.bottlenecks):
            a = self.cbr(b.cv2, f"{name}.bottlenecks.{j}.cv2", self.cbr(b.cv1, f"{name}.bottlenecks.{j}.cv1", a), res=a)
        return self.cbr(m.cv3, name + ".cv3", torch.cat((a, self.cbr(m.cv2, name + ".cv2", x)), 1))

    def sppf(self, m: cg.PoolPyramid, name: str, x):
        outs = [self.cbr(m.cv1, name + ".cv1", x)]
        for _ in range(3):
            outs.append(F.max_pool2d(outs[-1], m.k, 1, m.k // 2))
        return self.cbr(m.cv2, name + ".cv2", torch.cat(outs, 1))

    def head(self, m: cg._Head, name: str, x):
        out = []
        for br in ("cls_branch", "reg_branch"):
            seq = getattr(m, br)
            t = self.cbr(seq[1], f"{name}.{br}.1", self.cbr(seq[0], f"{name}.{br}.0", x))
            out.append(self.qconv(seq[2], None, f"{name}.{br}.2", t, False, out_bf16=False))
        return tuple(out)

    @torch.no_grad()
    def forward_from(self, stem: torch.Tensor):
        """``stem``: the bf16-valued fp32 NCHW output of the stem.  Returns ``[(cls, reg)] x 3`` fp32 as
        ``CustomNet.forward`` does."""
        bb, nk = self.model.backbone, self.model.neck
        up = lambda t: F.interpolate(t, scale_factor=2, mode="nearest")
        x = self.cbr(bb.stage1_conv, "backbone.stage1_conv", bf16(stem))
        if isinstance(bb.stage1_block, cg.CBR):
            p2 = self.cbr(bb.stage1_block, "backbone.stage1_block", x)
        else:
            p2 = self.csp(bb.stage1_block, "backbone.stage1_block", x)
        p3 = self.csp(bb.stage2_c3k2, "backbone.stage2_c3k2", self.cbr(bb.stage2_conv, "backbone.stage2_conv", p2))
        p4 = self.csp(bb.stage3_c3k2, "backbone.stage3_c3k2", self.cbr(bb.stage3_conv, "backbone.stage3_conv", p3))
        ctx = self.sppf(bb.sppf, "backbone.sppf", p4)
        f3 = self.csp(nk.fpn_c3k2_1, "neck.fpn_c3k2_1", torch.cat((up(self.cbr(nk.lateral_p3, "neck.lateral_p3", ctx)), p3), 1))
        f2 = self.csp(nk.fpn_c3k2_2, "neck.fpn_c3k2_2", torch.cat((up(self.cbr(nk.lateral_p2, "neck.lateral_p2", f3)), p2), 1))
        o3 = self.csp(nk.pan_c3k2_1, "neck.pan_c3k2_1", torch.cat((self.cbr(nk.down1, "neck.down1", f2), f3), 1))
        o4 = self.csp(nk.pan_c3k2_2, "neck.pan_c3k2_2", torch.cat((self.cbr(nk.down2, "neck.down2", o3), p4), 1))
        return [self.head(self.model.head_p2, "head_p2", f2), self.head(self.model.head_p3, "head_p3", o3),
                self.head(self.model.head_p4, "head_p4", o4)]
