"""``UninaCustomB200``: the reference's hand-written network ``UNINA_YOLO_DLA`` (model.py:308-365)
as a drop-in module on the libuyd plan: same constructor arguments, same 378-entry
``state_dict`` (``backbone.*``, ``neck.*``, ``head_p{2,3,4}.{cls,reg}_branch.*``), same forward
output ``[(cls[B,nc,H,W], reg[B,4,H,W]) x 3]``; ``predict_batched`` adds the TLBR decode and the greedy
class-aware NMS of the reference's post-processing (postprocess.hpp:44-145,
gpu_postprocess.h:42-80) for the whole batch in one launch and returns ``(det[B,max_det,6], count[B])``
on the device; ``predict`` returns per-image ``[N,6]`` rows (x1,y1,x2,y2,conf,cls).
``forward_camera`` / ``predict_camera`` take BGRA or NV12 camera bytes, which the stem reads, normalises
and resamples itself (no fp32 input tensor).  ``calibrate_int8`` / ``set_quantization`` / QAT checkpoints switch the
convs outside the float layers to INT8 (quant.py), with the YAML network's code (yolo.emit_quant_conv).
"""
from __future__ import annotations

import ctypes as C
import os
import types

import torch
import torch.nn as nn

from . import _lib
from . import quant as Q
from ._lib import UYD_F32, Detection, check
from . import preprocess as P
from .preprocess import norm_params
from .plan import NETWORK_INPUT, Plan, Slice
from .yolo import Conv, emit_plain_conv


class ConvBlock(nn.Module):
    """model.py:23-50 -- parameters under ``conv.*`` / ``bn.*`` (BN eps 1e-5)."""

    def __init__(self, cin, cout, k=3, s=1):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, k, s, k // 2, bias=False)
        self.bn = nn.BatchNorm2d(cout)
        self.act = nn.ReLU(inplace=True)
        self.k, self.s, self.g, self.c1, self.c2, self.cout = k, s, 1, cin, cout, cout

    # the YAML network's Conv + BN + ReLU emit: bf16 conv, or in the INT8 graph the quantised conv (with ``feeds``: this
    # output written as the next quantised conv's int8 input); a conv that reads the network input stays float
    emit = Conv.emit


class Bottleneck(nn.Module):
    """model.py:53-73 with expansion 1.0: 1x1 -> 3x3, residual."""

    def __init__(self, c):
        super().__init__()
        self.cv1 = ConvBlock(c, c, 1)
        self.cv2 = ConvBlock(c, c, 3)
        self.add = True

    def emit(self, p, src, dst=None):
        return self.cv2.emit(p, self.cv1.emit(p, src, feeds=self.cv2.conv), dst, res=src)


class C3k2(nn.Module):
    """model.py:76-110: cv3(cat(bottlenecks(cv1(x)), cv2(x)))."""

    def __init__(self, cin, cout, n=1):
        super().__init__()
        h = int(cout * 0.5)
        self.h = h
        self.cv1 = ConvBlock(cin, h, 1)
        self.cv2 = ConvBlock(cin, h, 1)
        self.bottlenecks = nn.Sequential(*(Bottleneck(h) for _ in range(n)))
        self.cv3 = ConvBlock(2 * h, cout, 1)

    def emit(self, p, src, dst=None):
        cat = p.buffer(src.h, src.w, 2 * self.h)
        t = self.cv1.emit(p, src)
        for i, b in enumerate(self.bottlenecks):
            t = b.emit(p, t, cat.sub(0, self.h) if i == len(self.bottlenecks) - 1 else None)
        self.cv2.emit(p, src, cat.sub(self.h, self.h))
        return self.cv3.emit(p, cat, dst)


class SPPF_DLA(nn.Module):
    """model.py:113-132."""

    def __init__(self, cin, cout, k=5):
        super().__init__()
        self.h = cin // 2
        self.cv1 = ConvBlock(cin, self.h, 1)
        self.cv2 = ConvBlock(self.h * 4, cout, 1)
        self.pool = nn.MaxPool2d(kernel_size=k, stride=1, padding=k // 2)

    def emit(self, p, src, dst=None):
        cat = p.buffer(src.h, src.w, 4 * self.h)
        self.cv1.emit(p, src, cat.sub(0, self.h))
        p.sppf_pool(cat, self.h)
        return self.cv2.emit(p, cat, dst)


class Backbone(nn.Module):
    def __init__(self, base_channels=32, lite_p2=False):
        super().__init__()
        c1, c2, c3, c4 = (base_channels * m for m in (1, 2, 4, 8))
        self.lite_p2 = lite_p2
        self.stem = ConvBlock(3, c1, 3, 2)
        self.stage1_conv = ConvBlock(c1, c2, 3, 2)
        self.stage1_block = ConvBlock(c2, c2, 3) if lite_p2 else C3k2(c2, c2, 1)
        self.stage2_conv = ConvBlock(c2, c3, 3, 2)
        self.stage2_c3k2 = C3k2(c3, c3, 2)
        self.stage3_conv = ConvBlock(c3, c4, 3, 2)
        self.stage3_c3k2 = C3k2(c4, c4, 2)
        self.sppf = SPPF_DLA(c4, c4)
        self.out_channels = [c2, c3, c4]


class Neck(nn.Module):
    def __init__(self, chans):
        super().__init__()
        c2, c3, c4 = chans
        self.lateral_p3 = ConvBlock(c4, c3, 1)
        self.fpn_c3k2_1 = C3k2(c3 * 2, c3, 1)
        self.lateral_p2 = ConvBlock(c3, c2, 1)
        self.fpn_c3k2_2 = C3k2(c2 * 2, c2, 1)
        self.down1 = ConvBlock(c2, c2, 3, 2)
        self.pan_c3k2_1 = C3k2(c2 + c3, c3, 1)
        self.down2 = ConvBlock(c3, c3, 3, 2)
        self.pan_c3k2_2 = C3k2(c3 + c4, c4, 1)
        self.out_channels = [c2, c3, c4]


class DetectionHead(nn.Module):
    """model.py:274-303: decoupled cls (nc) / reg (4, TLBR) branches."""

    def __init__(self, c, nc):
        super().__init__()
        self.cls_branch = nn.Sequential(ConvBlock(c, c, 3), ConvBlock(c, c, 3), nn.Conv2d(c, nc, 1))
        self.reg_branch = nn.Sequential(ConvBlock(c, c, 3), ConvBlock(c, c, 3), nn.Conv2d(c, 4, 1))

    def emit(self, p, f, head: Slice, nc: int):
        for branch, dst in ((self.cls_branch, head.sub(0, nc)), (self.reg_branch, head.sub(nc, 4))):
            # [0] -> [1] -> [2] each have one consumer: in the INT8 graph each writes the next conv's int8 input
            t = branch[1].emit(p, branch[0].emit(p, f, feeds=branch[1].conv), feeds=branch[2], feeds_f32=True)
            emit_plain_conv(p, branch[2], t, dst)


class UninaCustomB200(nn.Module):
    STRIDES = (4, 8, 16)
    # module-name patterns of the convs that stay bf16 in the INT8 graph (QuantSpec.covers: substring match).
    # PARITY UNPINNED: the reference picks them by pattern (train.py:779); SURVEY 3.5 records "stem" and "head_p2", the
    # rest of its list is not known.  The stem stays float whatever the patterns say (it reads the network input).
    FLOAT_LAYERS = ("stem", "head_p2")

    def __init__(self, num_classes: int = 4, base_channels: int = 32, lite_p2: bool = False):
        super().__init__()
        self.num_classes = num_classes
        self.backbone = Backbone(base_channels, lite_p2)
        self.neck = Neck(self.backbone.out_channels)
        for lvl, c in zip((2, 3, 4), self.neck.out_channels):
            setattr(self, f"head_p{lvl}", DetectionHead(c, num_classes))
        for name, mod in self.named_modules():
            if isinstance(mod, nn.Conv2d):
                mod._uyd_name = name            # the key of the pytorch-quantization ``_amax`` buffers
        self.quant = None                       # quant.QuantSpec when the INT8 path is active
        self._plans = {}
        self._post = {}
        self._graphs = {}
        self.eval()

    def refresh(self):
        self._plans.clear()
        self._graphs.clear()

    @torch.no_grad()
    def init_synthetic(self, seed: int = 0, reg_bias: float = 2.0, gain: float = 1.0) -> "UninaCustomB200":
        """Seeded data-free init (see synth.py); a positive reg bias keeps the TLBR boxes from
        inverting (the raw reg output is signed, model.py:296-300)."""
        from .synth import synthetic_init_

        synthetic_init_(self, seed, gain)
        for lvl in (2, 3, 4):
            getattr(self, f"head_p{lvl}").reg_branch[2].bias.fill_(reg_bias)
        self.refresh()
        return self

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """Accepts the reference schema (378 entries) plus, for QAT checkpoints, the pytorch-quantization
        ``<conv>._input_quantizer._amax`` / ``<conv>._weight_quantizer._amax`` buffers, which switch the INT8 path on
        with the default float layers."""
        plain, amax = Q.split_state_dict(state_dict)
        out = super().load_state_dict(plain, strict=strict, assign=assign)
        if amax:
            self.set_quantization(amax)
        self.refresh()
        return out

    def set_quantization(self, amax: dict | None, float_layers=FLOAT_LAYERS) -> "UninaCustomB200":
        """Switches the INT8 path on (``amax``: conv module name -> (input amax, weight amax)) or off (None).
        Convs whose module name contains one of ``float_layers`` stay bf16 (see FLOAT_LAYERS, PARITY UNPINNED), so do
        convs without an entry and the stem."""
        self.quant = Q.QuantSpec(dict(amax), tuple(float_layers)) if amax else None
        self.refresh()
        return self

    def quant_state_dict(self) -> dict:
        """The ``_amax`` buffers of the active quantisation in pytorch-quantization's naming."""
        return Q.amax_state_dict(self.quant)

    @torch.no_grad()
    def calibrate_int8(self, frames: torch.Tensor, float_layers=FLOAT_LAYERS, enable: bool = True, method: str = "max",
                       batch_size: int = 8, percentile: float = 99.99) -> dict:
        """Static INT8 scales from a calibration set, as ``UninaYoloB200.calibrate_int8`` computes them: ``frames``
        [N,3,H,W] walked in chunks of ``batch_size`` through the bf16 plan; ``method`` "max" (max |x|), "histogram" /
        "entropy" (the reference's default), "percentile" or "mse"; weights use the same rule on the host.  Returns
        ``{conv name: (amax_in, amax_w)}`` for every conv but the stem and, with ``enable``, switches the INT8 path on."""
        rule = Q.calibration_rule(method)
        saved, self.quant = self.quant, None
        try:
            x_all = self._prep(frames)
            _, _, H, W = x_all.shape
            B = min(batch_size, x_all.shape[0])
            dev = x_all.device.index if x_all.device.index is not None else torch.cuda.current_device()
            p = self._build_plan(dev, B, H, W, record_inputs=True)
            names = [n for n, s in p.conv_inputs.items() if s.buf >= 0]
            a_in = Q.collect_input_amax(p, x_all, B, names, rule, percentile)
        finally:
            self.quant = saved
        convs = {n: m for n, m in self.named_modules() if isinstance(m, nn.Conv2d)}
        amax = {n: (max(a, 1e-6), Q.weight_amax(convs[n].weight, rule, percentile)) for n, a in zip(names, a_in)}
        if enable:
            self.set_quantization(amax, float_layers)
        return amax

    def _apply(self, fn, recurse=True):
        self._plans.clear()
        self._graphs.clear()
        return super()._apply(fn, recurse)

    def _build_plan(self, device, max_batch, H, W, record_inputs: bool = False) -> Plan:
        """``record_inputs`` keeps the input slice of every conv in ``plan.conv_inputs`` (calibration)."""
        p = Plan(device, max_batch)
        p.in_hw = (H, W)
        p.quant = self.quant
        if record_inputs:
            p.conv_inputs = {}
        bb, nk, nc = self.backbone, self.neck, self.num_classes
        c2, c3, c4 = bb.out_channels
        h2, w2 = H // 4, W // 4
        # concat buffers of the neck (model.py:257-267): producers write their slice directly
        cat_f3 = p.buffer(h2 // 2, w2 // 2, 2 * c3)   # [up(lateral_p3(sppf)), p3]
        cat_f2 = p.buffer(h2, w2, 2 * c2)             # [up(lateral_p2(f3)), p2]
        cat_o3 = p.buffer(h2 // 2, w2 // 2, c2 + c3)  # [down1(f2), f3]
        cat_o4 = p.buffer(h2 // 4, w2 // 4, c3 + c4)  # [down2(o3), p4]
        stem = bb.stem.emit(p, NETWORK_INPUT)
        x = bb.stage1_conv.emit(p, stem)
        p2 = bb.stage1_block.emit(p, x, cat_f2.sub(c2, c2))
        p3 = bb.stage2_c3k2.emit(p, bb.stage2_conv.emit(p, p2), cat_f3.sub(c3, c3))
        p4 = bb.stage3_c3k2.emit(p, bb.stage3_conv.emit(p, p3), cat_o4.sub(c3, c4))
        ctx = bb.sppf.emit(p, p4)
        p.upsample2x(nk.lateral_p3.emit(p, ctx), cat_f3.sub(0, c3))
        f3 = nk.fpn_c3k2_1.emit(p, cat_f3, cat_o3.sub(c2, c3))
        p.upsample2x(nk.lateral_p2.emit(p, f3), cat_f2.sub(0, c2))
        f2 = nk.fpn_c3k2_2.emit(p, cat_f2)
        nk.down1.emit(p, f2, cat_o3.sub(0, c2))
        o3 = nk.pan_c3k2_1.emit(p, cat_o3)
        nk.down2.emit(p, o3, cat_o4.sub(0, c3))
        o4 = nk.pan_c3k2_2.emit(p, cat_o4)
        heads = []
        for lvl, f in zip((2, 3, 4), (f2, o3, o4)):
            head = p.buffer(f.h, f.w, nc + 4, UYD_F32)
            getattr(self, f"head_p{lvl}").emit(p, f, head, nc)
            heads.append(head)
        p.heads = heads
        p.feature_slices = {"stem": stem, "p2": p2, "p3": p3, "p4": p4, "sppf": ctx, "f2": f2, "o3": o3, "o4": o4}
        p.finalize()
        # uyd_nms_tlbr reads the head buffers in place: their device pointers and grids, as C arrays, once per plan
        ptrs = []
        for h in heads:
            ptr = C.c_void_p()
            check(_lib.lib().uyd_plan_buffer_ptr(p.handle, h.buf, C.byref(ptr)), "uyd_plan_buffer_ptr")
            ptrs.append(ptr.value)
        n = len(heads)
        p.tlbr_levels = ((C.c_void_p * n)(*ptrs), (C.c_int * n)(*[h.h for h in heads]), (C.c_int * n)(*[h.w for h in heads]),
                         (C.c_int * n)(*self.STRIDES))
        return p

    def plan_for(self, x) -> Plan:
        B, _, H, W = x.shape
        dev = x.device.index if x.device.index is not None else torch.cuda.current_device()
        p = self._plans.get((dev, H, W))
        if p is None or p.max_batch < B:
            if H % 32 or W % 32:
                raise ValueError("frame height/width must be multiples of 32")
            p = self._build_plan(dev, B, H, W)
            self._plans[(dev, H, W)] = p
        return p

    @torch.no_grad()
    def forward(self, x: torch.Tensor):
        """``[(cls, reg)] x 3`` NCHW fp32 (ONNX names p2_cls, p2_reg, ... model.py:382-383)."""
        x = self._prep(x)
        p = self.plan_for(x)
        p.run(x)
        return self._heads(p, x.shape[0], x.device)

    def _heads(self, p: Plan, B: int, device) -> list:
        nc = self.num_classes
        outs = []
        for h in p.heads:
            t = torch.empty(B, nc + 4, h.h, h.w, dtype=torch.float32, device=device)
            self._export(p, h, t, B)
            outs.append((t[:, :nc], t[:, nc:]))
        return outs

    def _prep(self, x: torch.Tensor) -> torch.Tensor:
        if self.training:
            raise RuntimeError("UninaCustomB200 implements the inference path only: call .eval()")
        if not torch.cuda.is_available():
            raise _lib.UydError("no CUDA device: the B200 path has no CPU fallback")
        if not x.is_cuda:
            x = x.cuda(non_blocking=True)
        return x.contiguous() if x.dtype == torch.uint8 else x.float().contiguous()

    @staticmethod
    def _export(p: Plan, h: Slice, out: torch.Tensor, batch: int):
        # NHWC fp32 head buffer -> NCHW through a plain permute of a device copy
        out.copy_(p.read(h, batch))

    def _nms_tlbr_into(self, p: Plan, batch: int, det, cnt, conf, iou, conformal_q, strict, max_det, max_nms) -> None:
        """uyd_nms_tlbr on the plan's head buffers, C call only (no allocation): safe inside CUDA-graph capture."""
        heads, gh, gw, strides = p.tlbr_levels
        check(_lib.lib().uyd_nms_tlbr(p.ctx, heads, gh, gw, strides, len(p.heads), batch, self.num_classes, conf, conformal_q,
                                      int(strict), iou, max_nms, max_det, C.c_void_p(det.data_ptr()), C.c_void_p(cnt.data_ptr()),
                                      C.c_void_p(torch.cuda.current_stream(p.device).cuda_stream)), "uyd_nms_tlbr")

    # batches up to this size replay a captured CUDA graph of the whole step (the plan's launches + one NMS launch are
    # launch-latency-bound below it); larger batches are launched directly.
    GRAPH_MAX_BATCH = 8

    def _graph_for(self, x: torch.Tensor, conf, iou, conformal_q, strict, max_det, max_nms):
        B, _, H, W = x.shape
        dev = x.device.index if x.device.index is not None else torch.cuda.current_device()
        key = (dev, B, H, W, x.dtype, float(conf), float(iou), float(conformal_q), bool(strict), int(max_det), int(max_nms))
        g = self._graphs.get(key)
        if g is not None:
            return g
        xs = torch.empty_like(x)
        det = torch.empty(B, max_det, 6, dtype=torch.float32, device=x.device)
        cnt = torch.empty(B, dtype=torch.int32, device=x.device)
        p = self.plan_for(xs)

        def body():
            p.run(xs)
            self._nms_tlbr_into(p, B, det, cnt, conf, iou, conformal_q, strict, max_det, max_nms)

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
        g = (graph, xs, det, cnt, p)  # the graph reads xs and writes the plan's buffers, det and cnt: keep them alive
        self._graphs[key] = g
        return g

    @torch.no_grad()
    def predict_batched(self, x: torch.Tensor, conf: float = 0.5, iou: float = 0.45, conformal_q: float = 0.0,
                        strict: bool = True, max_det: int = 1024, max_nms: int = 0, graph: bool | None = None):
        """Forward + TLBR decode + NMS of the whole batch, everything left on the device: (det[B,max_det,6], count[B]),
        rows (x1,y1,x2,y2,conf,cls) in kept order, zeros past the count.  One NMS launch reads the plan's head buffers in
        place (uyd_nms_tlbr); max_nms > 0 lets only the max_nms most confident cells of an image enter the NMS (ties: lower
        cell index).  ``graph`` (default: batch <= GRAPH_MAX_BATCH) replays the whole step as one CUDA graph."""
        x = self._prep(x)
        if graph is None:
            graph = x.shape[0] <= self.GRAPH_MAX_BATCH and os.environ.get("UYD_NO_GRAPH", "0") != "1"
        if graph:
            with torch.cuda.device(x.device):   # capture and replay on the frames' device, whatever the caller's current one is
                g, xs, det, cnt, _ = self._graph_for(x, conf, iou, conformal_q, strict, max_det, max_nms)
                xs.copy_(x)
                g.replay()
                return det.clone(), cnt.clone()
        p = self.plan_for(x)
        B = x.shape[0]
        # uyd_nms_tlbr defines every output element: no fill launches
        det = torch.empty(B, max_det, 6, dtype=torch.float32, device=x.device)
        cnt = torch.empty(B, dtype=torch.int32, device=x.device)
        p.run(x)
        self._nms_tlbr_into(p, B, det, cnt, conf, iou, conformal_q, strict, max_det, max_nms)
        return det, cnt

    def _camera(self, frames: torch.Tensor, size, norm, uv, letterbox=False):
        """(plan, uyd_camera_frames, batch) for camera bytes on the device; see forward_camera."""
        if self.training:
            raise RuntimeError("UninaCustomB200 implements the inference path only: call .eval()")
        if not (frames.is_cuda and frames.dtype == torch.uint8 and frames.stride(-1) == 1):
            raise ValueError("frames must be uint8 device bytes with unit stride in the last dimension")
        nv12 = uv is not None
        if nv12 and letterbox:
            raise ValueError("letterbox reads packed BGRA frames; NV12 frames are not letterboxed")
        if nv12:
            if frames.dim() != 3 or not (uv.is_cuda and uv.dtype == torch.uint8 and uv.stride(-1) == 1 and uv.dim() == 3
                                         and uv.shape[0] == frames.shape[0]):
                raise ValueError("NV12: frames = Y planes [B,H,W], uv = interleaved UV planes [B,H/2,W], uint8 on the device")
        elif frames.dim() != 4 or frames.shape[3] != 4:
            raise ValueError("BGRA frames must be [B,H,W,4]")
        B, H, W = frames.shape[:3]
        oh, ow = (H, W) if nv12 else P.camera_extent(H, W, size, letterbox)
        p = self.plan_for(types.SimpleNamespace(shape=(B, 3, oh, ow), device=frames.device))
        f = _lib.CameraFrames()
        f.format = _lib.CAM_NV12 if nv12 else (_lib.CAM_BGRA_LETTERBOX if letterbox else _lib.CAM_BGRA)
        f.width, f.height = W, H
        f.pitch, f.frame_stride, f.data = frames.stride(1), frames.stride(0), frames.data_ptr()
        if nv12:
            f.uv, f.uv_pitch, f.uv_frame_stride = uv.data_ptr(), uv.stride(1), uv.stride(0)
        f.norm = norm if norm is not None else norm_params()
        return p, f, B

    @torch.no_grad()
    def forward_camera(self, frames: torch.Tensor, size=None, norm=None, uv: torch.Tensor | None = None, letterbox: bool = False):
        """Camera bytes straight into the stem (replaces preprocess_bgra_resize / preprocess_nv12 and the CHW fp32
        tensor, perception_node.cpp:604-612): ``frames`` uint8 device ``[B,H,W,4]`` packed BGRA, resampled bilinearly
        (half-pixel rule) to ``size=(H',W')`` when given, or -- with ``uv`` ``[B,H/2,W]`` -- the Y planes ``[B,H,W]`` of
        NV12 frames (BT.601).  Rows may be padded (any pitch; BGRA pitch and frame stride multiples of 4).
        ``norm``: ``_lib.NormParams``, default ImageNet (``preprocess.norm_params()``), what the node feeds this network
        (NormParams() in perception_node.cpp); ``UninaYoloB200.forward_camera`` defaults to plain x / 255 instead.
        ``letterbox``: BGRA frames of any extent are letterboxed as the Ultralytics predictor does (aspect-kept cv2
        INTER_LINEAR resize, grey 114 around it) into ``size``, by default ``preprocess.letterbox_shape(H, W)``.
        Returns ``[(cls, reg)] x 3`` as ``forward`` does.  Only the base_channels-32 stem (Conv 3 -> 32) has a camera
        loader: other widths raise ``UydError`` (UYD_E_UNSUPPORTED)."""
        p, f, B = self._camera(frames, size, norm, uv, letterbox)
        p.run_camera(f, B)
        return self._heads(p, B, frames.device)

    def _camera_graph_for(self, frames: torch.Tensor, size, norm, uv, conf, iou, conformal_q, strict, max_det, max_nms,
                          letterbox=False):
        dev = frames.device.index if frames.device.index is not None else torch.cuda.current_device()
        n = norm if norm is not None else norm_params()
        key = ("camera", dev, tuple(frames.shape), uv is not None, tuple(uv.shape) if uv is not None else None,
               tuple(size) if size is not None else None, (n.mean_r, n.mean_g, n.mean_b, n.std_r, n.std_g, n.std_b),
               float(conf), float(iou), float(conformal_q), bool(strict), int(max_det), int(max_nms), bool(letterbox))
        g = self._graphs.get(key)
        if g is not None:
            return g
        fs = torch.empty(frames.shape, dtype=torch.uint8, device=frames.device)   # static, contiguous frame buffers
        uvs = torch.empty(uv.shape, dtype=torch.uint8, device=frames.device) if uv is not None else None
        p, f, B = self._camera(fs, size, n, uvs, letterbox)
        det = torch.empty(B, max_det, 6, dtype=torch.float32, device=frames.device)
        cnt = torch.empty(B, dtype=torch.int32, device=frames.device)

        def body():
            p.run_camera(f, B)
            self._nms_tlbr_into(p, B, det, cnt, conf, iou, conformal_q, strict, max_det, max_nms)
            if letterbox:
                P.letterbox_boxes(det, cnt, f.height, f.width, *P.camera_extent(f.height, f.width, size, True))

        fs.copy_(frames)
        if uv is not None:
            uvs.copy_(uv)
        side = torch.cuda.Stream(device=frames.device)
        side.wait_stream(torch.cuda.current_stream(frames.device))
        with torch.cuda.stream(side):  # warm-up outside capture (and the plan's argument checks)
            body()
        torch.cuda.current_stream(frames.device).wait_stream(side)
        torch.cuda.synchronize(frames.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body()
        g = (graph, fs, uvs, det, cnt, p, f)  # the graph reads fs / uvs and writes the plan's buffers, det and cnt
        self._graphs[key] = g
        return g

    @torch.no_grad()
    def predict_camera(self, frames: torch.Tensor, size=None, norm=None, uv=None, conf: float = 0.5, iou: float = 0.45,
                       conformal_q: float = 0.0, strict: bool = True, max_det: int = 1024, max_nms: int = 0,
                       graph: bool | None = None, letterbox: bool = False):
        """``forward_camera`` + TLBR decode + NMS, everything on the device: ``(det[B,max_det,6], count[B])`` as
        ``predict_batched`` returns them, with the same thresholds; frames, ``size``, ``uv`` and ``norm`` (default
        ImageNet, unlike ``UninaYoloB200.predict_camera``'s plain x / 255) as in ``forward_camera``.  ``graph``
        (default: batch <= GRAPH_MAX_BATCH) replays the whole step as one CUDA graph that reads static frame buffers;
        each call copies the frames into them.  With ``letterbox`` (see ``forward_camera``) the rows are in frame pixels
        (Ultralytics ``scale_boxes`` + ``clip_boxes``, one launch, inside the graph when there is one)."""
        if graph is None:
            graph = frames.shape[0] <= self.GRAPH_MAX_BATCH and os.environ.get("UYD_NO_GRAPH", "0") != "1"
        if graph:
            with torch.cuda.device(frames.device):
                g, fs, uvs, det, cnt, _, _ = self._camera_graph_for(frames, size, norm, uv, conf, iou, conformal_q, strict,
                                                                    max_det, max_nms, letterbox)
                fs.copy_(frames)
                if uv is not None:
                    uvs.copy_(uv)
                g.replay()
                return det.clone(), cnt.clone()
        p, f, B = self._camera(frames, size, norm, uv, letterbox)
        det = torch.empty(B, max_det, 6, dtype=torch.float32, device=frames.device)
        cnt = torch.empty(B, dtype=torch.int32, device=frames.device)
        p.run_camera(f, B)
        self._nms_tlbr_into(p, B, det, cnt, conf, iou, conformal_q, strict, max_det, max_nms)
        if letterbox:
            P.letterbox_boxes(det, cnt, f.height, f.width, *P.camera_extent(f.height, f.width, size, True))
        return det, cnt

    @torch.no_grad()
    def predict(self, x: torch.Tensor, conf: float = 0.5, iou: float = 0.45, conformal_q: float = 0.0,
                strict: bool = True, cap: int = 0):
        """Decode + NMS with the reference's runtime thresholds (config/params.yaml:13-14).
        Returns per-image ``[N,6]`` tensors (x1,y1,x2,y2,conf,cls), N <= 1024 (MAX_DETECTIONS), in kept order.
        ``cap`` > 0: only the ``cap`` most confident cells of an image enter the NMS (``predict_batched``'s max_nms)."""
        det, cnt = self.predict_batched(x, conf, iou, conformal_q, strict, 1024, cap)
        return [det[b, :n] for b, n in enumerate(cnt.tolist())]

    @torch.no_grad()
    def _predict_per_image(self, x: torch.Tensor, conf: float = 0.5, iou: float = 0.45, conformal_q: float = 0.0,
                           strict: bool = True, cap: int = 0):
        """The per-image composition ``predict`` had before ``predict_batched``: head export, then per image three
        ``uyd_decode_tlbr`` launches, one ``uyd_nms_detections`` launch and a host read of the count.  Kept as the
        reference the batched path is tested against and as the baseline of tools/custom_predict_bench.py; ``cap``
        smaller than the cell count keeps the cells that win the decode's atomic slots, not the most confident ones."""
        outs = self.forward(x)
        B = outs[0][0].shape[0]
        dev = outs[0][0].device
        di = dev.index if dev.index is not None else torch.cuda.current_device()
        L = _lib.lib()
        ctx = _lib.context(di)
        cells = sum(c.shape[2] * c.shape[3] for c, _ in outs)
        cap = cap or cells
        ws_bytes = int(L.uyd_nms_detections_workspace_bytes(cap))
        dets = torch.zeros(cap, 8, dtype=torch.float32, device=dev)          # 32-byte records
        kept = torch.zeros(1024, 8, dtype=torch.float32, device=dev)
        cell = torch.zeros(cap, dtype=torch.int32, device=dev)
        cnt = torch.zeros(2, dtype=torch.int32, device=dev)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        stream = C.c_void_p(torch.cuda.current_stream(di).cuda_stream)
        results = []
        for b in range(B):
            cnt.zero_()
            base = 0
            for (cls, reg), stride in zip(outs, self.STRIDES):
                gh, gw = cls.shape[2], cls.shape[3]
                cb, rb = cls[b].contiguous(), reg[b].contiguous()
                check(L.uyd_decode_tlbr(ctx, C.c_void_p(cb.data_ptr()), C.c_void_p(rb.data_ptr()), C.c_void_p(dets.data_ptr()),
                                        C.c_void_p(cell.data_ptr()), C.c_void_p(cnt.data_ptr()), cap, gw, gh, stride,
                                        self.num_classes, conf, conformal_q, int(strict), base, stream), "uyd_decode_tlbr")
                base += gh * gw
            check(L.uyd_nms_detections(ctx, C.c_void_p(dets.data_ptr()), C.c_void_p(cell.data_ptr()), C.c_void_p(cnt.data_ptr()), cap, iou,
                                       C.c_void_p(ws.data_ptr()), ws_bytes, C.c_void_p(kept.data_ptr()),
                                       C.c_void_p(cnt[1:].data_ptr()), stream), "uyd_nms_detections")
            n = int(cnt[1].item())
            k = kept[:n]
            rows = torch.cat((k[:, :5], k[:, 5:6].view(torch.int32).float()), 1)
            results.append(rows.clone())
        return results
