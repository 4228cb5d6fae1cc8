"""Camera-frame pre-processing on the GPU (reference: ros2_ws/src/perception/src/cuda_preprocess.cu:99-323,
the step in front of the hot path): packed BGRA / NV12 bytes -> the NCHW fp32 tensor ``UninaYoloB200`` consumes."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib
from ._lib import NormParams, check


def norm_params(mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225)) -> NormParams:
    """create_norm_params (cuda_preprocess.h:55-56); the defaults are ImageNet (create_norm_params_imagenet)."""
    return NormParams(*mean, *std)


UNIT = NormParams(0.0, 0.0, 0.0, 1.0, 1.0, 1.0)   # plain x / 255


def _stream(t: torch.Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def bgra(frames: torch.Tensor, params: NormParams = UNIT, size: tuple[int, int] | None = None) -> torch.Tensor:
    """``frames``: uint8 ``[B, H, W, 4]`` (BGRA, device) -> fp32 ``[B, 3, H', W']`` RGB, ``(x/255 - mean)/std``;
    ``size=(H', W')`` resizes with half-pixel bilinear sampling (preprocess_bgra_resize), else H' = H, W' = W."""
    assert frames.is_cuda and frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[3] == 4 and frames.is_contiguous()
    B, H, W, _ = frames.shape
    oh, ow = size or (H, W)
    out = torch.empty(B, 3, oh, ow, dtype=torch.float32, device=frames.device)
    L = _lib.lib()
    with torch.cuda.device(frames.device):   # the reference entry points carry no device: they run on the current one
        return _bgra(L, frames, out, params, size, B, H, W, oh, ow)


def _bgra(L, frames, out, params, size, B, H, W, oh, ow):
    if size is None or (oh, ow) == (H, W):
        check(L.uyd_preprocess_bgra_batch(C.c_void_p(frames.data_ptr()), C.c_void_p(out.data_ptr()), B, H * W * 4, W, H, W * 4,
                                          params, _stream(frames)), "uyd_preprocess_bgra_batch")
    else:
        check(L.uyd_preprocess_bgra_resize_batch(C.c_void_p(frames.data_ptr()), C.c_void_p(out.data_ptr()), B, H * W * 4, W, H,
                                                 W * 4, ow, oh, params, _stream(frames)), "uyd_preprocess_bgra_resize_batch")
    return out


def nv12(y_plane: torch.Tensor, uv_plane: torch.Tensor, params: NormParams = UNIT) -> torch.Tensor:
    """One NV12 frame: ``y_plane`` uint8 ``[H, W]``, ``uv_plane`` uint8 ``[H/2, W]`` (interleaved U, V) -> ``[1, 3, H, W]``."""
    assert y_plane.is_cuda and uv_plane.is_cuda and y_plane.dtype == torch.uint8 and uv_plane.dtype == torch.uint8
    H, W = y_plane.shape
    out = torch.empty(1, 3, H, W, dtype=torch.float32, device=y_plane.device)
    with torch.cuda.device(y_plane.device):
        check(_lib.lib().uyd_preprocess_nv12(C.c_void_p(y_plane.data_ptr()), C.c_void_p(uv_plane.data_ptr()), C.c_void_p(out.data_ptr()),
                                             W, H, y_plane.stride(0), uv_plane.stride(0), params, _stream(y_plane)), "uyd_preprocess_nv12")
    return out


def letterbox_geometry(h0: int, w0: int, H: int, W: int):
    """``(new_w, new_h, left, top, gain)`` of an h0 x w0 frame letterboxed into an H x W model input
    (uyd_letterbox_geometry: the Ultralytics LetterBox / scale_boxes rules)."""
    nw, nh, left, top, gain = C.c_int(), C.c_int(), C.c_int(), C.c_int(), C.c_double()
    check(_lib.lib().uyd_letterbox_geometry(w0, h0, W, H, C.byref(nw), C.byref(nh), C.byref(left), C.byref(top), C.byref(gain)),
          "uyd_letterbox_geometry")
    return nw.value, nh.value, left.value, top.value, gain.value


def letterbox_shape(h0: int, w0: int, imgsz: int = 640, stride: int = 32, auto: bool = True) -> tuple[int, int]:
    """``(H, W)`` of the model input the Ultralytics predictor letterboxes an h0 x w0 frame into: with ``auto`` the
    aspect-kept resize to fit ``imgsz`` padded up to a multiple of ``stride`` (1280 x 720 -> 384 x 640), else
    ``imgsz`` x ``imgsz``."""
    if not auto:
        return imgsz, imgsz
    new_w, new_h = letterbox_geometry(h0, w0, imgsz, imgsz)[:2]
    return new_h + (imgsz - new_h) % stride, new_w + (imgsz - new_w) % stride


def camera_extent(h0: int, w0: int, size, letterbox: bool) -> tuple[int, int]:
    """The plan extent a camera entry point runs h0 x w0 frames at: ``size`` when given, else ``letterbox_shape``
    with ``letterbox``, else the frame's own extent."""
    if size is not None:
        return int(size[0]), int(size[1])
    return letterbox_shape(h0, w0) if letterbox else (h0, w0)


def letterbox_boxes(det: torch.Tensor, count: torch.Tensor, h0: int, w0: int, H: int, W: int) -> None:
    """Rows ``det[b, :count[b]]`` (x1,y1,x2,y2,conf,cls) of a batch letterboxed from h0 x w0 frames into H x W, in place,
    from model-input to frame pixels (uyd_letterbox_boxes: Ultralytics ``scale_boxes`` + ``clip_boxes``).  One launch on
    the current stream, no allocation: usable under CUDA-graph capture."""
    assert det.is_cuda and det.dtype == torch.float32 and det.dim() == 3 and det.shape[2] == 6 and det.is_contiguous()
    assert count.is_cuda and count.dtype == torch.int32 and count.shape[0] == det.shape[0]
    dev = det.device.index if det.device.index is not None else torch.cuda.current_device()
    check(_lib.lib().uyd_letterbox_boxes(_lib.context(dev), C.c_void_p(det.data_ptr()), C.c_void_p(count.data_ptr()), det.shape[0],
                                         det.shape[1], w0, h0, W, H, _stream(det)), "uyd_letterbox_boxes")
