"""Oracle: numpy restatement of the Ultralytics predictor's letterbox and of ``scale_boxes``.  TEST INFRASTRUCTURE.

``LetterBox(center=True, scaleup=True)``: an aspect-preserving ``cv2.resize(INTER_LINEAR)`` of the frame, centred in
the model input with grey 114 around it.  The resize is cv2 4.x's fixed-point INTER_LINEAR for uint8 restated rule by
rule (11-bit coefficients, the SIMD vertical pass's rounding); tests/test_letterbox_host.py pins it byte for byte to
``cv2.resize`` + ``cv2.copyMakeBorder``.  The exact 2x downscale, for which cv2 switches to INTER_AREA, needs no
case of its own: the linear rules give coefficients 1024 / 1024 on the 2x2 block there, i.e. ``(a+b+c+d+2) >> 2``.
"""
from __future__ import annotations

import numpy as np

PAD = 114
COEF_SCALE = 2048  # INTER_RESIZE_COEF_SCALE


def letterbox_geometry(w0: int, h0: int, W: int, H: int):
    """(new_w, new_h, left, top, gain) of a w0 x h0 frame letterboxed into a W x H model input.  Python's round is
    half-to-even, as the C helper's nearbyint."""
    r = min(H / h0, W / w0)
    new_w, new_h = int(round(w0 * r)), int(round(h0 * r))
    return new_w, new_h, int(round((W - new_w) / 2 - 0.1)), int(round((H - new_h) / 2 - 0.1)), r


def letterbox_shape(h0: int, w0: int, imgsz: int = 640, stride: int = 32, auto: bool = True):
    """(H, W) of the model input the Ultralytics predictor letterboxes an h0 x w0 frame into: with ``auto`` the
    resized frame padded to the next multiple of ``stride`` (1280 x 720 -> 384 x 640), else ``imgsz`` square."""
    if not auto:
        return imgsz, imgsz
    r = min(imgsz / h0, imgsz / w0)
    new_w, new_h = int(round(w0 * r)), int(round(h0 * r))
    return new_h + (imgsz - new_h) % stride, new_w + (imgsz - new_w) % stride


def _taps(src: int, dst: int):
    """Source index and fractional weight per output index: cv2's (float)((d + 0.5) * scale - 0.5), floor, remainder."""
    scale = 1.0 / (dst / src)
    f = ((np.arange(dst, dtype=np.float64) + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    return s, (f - s.astype(np.float32)).astype(np.float32)


def _coef(f):
    return (np.rint((np.float32(1) - f) * np.float32(COEF_SCALE)).astype(np.int64),
            np.rint(f * np.float32(COEF_SCALE)).astype(np.int64))


def resize_linear(frame: np.ndarray, new_w: int, new_h: int) -> np.ndarray:
    """cv2.resize(frame, (new_w, new_h), interpolation=INTER_LINEAR) for uint8 [h, w, c]."""
    h0, w0 = frame.shape[:2]
    if (new_w, new_h) == (w0, h0):
        return frame.copy()
    sx, fx = _taps(w0, new_w)
    lo, hi = sx < 0, sx >= w0 - 1            # horizontal borders: the weight is clamped with the index
    fx[lo | hi] = 0
    sx = np.clip(sx, 0, w0 - 1)
    a0, a1 = _coef(fx)
    sy, fy = _taps(h0, new_h)                 # vertical: only the two row indices are clamped
    b0, b1 = _coef(fy)
    p = frame.astype(np.int64)
    hrow = p[:, sx] * a0[None, :, None] + p[:, np.minimum(sx + 1, w0 - 1)] * a1[None, :, None]   # [h0, new_w, c]
    h0r, h1r = hrow[np.clip(sy, 0, h0 - 1)], hrow[np.clip(sy + 1, 0, h0 - 1)]
    out = (((b0[:, None, None] * (h0r >> 4)) >> 16) + ((b1[:, None, None] * (h1r >> 4)) >> 16) + 2) >> 2
    return out.astype(np.uint8)


def letterbox_bgra(frame: np.ndarray, H: int, W: int) -> np.ndarray:
    """uint8 [h0, w0, c] (c = 3 or 4) -> uint8 [H, W, c]: the resized frame at (top, left), PAD everywhere else
    (all channels, alpha included, as cv2.copyMakeBorder with a scalar 114 pads them)."""
    h0, w0, c = frame.shape
    new_w, new_h, left, top, _ = letterbox_geometry(w0, h0, W, H)
    out = np.full((H, W, c), PAD, dtype=np.uint8)
    out[top:top + new_h, left:left + new_w] = resize_linear(frame, new_w, new_h)
    return out


def scale_boxes(boxes: np.ndarray, w0: int, h0: int, W: int, H: int) -> np.ndarray:
    """Rows (x1, y1, x2, y2, ...) in model-input pixels -> frame pixels, fp32: subtract the pad, multiply by the fp32
    reciprocal of the gain (what torch does for ``boxes /= gain`` with a Python float on a CUDA tensor), clamp to the
    frame.  Columns past 4 are returned unchanged."""
    _, _, left, top, gain = letterbox_geometry(w0, h0, W, H)
    out = np.array(boxes, dtype=np.float32, copy=True)
    inv = np.float32(1) / np.float32(gain)
    out[..., [0, 2]] = (out[..., [0, 2]] - np.float32(left)) * inv
    out[..., [1, 3]] = (out[..., [1, 3]] - np.float32(top)) * inv
    out[..., [0, 2]] = np.minimum(np.maximum(out[..., [0, 2]], np.float32(0)), np.float32(w0))
    out[..., [1, 3]] = np.minimum(np.maximum(out[..., [1, 3]], np.float32(0)), np.float32(h0))
    return out


__all__ = ["letterbox_geometry", "letterbox_shape", "resize_linear", "letterbox_bgra", "scale_boxes", "PAD"]
