"""Letterboxing without a GPU: the numpy restatement of the Ultralytics letterbox (oracle/letterbox.py) against cv2
itself, and the geometry of the library's uyd_letterbox_geometry / preprocess.letterbox_shape against the oracle."""
import numpy as np
import pytest

from oracle import letterbox as lb

# (frame width, frame height) -> (plan height, plan width)
PAIRS = [
    ((1280, 720), (384, 640)),   # exact 2x in both axes: cv2's INTER_AREA switch
    ((1280, 720), (640, 640)),
    ((1920, 1080), (384, 640)),  # 3x
    ((320, 240), (480, 640)),    # upscale
    ((641, 479), (480, 640)),    # odd, 1-row pads
    ((1280, 725), (384, 640)),   # new_h = round(362.5) = 362, half to even
    ((640, 384), (384, 640)),    # already at the plan extent: a copy
]


def _cv2_letterbox(cv2, frame, H, W):
    h0, w0 = frame.shape[:2]
    new_w, new_h, left, top, _ = lb.letterbox_geometry(w0, h0, W, H)
    img = frame if (new_w, new_h) == (w0, h0) else cv2.resize(frame, (new_w, new_h), interpolation=cv2.INTER_LINEAR)
    return cv2.copyMakeBorder(img, top, H - new_h - top, left, W - new_w - left, cv2.BORDER_CONSTANT, value=(114,) * 4)


@pytest.mark.parametrize("channels", [3, 4])
@pytest.mark.parametrize("frame,plan", PAIRS)
def test_oracle_letterbox_equals_cv2(frame, plan, channels):
    cv2 = pytest.importorskip("cv2")
    (w0, h0), (H, W) = frame, plan
    img = np.random.default_rng(w0 * 7 + h0 + channels).integers(0, 256, (h0, w0, channels), dtype=np.uint8)
    got = lb.letterbox_bgra(img, H, W)
    want = _cv2_letterbox(cv2, img, H, W)
    assert got.shape == want.shape == (H, W, channels)
    assert got.tobytes() == want.tobytes()


def test_oracle_geometry_cases():
    assert lb.letterbox_geometry(1280, 720, 640, 384) == (640, 360, 0, 12, 0.5)
    assert lb.letterbox_geometry(1280, 725, 640, 384)[:4] == (640, 362, 0, 11)   # 362.5 -> 362
    assert lb.letterbox_shape(720, 1280) == (384, 640)
    assert lb.letterbox_shape(720, 1280, auto=False) == (640, 640)


def _lib_or_none():
    from unina_yolo_dla_b200 import _lib

    return _lib.lib() if _lib.LIB_PATH.exists() else None


@pytest.mark.parametrize("frame,plan", PAIRS + [((1, 7), (64, 64)), ((1000, 3), (640, 640)), ((33, 17), (96, 128))])
def test_library_geometry_equals_oracle(frame, plan):
    (w0, h0), (H, W) = frame, plan
    want = lb.letterbox_geometry(w0, h0, W, H)
    if _lib_or_none() is None:
        pytest.skip("libuyd.so not built")
    from unina_yolo_dla_b200 import preprocess

    assert preprocess.letterbox_geometry(h0, w0, H, W) == want


@pytest.mark.parametrize("h0,w0", [(720, 1280), (1080, 1920), (240, 320), (479, 641), (725, 1280), (384, 640), (1280, 720), (17, 33)])
@pytest.mark.parametrize("auto", [True, False])
def test_letterbox_shape_equals_oracle(h0, w0, auto):
    if _lib_or_none() is None:
        pytest.skip("libuyd.so not built")
    from unina_yolo_dla_b200 import preprocess

    assert preprocess.letterbox_shape(h0, w0, auto=auto) == lb.letterbox_shape(h0, w0, auto=auto)
    assert preprocess.letterbox_shape(h0, w0, 320, 32, auto) == lb.letterbox_shape(h0, w0, 320, 32, auto)


def test_library_geometry_rejects_bad_arguments():
    import ctypes as C

    L = _lib_or_none()
    if L is None:
        pytest.skip("libuyd.so not built")
    o = [C.c_int() for _ in range(4)] + [C.c_double()]
    refs = [C.byref(v) for v in o]
    assert L.uyd_letterbox_geometry(0, 720, 640, 384, *refs) == 10001
    assert L.uyd_letterbox_geometry(1280, 720, 640, -1, *refs) == 10001
    assert L.uyd_letterbox_geometry(1280, 720, 640, 384, None, *refs[1:]) == 10001
