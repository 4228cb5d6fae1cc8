"""Camera bytes straight into the model.py network's stem (UninaCustomB200.forward_camera / predict_camera,
uyd_plan_run_camera on the Conv 3 -> 32 mma stem) against the two-step path it replaces: uyd_preprocess_* into an fp32
NCHW tensor, then forward / predict_batched."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

UYD_E_ARG, UYD_E_UNSUPPORTED = 10001, 10003


def _model(bc=32, seed=1):
    import unina_yolo_dla_b200 as uyd

    return uyd.UninaCustomB200(4, bc).init_synthetic(seed=seed).cuda()


def _bgra(batch, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (batch, h, w, 4), generator=g, dtype=torch.uint8).cuda()


def _nv12(batch, h, w, seed):
    g = torch.Generator().manual_seed(seed)
    y = torch.randint(0, 256, (batch, h, w), generator=g, dtype=torch.uint8).cuda()
    uv = torch.randint(0, 256, (batch, h // 2, w), generator=g, dtype=torch.uint8).cuda()
    return y, uv


def _nv12_two_step(y, uv, norm):
    from unina_yolo_dla_b200 import preprocess

    return torch.cat([preprocess.nv12(y[b], uv[b], norm) for b in range(y.shape[0])])


def _imagenet():
    from unina_yolo_dla_b200 import preprocess

    return preprocess.norm_params()


def _conf_for(outs):
    """A threshold every image clears at least once: 0.9 x the smallest per-image best class score."""
    best = torch.stack([c.flatten(1).max(1).values for c, _ in outs], 1).max(1).values
    return float(torch.sigmoid(best.min()) * 0.9)


def _assert_heads_equal(a, b):
    for (ca, ra), (cb, rb) in zip(a, b):
        assert torch.equal(ca, cb) and torch.equal(ra, rb)


@pytest.mark.parametrize("batch,size", [(3, 320), (64, 640)])
def test_bgra_at_extent_byte_equal(batch, size):
    from unina_yolo_dla_b200 import preprocess

    m = _model()
    frames = _bgra(batch, size, size, seed=batch)
    norm = _imagenet()
    x = preprocess.bgra(frames, norm)
    ref = m.forward(x)
    _assert_heads_equal(m.forward_camera(frames), ref)   # default norm: ImageNet
    conf = _conf_for(ref)
    d0, c0 = m.predict_batched(x, conf=conf, graph=False)
    assert int(c0.min()) > 0
    for graph in (False, True):
        if graph and batch > m.GRAPH_MAX_BATCH:
            continue
        d1, c1 = m.predict_camera(frames, norm=norm, conf=conf, graph=graph)
        assert torch.equal(c0, c1) and torch.equal(d0, d1)


def test_unit_norm_equals_uint8_path():
    from unina_yolo_dla_b200 import preprocess

    m = _model()
    frames = _bgra(4, 320, 320, seed=7)
    x8 = frames[..., [2, 1, 0]].permute(0, 3, 1, 2).contiguous()   # BGRA -> RGB NCHW uint8
    ref = m.forward(x8)
    conf = _conf_for(ref)
    d0, c0 = m.predict_batched(x8, conf=conf, graph=False)
    assert int(c0.min()) > 0
    _assert_heads_equal(m.forward_camera(frames, norm=preprocess.UNIT), ref)
    d1, c1 = m.predict_camera(frames, norm=preprocess.UNIT, conf=conf, graph=False)
    assert torch.equal(c0, c1) and torch.equal(d0, d1)


def test_unaligned_layout_equals_contiguous():
    """Row pitch 4 W + 4 and a frame stride that is not a multiple of 16: the 4-byte load fallback."""
    m = _model()
    B, H, W = 3, 320, 320
    frames = _bgra(B, H, W, seed=11)
    pitch = 4 * W + 4
    stride = H * pitch + 4                      # % 16 == 4
    buf = torch.zeros(B * stride + 16, dtype=torch.uint8, device="cuda")
    padded = buf.as_strided((B, H, W, 4), (stride, pitch, 4, 1), 4)
    padded.copy_(frames)
    assert padded.data_ptr() % 16 != 0 and padded.stride(0) % 16 != 0
    _assert_heads_equal(m.forward_camera(padded), m.forward_camera(frames))


def _rel_max(a, b):
    """Largest |a - b| over the range of b, for the class and the regression maps of every level."""
    cls = max(float((ca - cb).abs().max() / (cb.max() - cb.min())) for (ca, _), (cb, _) in zip(a, b))
    reg = max(float((ra - rb).abs().max() / (rb.max() - rb.min())) for (_, ra), (_, rb) in zip(a, b))
    return cls, reg


@pytest.mark.parametrize("case", ["bgra_1280x720", "bgra_480x640", "nv12_640", "nv12_320x480"])
def test_resize_and_nv12_within_tolerance(case):
    """Against the two-step path.  The loader's bilinear and BT.601 expressions may contract into FMAs differently from
    preprocess.cu's, so exactness is not promised; the bound is the model.py variant's pinned-oracle tolerance
    (regression maps 1.9e-3, class maps 1.33e-2 of range).  Measured on B200: largest difference 0 in all four cases
    (class and regression maps byte-equal)."""
    from unina_yolo_dla_b200 import preprocess

    m = _model()
    norm = _imagenet()
    if case.startswith("bgra"):
        w, h = map(int, case.split("_")[1].split("x"))
        frames = _bgra(2, h, w, seed=w + h)
        ref = m.forward(preprocess.bgra(frames, norm, size=(640, 640)))
        got = m.forward_camera(frames, size=(640, 640), norm=norm)
    else:
        dims = case.split("_")[1]
        h, w = (640, 640) if dims == "640" else tuple(map(int, dims.split("x")))
        y, uv = _nv12(2, h, w, seed=h + w)
        ref = m.forward(_nv12_two_step(y, uv, norm))
        got = m.forward_camera(y, norm=norm, uv=uv)
    cls, reg = _rel_max(got, ref)
    assert cls <= 1.33e-2 and reg <= 1.9e-3, f"{case}: class {cls:.3g}, regression {reg:.3g} of range"


def test_batch_independence():
    m = _model()
    frames = _bgra(5, 320, 320, seed=3)
    full = m.forward_camera(frames)
    for b in (0, 4):
        one = m.forward_camera(frames[b:b + 1].clone())
        for (c, r), (c1, r1) in zip(full, one):
            assert torch.equal(c[b:b + 1], c1) and torch.equal(r[b:b + 1], r1)


@pytest.mark.parametrize("batch", [1, 8])
def test_graph_replay_refreshes_frames(batch):
    m = _model()
    a, b = _bgra(batch, 320, 320, seed=20 + batch), _bgra(batch, 320, 320, seed=40 + batch)
    conf = _conf_for(m.forward_camera(a))
    for frames in (a, b, a):
        d0, c0 = m.predict_camera(frames, conf=conf, graph=False)
        d1, c1 = m.predict_camera(frames, conf=conf, graph=True)
        assert torch.equal(c0, c1) and torch.equal(d0, d1)
    y, uv = _nv12(batch, 320, 320, seed=60 + batch)
    for frames in (y, torch.flip(y, (1,))):
        d0, c0 = m.predict_camera(frames, uv=uv, conf=conf, graph=False)
        d1, c1 = m.predict_camera(frames, uv=uv, conf=conf, graph=True)
        assert torch.equal(c0, c1) and torch.equal(d0, d1)


def _run_camera_code(p, frames, uv=None, norm=None, width=None, height=None, pitch=None):
    from unina_yolo_dla_b200 import _lib

    f = _lib.CameraFrames()
    f.format = _lib.CAM_NV12 if uv is not None else _lib.CAM_BGRA
    f.width = width if width is not None else frames.shape[2]
    f.height = height if height is not None else frames.shape[1]
    f.pitch = pitch if pitch is not None else frames.stride(1)
    f.frame_stride = frames.stride(0)
    f.data = frames.data_ptr()
    if uv is not None:
        f.uv, f.uv_pitch, f.uv_frame_stride = uv.data_ptr(), uv.stride(1), uv.stride(0)
    f.norm = norm if norm is not None else _imagenet()
    code = _lib.lib().uyd_plan_run_camera(p.handle, C.byref(f), frames.shape[0], None, None)
    torch.cuda.synchronize()
    return code


def _sentinel_plan(m, B, H, W):
    """The plan for B x H x W with its stem output and head buffers set to known values."""
    p = m.plan_for(torch.empty(B, 3, H, W, device="cuda"))
    stem = p.feature_slices["stem"]
    p.write(stem, torch.full((B, stem.c, H // 2, W // 2), 3.0, device="cuda"))
    snap = [p.read(s, B) for s in [stem, *p.heads]]
    return p, [stem, *p.heads], snap


def _untouched(p, slices, snap, B):
    return all(torch.equal(p.read(s, B), v) for s, v in zip(slices, snap))


def test_rejected_without_launch():
    from unina_yolo_dla_b200 import _lib

    B, H, W = 2, 320, 320
    frames = _bgra(B, H, W, seed=5)
    for bc in (8, 16):
        m = _model(bc)
        p, sl, snap = _sentinel_plan(m, B, H, W)
        assert _run_camera_code(p, frames) == UYD_E_UNSUPPORTED
        assert _untouched(p, sl, snap, B)
        with pytest.raises(_lib.UydError):
            m.forward_camera(frames)
        with pytest.raises(_lib.UydError):
            m.predict_camera(frames, graph=False)
        with pytest.raises(_lib.UydError):
            m.predict_camera(frames[:1], graph=True)
    m = _model(32)
    p, sl, snap = _sentinel_plan(m, B, H, W)
    y, uv = _nv12(B, 256, 320, seed=6)
    assert _run_camera_code(p, y, uv=uv) == UYD_E_ARG                                  # NV12 of another extent
    assert _run_camera_code(p, frames, pitch=4 * W + 2) == UYD_E_ARG                    # BGRA pitch % 4 != 0
    zero_std = _lib.NormParams(0.485, 0.456, 0.406, 0.229, 0.0, 0.225)
    assert _run_camera_code(p, frames, norm=zero_std) == UYD_E_ARG                      # zero std
    assert _untouched(p, sl, snap, B)
