"""Pre-processing row (SURVEY.md 8f-1): our kernels vs the reference's own CUDA kernels (compiled from
/root/reference by oracle/build.py into oracle/_ref/, run here on the GPU) and vs the numpy restatement."""
import ctypes as C
import hashlib
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
REF_SO = Path(__file__).resolve().parents[1] / "oracle" / "_ref" / "libref_preprocess.so"
STORED = Path(__file__).resolve().parent / "golden" / "preprocess_ref.npz"   # tests/golden/make_preprocess_golden.py
STORED_WHOLE = 1 << 16   # outputs up to this many elements are stored whole, larger ones as a seeded sample


class RefNorm(C.Structure):
    _fields_ = [(n, C.c_float) for n in ("mean_r", "mean_g", "mean_b", "std_r", "std_g", "std_b")]


def load_ref():
    """The reference's own kernels, or None where they were not built (the reference sources are not part of this
    repository): the tests then compare with their output stored in tests/golden/preprocess_ref.npz."""
    if not REF_SO.exists():
        return None
    L = C.CDLL(str(REF_SO))
    L.preprocess_bgra_resize.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, RefNorm, C.c_void_p]
    L.preprocess_bgra.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, RefNorm, C.c_void_p]
    L.preprocess_nv12.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, RefNorm, C.c_void_p]
    return L


@pytest.fixture(scope="module")
def ref():
    return load_ref()


def stored_sample_index(n: int) -> torch.Tensor:
    if n <= STORED_WHOLE:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(0))[:4096].sort().values


def _against_stored(name: str, got: torch.Tensor, tol: float) -> None:
    """``got`` vs the reference output stored for case ``name``: tol = 0 compares bit for bit (sha256 of the whole
    output), otherwise the largest absolute difference over the stored elements must stay within tol."""
    g = np.load(STORED)
    flat = got.detach().flatten().cpu()
    if tol == 0:
        assert hashlib.sha256(flat.numpy().tobytes()).hexdigest() == str(g[name + "__sha256"]), name
    else:
        assert float(np.abs(flat[stored_sample_index(flat.numel())].numpy() - g[name]).max()) <= tol, name


IMAGENET = (0.485, 0.456, 0.406, 0.229, 0.224, 0.225)


def _frames(B, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (B, H, W, 4), generator=g, dtype=torch.uint8)


@pytest.mark.parametrize("H,W", [(640, 640), (96, 132), (37, 50)])
def test_bgra_matches_reference_kernel_and_numpy(ref, H, W):
    from unina_yolo_dla_b200 import preprocess as pre
    from oracle import preproc as op

    x = _frames(2, H, W, 1).cuda()
    got = pre.bgra(x, pre.norm_params())
    want = got
    if ref is not None:
        want = torch.empty_like(got)
        for b in range(2):
            assert ref.preprocess_bgra(x[b].data_ptr(), want[b].data_ptr(), W, H, W * 4, RefNorm(*IMAGENET), None) == 0
        torch.cuda.synchronize()
        assert torch.equal(got, want)                               # same expression, same compiler: bit-exact
    else:
        _against_stored(f"bgra_{H}x{W}", got, 0)
    assert np.allclose(op.bgra(x[1].cpu().numpy()), want[1].cpu().numpy(), rtol=0, atol=1e-6)
    unit = pre.bgra(x)                                              # plain x / 255 feeds the YAML model
    rgb = x[..., [2, 1, 0]].permute(0, 3, 1, 2).cpu().numpy().astype(np.float32)
    assert np.array_equal(unit.cpu().numpy(), rgb / np.float32(255))    # IEEE division, exactly the stem's uint8 path


@pytest.mark.parametrize("src,dst", [((720, 1280), (640, 640)), ((480, 640), (640, 640)), ((100, 75), (64, 96))])
def test_bgra_resize_matches_reference_kernel_and_numpy(ref, src, dst):
    from unina_yolo_dla_b200 import preprocess as pre
    from oracle import preproc as op

    (H, W), (oh, ow) = src, dst
    x = _frames(2, H, W, 2).cuda()
    got = pre.bgra(x, pre.norm_params(), size=(oh, ow))
    want = got
    if ref is not None:
        want = torch.empty_like(got)
        for b in range(2):
            assert ref.preprocess_bgra_resize(x[b].data_ptr(), want[b].data_ptr(), W, H, W * 4, ow, oh, RefNorm(*IMAGENET), None) == 0
        torch.cuda.synchronize()
        assert float((got - want).abs().max()) <= 1e-6              # normalised units; fma contraction only
    else:
        _against_stored(f"resize_{H}x{W}_{oh}x{ow}", got, 1e-6)
    assert np.allclose(op.bgra_resize(x[0].cpu().numpy(), oh, ow), want[0].cpu().numpy(), rtol=0, atol=2e-5)


@pytest.mark.parametrize("H,W", [(64, 96), (50, 38)])
def test_nv12_matches_reference_kernel_and_numpy(ref, H, W):
    from unina_yolo_dla_b200 import preprocess as pre
    from oracle import preproc as op

    g = torch.Generator().manual_seed(3)
    yp = torch.randint(0, 256, (H, W), generator=g, dtype=torch.uint8).cuda()
    uv = torch.randint(0, 256, ((H + 1) // 2, W + (W % 2)), generator=g, dtype=torch.uint8).cuda()
    got = pre.nv12(yp, uv, pre.norm_params())
    want = got
    if ref is not None:
        want = torch.empty_like(got)
        assert ref.preprocess_nv12(yp.data_ptr(), uv.data_ptr(), want.data_ptr(), W, H, yp.stride(0), uv.stride(0), RefNorm(*IMAGENET), None) == 0
        torch.cuda.synchronize()
        assert float((got - want).abs().max()) <= 1e-6
    else:
        _against_stored(f"nv12_{H}x{W}", got, 1e-6)
    assert np.allclose(op.nv12(yp.cpu().numpy(), uv.cpu().numpy()), want[0].cpu().numpy(), rtol=0, atol=2e-5)


def test_preprocessed_camera_frame_feeds_the_model():
    """BGRA camera bytes -> preprocess (x / 255) -> predict equals predict on the equivalent uint8 NCHW frames."""
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200 import preprocess as pre

    m = uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0).cuda()
    cam = _frames(2, 320, 320, 4).cuda()
    rgb = cam[..., [2, 1, 0]].permute(0, 3, 1, 2).contiguous()
    m.calibrate_cls_bias(rgb, 300, 0.25)
    d0, c0 = m.predict_batched(pre.bgra(cam), graph=False)
    d1, c1 = m.predict_batched(rgb, graph=False)
    assert int(c0.sum()) > 0 and torch.equal(c0, c1) and torch.equal(d0, d1)


def test_camera_bytes_feed_the_stem_directly(ref):
    """f-1: uyd_plan_run_camera (BGRA / BGRA + bilinear resize / NV12 read by the stem itself, no CHW fp32 tensor) vs
    the two-step path through the REFERENCE's own pre-processing kernels + the fp32 forward.  Where those kernels were
    not built, the two-step path runs our standalone kernels, after checking them against the reference output stored
    for these frames."""
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200 import preprocess as pre

    m = uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0).cuda()
    norm = pre.norm_params()                                        # ImageNet mean / std
    # (a) BGRA at the model's extent: the same IEEE expression per pixel -> bit-identical prediction
    cam = _frames(3, 320, 320, 7).cuda()
    want_in = pre.bgra(cam, norm)
    if ref is not None:
        for b in range(3):
            assert ref.preprocess_bgra(cam[b].data_ptr(), want_in[b].data_ptr(), 320, 320, 320 * 4, RefNorm(*IMAGENET), None) == 0
    else:
        _against_stored("camera_bgra", want_in, 0)
    y_ref = m(want_in, raw_heads=False)
    y_cam = m.forward_camera(cam, norm=norm)
    torch.cuda.synchronize()
    assert torch.equal(y_cam, y_ref)
    # plain x / 255 (the YAML model's own pre-process) equals the uint8 NCHW path
    rgb = cam[..., [2, 1, 0]].permute(0, 3, 1, 2).contiguous()
    assert torch.equal(m.forward_camera(cam), m(rgb, raw_heads=False))
    # (b) 1280 x 720 -> 640 x 640 bilinear inside the stem vs the reference resize kernel (fma contraction only)
    big = _frames(2, 720, 1280, 8).cuda()
    want_in = pre.bgra(big, norm, size=(640, 640))
    if ref is not None:
        for b in range(2):
            assert ref.preprocess_bgra_resize(big[b].data_ptr(), want_in[b].data_ptr(), 1280, 720, 1280 * 4, 640, 640, RefNorm(*IMAGENET), None) == 0
    else:
        _against_stored("camera_resize", want_in, 1e-6)
    y_ref = m(want_in, raw_heads=False)
    y_cam = m.forward_camera(big, size=(640, 640), norm=norm)
    torch.cuda.synchronize()
    assert float((y_cam[:, :4] - y_ref[:, :4]).abs().max() / y_ref[:, :4].abs().max()) <= 2e-3
    assert float((y_cam[:, 4:] - y_ref[:, 4:]).abs().max()) <= 2e-3
    # (c) NV12
    g = torch.Generator().manual_seed(9)
    yp = torch.randint(0, 256, (2, 320, 320), generator=g, dtype=torch.uint8).cuda()
    uvp = torch.randint(0, 256, (2, 160, 320), generator=g, dtype=torch.uint8).cuda()
    want_in = torch.cat([pre.nv12(yp[b], uvp[b], norm) for b in range(2)])
    if ref is not None:
        for b in range(2):
            assert ref.preprocess_nv12(yp[b].data_ptr(), uvp[b].data_ptr(), want_in[b].data_ptr(), 320, 320, 320, 320, RefNorm(*IMAGENET), None) == 0
    else:
        _against_stored("camera_nv12", want_in, 1e-6)
    y_ref = m(want_in, raw_heads=False)
    y_cam = m.forward_camera(yp, norm=norm, uv=uvp)
    torch.cuda.synchronize()
    assert float((y_cam[:, :4] - y_ref[:, :4]).abs().max() / y_ref[:, :4].abs().max()) <= 2e-3
    assert float((y_cam[:, 4:] - y_ref[:, 4:]).abs().max()) <= 2e-3
    det, cnt = m.predict_camera(cam, conf=0.05)
    assert det.shape == (3, 300, 6) and cnt.shape == (3,)


def test_predict_stream_nv12_equals_predict_camera():
    """The streaming API on camera frames: NV12 host batches [B, 3H/2, W] -> same rows as predict_camera per batch."""
    import unina_yolo_dla_b200 as uyd

    m = uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0).cuda()
    g = torch.Generator().manual_seed(21)
    batches = [torch.randint(0, 256, (n, 480, 320), generator=g, dtype=torch.uint8).pin_memory() for n in (6, 6, 3)]
    got = [(d.clone(), c.clone()) for d, c in m.predict_stream(iter(batches), conf=0.05, camera="nv12")]
    assert len(got) == 3
    for (d, c), b in zip(got, batches):
        bd = b.cuda()
        wd, wc = m.predict_camera(bd[:, :320], uv=bd[:, 320:], conf=0.05)
        assert torch.equal(c, wc.cpu()) and torch.equal(d, wd.cpu())
