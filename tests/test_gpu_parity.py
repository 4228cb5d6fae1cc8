"""GPU parity tests (run on the B200 box): the CUDA path through the C ABI vs the CPU oracle."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def T():
    import uyd_testlib
    return uyd_testlib


@pytest.fixture(scope="module")
def R():
    import fp64ref
    return fp64ref


DIRECT_CASES = [
    # cin, cout, k, stride, H, W, kwargs
    (4, 4, 3, 1, 24, 40, dict(residual=True, in_total=8, in_coff=4, out_total=8, out_coff=4)),
    (8, 4, 1, 1, 16, 16, dict()),
    (8, 8, 3, 1, 20, 20, dict(residual=True, in_total=32, in_coff=8, out_total=32, out_coff=16)),
    (16, 16, 3, 1, 12, 20, dict()),
    (32, 16, 1, 1, 16, 24, dict(out_total=32, out_coff=16)),
    (16, 32, 3, 2, 32, 32, dict()),
    (64, 64, 3, 1, 16, 16, dict()),
    (96, 16, 1, 1, 16, 16, dict()),
    (32, 4, 1, 1, 16, 16, dict(relu=False, out_f32=True, out_total=68, out_coff=64)),
    (64, 64, 1, 1, 8, 8, dict(relu=False, out_f32=True, out_total=68, out_coff=0)),
]


@pytest.mark.parametrize("case", DIRECT_CASES, ids=lambda c: f"{c[0]}-{c[1]}-k{c[2]}s{c[3]}")
def test_direct_conv_matches_torch(T, R, case):
    cin, cout, k, s, H, W, kw = case
    R.assert_within(*T.run_single_conv(cin, cout, k, s, H, W, impl=T.IMPL_DIRECT, **kw), str(case))


def test_depthwise_conv_matches_torch(T, R):
    for c in (32, 64, 128):
        R.assert_within(*T.run_single_conv(c, c, 3, 1, 20, 28, impl=T.IMPL_DIRECT, depthwise=True), f"dw {c}")


TC_CASES = [
    # flat 1x1
    (64, 64, 1, 1, 16, 24, dict()),
    (32, 16, 1, 1, 20, 20, dict(out_total=32, out_coff=16)),
    (16, 32, 1, 1, 16, 16, dict()),
    (192, 32, 1, 1, 16, 16, dict()),
    (96, 16, 1, 1, 24, 24, dict(out_total=32)),
    (80, 64, 1, 1, 16, 16, dict()),
    (160, 128, 1, 1, 8, 8, dict()),
    (256, 128, 1, 1, 8, 8, dict()),
    (64, 64, 1, 1, 8, 8, dict(relu=False, out_f32=True, out_total=68)),
    (32, 4, 1, 1, 16, 16, dict(relu=False, out_f32=True, out_total=68, out_coff=64)),
    (64, 32, 1, 1, 16, 16, dict(in_total=192, in_coff=128)),
    # 3x3 stride 1 (halo) incl. partial tiles and residual
    (64, 64, 3, 1, 32, 16, dict()),
    (64, 64, 3, 1, 40, 40, dict()),
    (128, 64, 3, 1, 24, 24, dict()),
    (32, 64, 3, 1, 32, 32, dict()),
    (16, 16, 3, 1, 40, 40, dict(residual=True)),
    # 3x3 stride 2: per-tap boxes with TMA traversal stride; Cin = 32 -> one contiguous pixel-pair box per tile (PAIRS)
    (16, 32, 3, 2, 64, 64, dict()),
    (32, 64, 3, 2, 32, 48, dict()),
    (64, 128, 3, 2, 32, 32, dict()),
    (32, 32, 3, 2, 80, 80, dict(in_total=96, in_coff=32)),     # input is a channel slice (pair = 2 x 64 B at pitch 192 B)
    (32, 64, 3, 2, 160, 160, dict(out_total=128, out_coff=64)),  # more tiles than SMs, partial tiles on neither edge
    (32, 32, 3, 2, 36, 52, dict()),                              # partial tiles on both edges
    # BIG variant (weights streamed through their own TMA pipeline, two M-tiles per CTA): the model.py layers
    (128, 128, 3, 1, 40, 40, dict()),                            # halo, partial 16 x 16 regions on both edges
    (128, 128, 3, 1, 48, 80, dict(residual=True)),               # more regions than one wave of the pipeline, residual
    (256, 256, 3, 1, 24, 40, dict()),                            # N = 256: single accumulator pair
    (128, 256, 3, 2, 48, 48, dict()),                            # stride 2: strided box per tap
    (128, 128, 3, 2, 40, 72, dict(in_total=192, in_coff=64)),    # stride 2 from a channel slice
    (512, 256, 1, 1, 20, 20, dict()),                            # 1x1, 8 channel blocks, ragged last 256-pixel tile
    (256, 256, 1, 1, 40, 40, dict(out_total=512, out_coff=256)),
    (128, 192, 3, 1, 20, 20, dict()),                            # N = 192 (not a power of two)
]


@pytest.mark.parametrize("case", TC_CASES, ids=lambda c: f"{c[0]}-{c[1]}-k{c[2]}s{c[3]}-{c[4]}x{c[5]}")
def test_tensor_core_conv_matches_torch(T, R, case):
    cin, cout, k, s, H, W, kw = case
    R.assert_within(*T.run_single_conv(cin, cout, k, s, H, W, batch=3, impl=T.IMPL_TC, **kw), str(case))


def test_tensor_core_conv_many_tiles_and_partial_batch(T, R):
    # more tiles than SMs (persistent loop, both TMEM accumulators, stage wrap-around) and
    # a run with fewer images than the plan was built for
    R.assert_within(*T.run_single_conv(64, 64, 3, 1, 160, 160, batch=2, impl=T.IMPL_TC, max_batch=4), "3x3 b2/4")
    R.assert_within(*T.run_single_conv(64, 64, 1, 1, 160, 160, batch=3, impl=T.IMPL_TC, max_batch=4), "1x1 b3/4")


@pytest.mark.parametrize("stages", [0, 2, 3, 4, 5, 7])
@pytest.mark.parametrize("single", [False, True])
def test_tensor_core_conv_issuer_split_for_every_ring_size(T, R, stages, single, monkeypatch):
    """conv_tc's two MMA-issuing warps take alternate tiles only when the stage ring splits evenly between them
    (TcParams::dual); an odd ring, or one too short to halve, must fall back to one issuer.  Every ring size, with and
    without the second issuer, over enough tiles per CTA (15-31) for the ring to wrap several times -- 1x1 (one block
    per tile), 1x1 with three channel blocks per tile, 3x3 HALO with two, and the stride-2 PERTAP / PAIRS forms."""
    if stages:
        monkeypatch.setenv("UYD_TC_STAGES", str(stages))
    if single:
        monkeypatch.setenv("UYD_TC_SINGLE_ISSUER", "1")
    for cin, cout, k, s, H, W, B in ((64, 32, 1, 1, 160, 160, 12), (192, 64, 1, 1, 80, 80, 48), (128, 64, 3, 1, 80, 80, 48),
                                     (64, 64, 3, 2, 160, 160, 24), (32, 64, 3, 2, 160, 160, 24)):
        R.assert_within(*T.run_single_conv(cin, cout, k, s, H, W, batch=B, impl=T.IMPL_TC), str((cin, cout, k, s, stages, single)))


def test_sppf_pool_and_upsample_are_exact(T):
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd

    g = torch.Generator().manual_seed(1)
    x = T.bf16_round(torch.randn(2, 64, 40, 40, generator=g))
    p = uyd.Plan(0, 2)
    cat = p.buffer(40, 40, 256)
    up = p.buffer(80, 80, 96)
    p.sppf_pool(cat, 64)
    p.upsample2x(cat.sub(0, 64), up.sub(32, 64))
    p.finalize()
    p.write(cat.sub(0, 64), x)
    p.run_no_input(2)
    y1 = F.max_pool2d(x, 5, 1, 2)
    y2 = F.max_pool2d(y1, 5, 1, 2)
    y3 = F.max_pool2d(y2, 5, 1, 2)
    got = p.read(cat, 2).cpu()
    assert torch.equal(got, torch.cat((x, y1, y2, y3), 1))
    assert torch.equal(p.read(up.sub(32, 64), 2).cpu(), F.interpolate(x, scale_factor=2, mode="nearest"))


def test_dfl_decode_matches_oracle(T):
    import ctypes as C
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200 import _lib
    from oracle import yolo_graph as yg

    det = yg.Detect(4, (32, 64, 128))
    det.stride = torch.tensor([4.0, 8.0, 16.0])
    g = torch.Generator().manual_seed(2)
    B = 3
    raws = [torch.randn(B, 68, s, s, generator=g) * 2 for s in (20, 10, 5)]
    want = det.decode(raws)
    A = want.shape[2]
    y = torch.empty(B, 8, A, device="cuda")
    off = 0
    for r, st in zip(raws, (4.0, 8.0, 16.0)):
        nhwc = r.permute(0, 2, 3, 1).contiguous().cuda()
        _lib.check(_lib.lib().uyd_decode_dfl(_lib.context(0), C.c_void_p(nhwc.data_ptr()), B, r.shape[2], r.shape[3], 16, 4,
                                             st, C.c_void_p(y.data_ptr()), A, off, None))
        off += r.shape[2] * r.shape[3]
    torch.cuda.synchronize()
    got = y.cpu()
    assert float((got[:, :4] - want[:, :4]).abs().max()) < 2e-3  # pixels; fp32 exp differences only
    assert float((got[:, 4:] - want[:, 4:]).abs().max()) < 2e-6


NMS_CASES = [
    dict(B=4, nc=4, A=33600, frac=0.05, conf=0.25, iou=0.7, cluster=False),
    dict(B=3, nc=4, A=33600, frac=0.9, conf=0.25, iou=0.45, cluster=True),      # > 300 kept and heavy suppression
    dict(B=2, nc=4, A=33600, frac=1.0, conf=0.001, iou=0.7, cluster=True, max_nms=3000),  # top-max_nms truncation
    dict(B=2, nc=1, A=2100, frac=0.5, conf=0.25, iou=0.5, cluster=True),
    dict(B=2, nc=4, A=600, frac=0.0, conf=0.25, iou=0.7, cluster=False),         # empty images
]


@pytest.mark.parametrize("cfg", NMS_CASES, ids=lambda c: f"A{c['A']}-f{c['frac']}-iou{c['iou']}")
def test_nms_is_bit_exact_vs_oracle(T, cfg):
    import unina_yolo_dla_b200 as uyd
    from oracle import postproc as pp

    y = T.synth_predictions(cfg["B"], cfg["nc"], cfg["A"], seed=3, frac_conf=cfg["frac"], cluster=cfg["cluster"])
    # exact ties in score and coordinates on purpose
    y[:, :, 100:140] = y[:, :, 60:100]
    max_nms = cfg.get("max_nms", 30000)
    want, widx = pp.non_max_suppression(y, cfg["conf"], cfg["iou"], 300, max_nms, return_index=True)
    m = uyd.UninaYoloB200.from_yaml(nc=cfg["nc"])
    junk = torch.full((1 << 20,), 7.0, device="cuda")  # the outputs are torch.empty: make recycled memory non-zero
    del junk
    det, cnt, idx = m.nms(torch.from_numpy(y).cuda(), cfg["conf"], cfg["iou"], 300, max_nms, return_index=True)
    det, cnt, idx = det.cpu().numpy(), cnt.cpu().numpy(), idx.cpu().numpy()
    for b in range(cfg["B"]):
        n = len(want[b])
        assert cnt[b] == n
        np.testing.assert_array_equal(idx[b, :n], widx[b])          # kept-index sets, in order
        assert det[b, :n].tobytes() == want[b].tobytes()            # rows bit-exact
        assert not det[b, n:].any() and (idx[b, n:] == -1).all()    # every output element is defined


def _paired_models(seed=0, gain=1.0):
    """Product model with the seeded synthetic init + the oracle carrying the same state_dict."""
    import unina_yolo_dla_b200 as uyd
    from oracle import yolo_graph as yg

    m = uyd.UninaYoloB200.from_yaml().init_synthetic(seed, gain=gain)
    ref = yg.DetectionModel(yg.default_yaml_path())
    ref.load_state_dict(m.state_dict(), strict=True)
    return m.cuda(), ref.eval()


def test_full_forward_matches_oracle_bf16(T):
    """North-star tolerance: max relative error <= 1e-2 on head logits and box coordinates vs
    the fp32 CPU forward, same seeded random-init weights, same synthetic 640x640 frames."""
    from oracle import init as oi

    m, ref = _paired_models(seed=0)
    x = oi.seeded_frames(2, 640, seed=5)
    with torch.no_grad():
        y_ref, raw_ref = ref(x)
    y, raws = m(x.cuda())
    torch.cuda.synchronize()
    for a, b in zip(raws, raw_ref):
        assert a.shape == b.shape
        # north-star tolerance: max relative error on head logits <= 1e-2 (relative to the tensor's range)
        assert T.rel_err(a.cpu()[:, :64], b[:, :64]) <= 1e-2
        assert T.rel_err(a.cpu()[:, 64:], b[:, 64:]) <= 1e-2
    assert T.rel_err(y.cpu()[:, :4], y_ref[:, :4]) <= 1e-2
    assert float((y.cpu()[:, 4:] - y_ref[:, 4:]).abs().max()) <= 1e-2


def test_uint8_frames_equal_float_frames_divided_by_255(T):
    """The stem's fused pre-process (x / 255, reference predictor semantics) is exact."""
    m, _ = _paired_models(seed=2)
    g = torch.Generator().manual_seed(4)
    u8 = (torch.rand(2, 3, 320, 320, generator=g) * 255).to(torch.uint8)
    y8 = m(u8.cuda(), raw_heads=False)
    yf = m((u8.float() / 255).cuda(), raw_heads=False)
    torch.cuda.synchronize()
    assert torch.equal(y8, yf)


def test_predict_returns_reference_rows(T):
    from oracle import postproc as pp

    m, ref = _paired_models(seed=0)
    from oracle import init as oi
    x = oi.seeded_frames(2, 640, seed=5).cuda()
    m.calibrate_cls_bias(x, 800, 0.25)
    y = m(x, raw_heads=False)
    res = m.predict(x, conf=0.25, iou=0.7)
    want = pp.non_max_suppression(y.cpu().numpy(), 0.25, 0.7, 300)
    assert len(res) == 2
    for r, w in zip(res, want):
        assert r.shape[1] == 6 and r.cpu().numpy().tobytes() == w.tobytes()
        assert 0 < len(w) <= 300


@pytest.mark.parametrize("c,H,W", [(8, 64, 80), (16, 40, 80), (32, 40, 40), (16, 80, 80), (8, 160, 160)])
def test_fused_c3k_matches_torch(T, R, c, H, W):
    """Fused C3k block vs the seven torch convs with bf16 rounding at the same points."""
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd

    g = torch.Generator().manual_seed(c + H)
    B, h = 3, c // 2
    shapes = [(h, c, 1), (h, c, 1), (h, h, 3), (h, h, 3), (h, h, 3), (h, h, 3), (c, c, 1)]
    ws = [torch.randn(co, ci, k, k, generator=g) / (ci * k * k) ** 0.5 for co, ci, k in shapes]
    bs = [torch.randn(co, generator=g) * 0.1 for co, _, _ in shapes]
    x = torch.randn(B, c, H, W, generator=g)
    p = uyd.Plan(0, B)
    src = p.buffer(H, W, 3 * c)          # input and output live in channel slices of wider buffers
    dst = p.buffer(H, W, 2 * c)
    s_in, s_out = src.sub(c, c), dst.sub(c, c)
    p.c3k(s_in, s_out, [w.numpy() for w in ws], [b.numpy() for b in bs])
    p.finalize()
    got, = T.run_canaried(p, [(s_in, x)], [s_out], B)    # nothing written outside the slice
    r = T.bf16_round
    cb = lambda t, i: r(F.conv2d(t, r(ws[i]), bs[i], padding=ws[i].shape[2] // 2).relu())
    xin = r(x)
    a_, b_ = cb(xin, 0), cb(xin, 1)
    u = r(a_ + F.conv2d(cb(a_, 2), r(ws[3]), bs[3], padding=1).relu())
    v = r(u + F.conv2d(cb(u, 4), r(ws[5]), bs[5], padding=1).relu())
    want = cb(torch.cat((v, b_), 1), 6)
    assert T.rel_err(got, want) < 1e-2
    R.assert_within(got, *R.c3k(xin, [r(w) for w in ws], bs), f"c3k {c} {H}x{W}")


@pytest.mark.parametrize("c,H,W,B", [(16, 80, 80, 3), (16, 40, 80, 5), (32, 40, 40, 4), (16, 20, 40, 2), (32, 20, 80, 3), (16, 80, 80, 40), (32, 40, 40, 70)])
def test_tcgen05_c3k_matches_torch_and_the_mma_sync_kernel(T, R, c, H, W, B, monkeypatch):
    """Third-generation C3k block (csrc/c3k_tc.cu: tcgen05, no-swizzle two-tap descriptors over a flat frame, six stage
    pipelines side by side): same seven convs as the torch reference with bf16 rounding at the same points; ragged strips (H not a
    multiple of the strip height), widths that are not a multiple of anything, several CTAs per SM-wave."""
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd

    g = torch.Generator().manual_seed(c + H + W)
    h = c // 2
    shapes = [(h, c, 1), (h, c, 1), (h, h, 3), (h, h, 3), (h, h, 3), (h, h, 3), (c, c, 1)]
    ws = [torch.randn(co, ci, k, k, generator=g) / (ci * k * k) ** 0.5 for co, ci, k in shapes]
    bs = [torch.randn(co, generator=g) * 0.1 for co, _, _ in shapes]
    x = torch.randn(B, c, H, W, generator=g)
    outs = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("UYD_C3K_TC", mode)
        p = uyd.Plan(0, B)
        src = p.buffer(H, W, 3 * c)
        dst = p.buffer(H, W, 2 * c)
        s_in, s_out = src.sub(c, c), dst.sub(c, c)
        if not p.c3k_supported(s_in, s_out):
            pytest.skip("shape outside the mma.sync kernel's rule; the tcgen05 kernel is checked against torch below")
        p.c3k(s_in, s_out, [w.numpy() for w in ws], [b.numpy() for b in bs])
        p.finalize()
        outs[mode], = T.run_canaried(p, [(s_in, x)], [s_out], B)
    r = T.bf16_round
    cb = lambda t, i: r(F.conv2d(t, r(ws[i]), bs[i], padding=ws[i].shape[2] // 2).relu())
    xin = r(x)
    a_, b_ = cb(xin, 0), cb(xin, 1)
    u = r(a_ + F.conv2d(cb(a_, 2), r(ws[3]), bs[3], padding=1).relu())
    v = r(u + F.conv2d(cb(u, 4), r(ws[5]), bs[5], padding=1).relu())
    want = cb(torch.cat((v, b_), 1), 6)
    assert T.rel_err(outs["1"], want) < 1e-2
    assert T.rel_err(outs["1"], outs["0"]) < 1e-2
    ref, slack = R.c3k(xin, [r(w) for w in ws], bs)
    for mode, got in outs.items():
        R.assert_within(got, ref, slack, f"c3k UYD_C3K_TC={mode} {c} {H}x{W} b{B}")


def test_dense_scene_1280_nms_stress_is_bit_exact(T):
    """BASELINE config 5: 1280x1280 (134 400 anchors), ~100k candidates per image: exercises the
    top-30000 truncation and the early exit at 300 kept boxes."""
    import unina_yolo_dla_b200 as uyd
    from oracle import postproc as pp

    A = 102400 + 25600 + 6400
    y = T.synth_predictions(3, 4, A, seed=9, frac_conf=0.75, img=1280.0, cluster=True)
    want, widx = pp.non_max_suppression(y, 0.25, 0.7, 300, 30000, return_index=True)
    m = uyd.UninaYoloB200.from_yaml()
    det, cnt, idx = m.nms(torch.from_numpy(y).cuda(), 0.25, 0.7, 300, 30000, return_index=True)
    det, cnt, idx = det.cpu().numpy(), cnt.cpu().numpy(), idx.cpu().numpy()
    assert (y[:, 4:].max(1) > 0.25).sum(1).min() > 90000
    for b in range(3):
        n = len(want[b])
        assert cnt[b] == n
        np.testing.assert_array_equal(idx[b, :n], widx[b])
        assert det[b, :n].tobytes() == want[b].tobytes()


def test_full_forward_1280_matches_oracle(T):
    from oracle import init as oi

    m, ref = _paired_models(seed=1)
    x = oi.seeded_frames(1, 1280, seed=6)
    with torch.no_grad():
        y_ref, raw_ref = ref(x)
    y, raws = m(x.cuda())
    torch.cuda.synchronize()
    assert y.shape == (1, 8, 134400)
    for a, b in zip(raws, raw_ref):
        assert T.rel_err(a.cpu()[:, :64], b[:, :64]) <= 1e-2 and T.rel_err(a.cpu()[:, 64:], b[:, 64:]) <= 1e-2
    assert T.rel_err(y.cpu()[:, :4], y_ref[:, :4]) <= 1e-2


@pytest.mark.parametrize("cin,H,W", [(32, 40, 80), (64, 16, 40), (32, 160, 160)])
def test_fused_cls_branch_matches_torch(T, R, cin, H, W):
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200._lib import UYD_F32

    g = torch.Generator().manual_seed(cin + W)
    B, mid, nc = 2, 32, 4
    ws = [torch.randn(cin, 1, 3, 3, generator=g) / 3, torch.randn(mid, cin, 1, 1, generator=g) / cin ** 0.5,
          torch.randn(mid, 1, 3, 3, generator=g) / 3, torch.randn(mid, mid, 1, 1, generator=g) / mid ** 0.5,
          torch.randn(nc, mid, 1, 1, generator=g) / mid ** 0.5]
    bs = [torch.randn(w.shape[0], generator=g) * 0.1 for w in ws]
    x = torch.randn(B, cin, H, W, generator=g)
    p = uyd.Plan(0, B)
    src = p.buffer(H, W, cin)
    head = p.buffer(H, W, 68, UYD_F32)
    dst = head.sub(64, nc)
    p.cls_branch(src, dst, mid, [w.numpy() for w in ws], [b.numpy() for b in bs])
    p.finalize()
    got, = T.run_canaried(p, [(src, x)], [dst], B)
    r = T.bf16_round
    R.assert_within(got, *R.cls_branch(r(x), [r(w) for w in ws], bs), f"cls {cin} {H}x{W}")


def test_graph_replay_equals_direct_launch(T):
    """Small batches replay a captured CUDA graph of the whole step: same bytes as the direct path."""
    from oracle import init as oi

    m, _ = _paired_models(seed=0)
    x = oi.seeded_frames(2, 320, seed=8).cuda()
    m.calibrate_cls_bias(x, 400, 0.25)
    d0, c0 = m.predict_batched(x, graph=False)
    for _ in range(3):                       # capture, then two replays with fresh input copies
        d1, c1 = m.predict_batched(x, graph=True)
    torch.cuda.synchronize()
    assert int(c0.sum()) > 0 and torch.equal(c0, c1) and torch.equal(d0, d1)
    x2 = oi.seeded_frames(2, 320, seed=9).cuda()
    d2, c2 = m.predict_batched(x2, graph=True)
    d3, c3 = m.predict_batched(x2, graph=False)
    assert torch.equal(c2, c3) and torch.equal(d2, d3) and not torch.equal(d2, d0)


def test_predict_stream_equals_predict_batched(T):
    """The double-buffered streaming API returns, in order, what predict_batched returns per batch
    (incl. a ragged last batch), as pinned host tensors."""
    m, _ = _paired_models(seed=0)
    g = torch.Generator().manual_seed(12)
    batches = [(torch.rand(n, 3, 320, 320, generator=g) * 255).to(torch.uint8).pin_memory() for n in (12, 12, 12, 5)]
    m.calibrate_cls_bias(batches[0].cuda(), 400, 0.25)
    want = [tuple(t.cpu() for t in m.predict_batched(b.cuda())) for b in batches]
    got = [(d.clone(), c.clone()) for d, c in m.predict_stream(iter(batches))]
    assert len(got) == len(want)
    for (d, c), (wd, wc) in zip(got, want):
        assert int(wc.sum()) > 0 and torch.equal(c, wc) and torch.equal(d, wd)
    dev = [(d.cpu(), c.cpu()) for d, c in m.predict_stream(iter(batches[:1]), to_host=False)]
    assert torch.equal(dev[0][0], want[0][0]) and torch.equal(dev[0][1], want[0][1])
    assert list(m.predict_stream(iter([]))) == []
    # a consumer may hold result k while it handles k + 1 and k + 2 (tracking, frame differencing): no clone here
    six = [batches[i % 3] for i in range(6)]
    held = []
    for k, (d, c) in enumerate(m.predict_stream(iter(six))):
        held.append((d, c))
        for back in (1, 2):
            if k - back >= 0:
                hd, hc = held[k - back]
                wd, wc = want[(k - back) % 3]
                assert torch.equal(hc, wc) and torch.equal(hd, wd), f"result {k - back} was overwritten by step {k}"
    # device-resident batches are used in place (no staging copy), results come back on the caller's stream although the
    # NMS of step i runs on the post-processing stream under the forward of step i + 1
    res = [b.cuda() for b in batches]
    got_dev = [(d.cpu(), c.cpu()) for d, c in m.predict_stream(iter(res), to_host=False)]
    assert len(got_dev) == len(want)
    for (d, c), (wd, wc) in zip(got_dev, want):
        assert torch.equal(c, wc) and torch.equal(d, wd)
    got_mixed = [(d.clone(), c.clone()) for d, c in m.predict_stream(iter([res[0], res[1]]), to_host=True)]
    assert torch.equal(got_mixed[1][0], want[1][0]) and torch.equal(got_mixed[1][1], want[1][1])


CHAIN_CASES = [
    # cin, n1, n2, dw1, final, H, W
    (64, 64, 64, False, "store_f32", 32, 24),
    (64, 64, 64, False, "dfl", 40, 40),
    (64, 64, 64, False, "dfl", 160, 160),     # more tiles than SMs: persistent loop, both epilogue groups, stage wrap
    (32, 32, 32, True, "store_bf16", 40, 40),
    (64, 64, 32, True, "store_bf16", 24, 40),
    (32, 32, 32, True, "pw3", 40, 40),
    (32, 32, 32, True, "pw3", 160, 160),
    (32, 64, 64, False, "store_bf16", 20, 20),
    (64, 32, 32, False, "store_bf16", 20, 20),
]


@pytest.mark.parametrize("case", CHAIN_CASES, ids=lambda c: f"{c[0]}-{c[1]}-{c[2]}-{'dw' if c[3] else 'dense'}-{c[4]}-{c[5]}x{c[6]}")
def test_chained_head_kernel_matches_torch(T, R, case):
    """3x3 conv -> 1x1 conv -> final stage in one tcgen05 launch vs torch with bf16 rounding at the same points;
    raw outputs and decoded outputs (DFL boxes, sigmoid scores) of the same launch configuration."""
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200._lib import CHAIN_DFL, CHAIN_PW3, CHAIN_STORE, UYD_BF16, UYD_F32

    cin, n1, n2, dw1, final, H, W = case
    g = torch.Generator().manual_seed(cin + n1 + H)
    B, nc = 2, 4
    r = T.bf16_round
    x = torch.randn(B, cin, H, W, generator=g)
    w1 = torch.randn(n1, 1 if dw1 else cin, 3, 3, generator=g) / (9 * (1 if dw1 else cin)) ** 0.5
    w2 = torch.randn(n2, n1, generator=g) / n1 ** 0.5
    w3 = torch.randn(nc, n2, generator=g) / n2 ** 0.5
    b1, b2, b3 = (torch.randn(n, generator=g) * 0.1 for n in (n1, n2, nc))
    if final == "dfl":
        w2, b2 = w2 * 3, b2 + 1.0

    def run(decoded):
        p = uyd.Plan(0, B)
        src = p.buffer(H, W, cin + 8).sub(8, cin)          # the input lives in a channel slice
        A, a_off = H * W + 7, 3
        geo = dict(a_total=A, a_off=a_off, no=4 + nc, stride=8.0)
        out = None
        if final == "store_f32":
            out = p.buffer(H, W, 68, UYD_F32).sub(0, n2)
            p.chain(src, w1.numpy(), b1.numpy(), w2.numpy(), b2.numpy(), dw1=dw1, final=CHAIN_STORE, out=out)
        elif final == "store_bf16":
            out = p.buffer(H, W, n2 + 16).sub(16, n2)
            p.chain(src, w1.numpy(), b1.numpy(), w2.numpy(), b2.numpy(), dw1=dw1, relu2=True, final=CHAIN_STORE, out=out)
        elif final == "dfl":
            out = None if decoded else p.buffer(H, W, 68, UYD_F32).sub(0, 64)
            p.chain(src, w1.numpy(), b1.numpy(), w2.numpy(), b2.numpy(), dw1=dw1, final=CHAIN_DFL, out=out, y_ch0=0, **geo)
        else:
            out = None if decoded else p.buffer(H, W, 68, UYD_F32).sub(64, nc)
            p.chain(src, w1.numpy(), b1.numpy(), w2.numpy(), b2.numpy(), dw1=dw1, relu2=True, final=CHAIN_PW3, w3=w3.numpy(),
                    b3=b3.numpy(), out=out, y_ch0=4, **geo)
        p.finalize()
        y = torch.full((B, 4 + nc, A), -7.0, device="cuda")
        got = T.run_canaried(p, [(src, x)], [out] if out is not None else [], B,
                             run=lambda: p.run_no_input(B, y) if decoded else p.run_no_input(B))
        return (got[0] if out is not None else None), y.cpu(), a_off

    what = f"chain {case}"
    if final == "store_f32":
        got, _, _ = run(False)
        R.assert_within(got, *R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1), what)
    elif final == "store_bf16":
        got, _, _ = run(False)
        R.assert_within(got, *R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1, relu2=True, bf16_2=True), what)
    elif final == "dfl":
        raw, _, _ = run(False)
        R.assert_within(raw, *R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1), what)
        _, y, a_off = run(True)
        d = (raw.view(B, 4, 16, H * W).softmax(2) * torch.arange(16.0).view(1, 1, 16, 1)).sum(2)
        ax = (torch.arange(H * W) % W).float() + 0.5
        ay = (torch.arange(H * W) // W).float() + 0.5
        x1, y1, x2, y2 = ax - d[:, 0], ay - d[:, 1], ax + d[:, 2], ay + d[:, 3]
        want = torch.stack(((x1 + x2) / 2, (y1 + y2) / 2, x2 - x1, y2 - y1), 1) * 8.0
        assert float((y[:, :4, a_off:a_off + H * W] - want).abs().max()) < 2e-3      # same logits: only exp differs
        assert float((y[:, 4:] + 7.0).abs().max()) == 0.0 and float((y[:, :, :a_off] + 7.0).abs().max()) == 0.0
        assert float((y[:, :, a_off + H * W:] + 7.0).abs().max()) == 0.0            # nothing outside its anchors / channels
    else:
        raw, _, _ = run(False)
        R.assert_within(raw, *R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1, relu2=True, w3=r(w3), b3=b3), what)
        _, y, a_off = run(True)
        assert float((y[:, 4:, a_off:a_off + H * W] - raw.sigmoid().flatten(2)).abs().max()) < 1e-5
        assert float((y[:, :4] + 7.0).abs().max()) == 0.0


def test_fused_decode_plan_equals_raw_head_plan(T):
    """forward(raw_heads=False) runs the plan whose head kernels decode in their epilogue; it must
    reproduce the decode of the raw-head plan (same logits, same arithmetic)."""
    from oracle import init as oi

    m, ref = _paired_models(seed=0)
    x = oi.seeded_frames(2, 640, seed=5)
    y_raw, _ = m(x.cuda())
    y_fused = m(x.cuda(), raw_heads=False)
    torch.cuda.synchronize()
    assert m.plan_for(x.cuda(), fused=True).fused
    assert float((y_raw[:, :4] - y_fused[:, :4]).abs().max()) < 2e-3
    assert float((y_raw[:, 4:] - y_fused[:, 4:]).abs().max()) < 1e-5
    with torch.no_grad():
        y_ref, _ = ref(x)
    assert T.rel_err(y_fused.cpu()[:, :4], y_ref[:, :4]) <= 1e-2
    assert float((y_fused.cpu()[:, 4:] - y_ref[:, 4:]).abs().max()) <= 1e-2


@pytest.mark.parametrize("H,W,u8,pw", [(64, 96, False, False), (160, 128, True, False), (640, 640, False, False),
                                        (64, 96, True, True), (100, 136, False, True), (640, 640, True, True)])
def test_fused_stem_matches_torch(T, R, H, W, u8, pw, B=2):
    """Conv(3,16,3,2) -> Conv(16,32,3,2) (-> 1x1 Conv(32,16), model.2.cv1) in one launch: the frame is rounded to
    tf32 (2^-11), the 16- and 32-channel intermediates are rounded to bf16 exactly where the unfused plan rounds them."""
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd

    g = torch.Generator().manual_seed(H + W)
    r = T.bf16_round
    w0, w1 = torch.randn(16, 3, 3, 3, generator=g) / 27 ** 0.5, torch.randn(32, 16, 3, 3, generator=g) / 144 ** 0.5
    w2 = torch.randn(16, 32, 1, 1, generator=g) / 32 ** 0.5
    b0, b1, b2 = (torch.randn(n, generator=g) * 0.1 for n in (16, 32, 16))
    if u8:
        xin = (torch.rand(B, 3, H, W, generator=g) * 255).to(torch.uint8)
        xf = xin.float() / 255
    else:
        xin = xf = torch.rand(B, 3, H, W, generator=g)
    p = uyd.Plan(0, B)
    if pw:
        dst = p.buffer(H // 4, W // 4, 36).sub(4, 16)
        p.stem2(dst, w0.numpy(), b0.numpy(), w1.numpy(), b1.numpy(), w2.numpy(), b2.numpy())
    else:
        dst = p.buffer(H // 4, W // 4, 56).sub(16, 32)
        p.stem2(dst, w0.numpy(), b0.numpy(), w1.numpy(), b1.numpy())
    p.finalize()
    xc = xin.cuda()
    got, = T.run_canaried(p, [], [dst], B, run=lambda: p.run(xc))   # nothing outside the slice
    ref, slack = R.stem2(xf, r(w0), b0, r(w1), b1, *((r(w2), b2) if pw else ()))
    R.assert_within(got, ref, slack, f"stem2 {H}x{W} u8={u8} pw={pw} b{B}")
    # the tf32 frame (2^-11) flips many layer-0 roundings, which the carried bound must allow for: keep the
    # whole-tensor check beside it
    t = r(F.conv2d(xf, r(w0), b0, stride=2, padding=1).relu())
    want = r(F.conv2d(t, r(w1), b1, stride=2, padding=1).relu())
    if pw:
        want = r(F.conv2d(want, r(w2), b2).relu())
    assert T.rel_err(got, want) < 6e-3


@pytest.mark.parametrize("u8,pw", [(False, True), (True, False)])
def test_fused_stem_persistent_ctas(T, R, u8, pw):
    """Enough tiles (8 x 1600 > 8 per SM) for the persistent variant: CTAs walk the tiles with the layer-1 weight
    fragments in registers; a tile's shared-memory planes are recycled by the next one."""
    test_fused_stem_matches_torch(T, R, 640, 640, u8, pw, B=8)


@pytest.mark.parametrize("H,W,u8,B", [(64, 96, False, 2), (70, 94, False, 1), (70, 94, True, 2), (256, 256, True, 3),
                                       (640, 640, False, 8), (34, 258, False, 2), (36, 260, True, 2)])
def test_model_py_stem_3_to_32_on_mma_sync_matches_torch(T, R, H, W, u8, B):
    """model.py:173 backbone.stem, Conv(3, 32, 3, 2) (conv_stem_mma_kernel): the frame enters as hi + lo bf16 planes
    (2^-17 relative), weights are bf16, fp32 accumulation, one rounding to bf16.  Odd extents take the scalar staging
    path, extents that are not multiples of the 8 x 64 tile the partial-tile stores, 8 x 640 x 640 the persistent
    loop with the register prefetch (more tiles than resident CTAs)."""
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200.plan import NETWORK_INPUT

    g = torch.Generator().manual_seed(H * 7 + W)
    r = T.bf16_round
    w, b = torch.randn(32, 3, 3, 3, generator=g) / 27 ** 0.5, torch.randn(32, generator=g) * 0.1
    if u8:
        xin = (torch.rand(B, 3, H, W, generator=g) * 255).to(torch.uint8)
        xf = xin.float() / 255
    else:
        xin = xf = torch.rand(B, 3, H, W, generator=g)
    oh, ow = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
    p = uyd.Plan(0, B)
    dst = p.buffer(oh, ow, 48).sub(8, 32)
    p.conv(NETWORK_INPUT, dst, w.numpy(), b.numpy(), 3, 2, relu=True)
    p.finalize()
    xc = xin.cuda()
    got, = T.run_canaried(p, [], [dst], B, run=lambda: p.run(xc))    # nothing outside the slice
    want = F.conv2d(xf, r(w), b, stride=2, padding=1).relu()
    # the bf16 rounding of the output is the only error source that matters: compare before rounding the reference too
    assert float((got - want).abs().max()) <= 2.0 ** -8 * float(want.abs().max()) + 1e-6
    assert T.rel_err(got, r(want)) < 4e-3
    ref, slack = R.conv(xf, r(w), b, stride=2, bf16_out=True, slack_in=R.FRAME_HILO * xf.double().abs())
    R.assert_within(got, ref, slack, f"stem mma {H}x{W} u8={u8} b{B}")


def test_plan_errors_are_reported_not_thrown(T):
    """The C ABI returns an error code + message (gpu_postprocess.h convention: cudaError_t-like int, no exceptions
    across the boundary); the Python host turns it into UydError.  Misaligned / misplaced ops are refused at build time."""
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200._lib import UydError

    z = lambda *s: np.zeros(s, np.float32)
    p = uyd.Plan(0, 1)
    dst = p.buffer(16, 16, 40).sub(2, 16)                     # 4-byte aligned slice: the folded stem needs 8
    with pytest.raises(UydError):
        p.stem2(dst, z(16, 3, 3, 3), z(16), z(32, 16, 3, 3), z(32), z(16, 32), z(16))
    p = uyd.Plan(0, 1)
    a, b = p.buffer(16, 16, 32), p.buffer(16, 16, 32)
    p.conv(a, b, z(32, 32, 1, 1), z(32), 1, 1)
    with pytest.raises(UydError):                              # only the first op may read the network input
        p.stem2(p.buffer(16, 16, 32), z(16, 3, 3, 3), z(16), z(32, 16, 3, 3), z(32))
    p.finalize()
    with pytest.raises(UydError):                              # no op may be added after finalize
        p.conv(a, b, z(32, 32, 1, 1), z(32), 1, 1)


@pytest.mark.parametrize("ca,cb,cout,h,w", [(64, 32, 16, 40, 40), (128, 64, 32, 24, 40), (64, 32, 16, 160, 160)])
def test_upsample_concat_conv_fold_matches_torch(T, R, ca, cb, cout, h, w):
    """Upsample(x2) + Concat + 1x1 Conv computed as relu(up(W_a a) + W_b b + bias): the half-resolution partial
    sums stay fp32 and are added inside the tensor-core conv's epilogue."""
    import torch.nn.functional as F
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200._lib import UYD_F32

    g = torch.Generator().manual_seed(ca + w)
    B = 2
    r = T.bf16_round
    lo, sk = torch.randn(B, ca, h // 2, w // 2, generator=g), torch.randn(B, cb, h, w, generator=g)
    wt = torch.randn(cout, ca + cb, 1, 1, generator=g) / (ca + cb) ** 0.5
    bias = torch.randn(cout, generator=g) * 0.1
    p = uyd.Plan(0, B)
    s_lo, s_sk = p.buffer(h // 2, w // 2, ca), p.buffer(h, w, cb + 16).sub(16, cb)
    part = p.buffer(h // 2, w // 2, cout, UYD_F32)
    dst = p.buffer(h, w, 2 * cout).sub(cout, cout)
    p.conv(s_lo, part, wt[:, :ca].numpy(), bias.numpy() * 0, 1, 1, relu=False)
    p.conv(s_sk, dst, wt[:, ca:].numpy(), bias.numpy(), 1, 1, relu=True, pre=part)
    p.finalize()
    got_part, got = T.run_canaried(p, [(s_lo, lo), (s_sk, sk)], [part, dst], B)
    pref, pslack = R.conv(r(lo), r(wt[:, :ca]), bias * 0, relu=False)
    R.assert_within(got_part, pref, pslack, f"fold partial sums {ca} {h}x{w}")
    ref, slack = R.conv(r(sk), r(wt[:, ca:]), bias, pre=pref, pre_slack=pslack, bf16_out=True)
    R.assert_within(got, ref, slack, f"fold {ca}+{cb}->{cout} {h}x{w}")
