"""INT8 inference of the model.py network (UninaCustomB200.calibrate_int8 / set_quantization / QAT checkpoints) and the
streamed-weight tcgen05 kind::i8 conv it runs its 256-output and large-weight layers on: byte-exact against the
integer references oracle/quant.py and oracle/custom_quant_graph.py."""
import numpy as np
import pytest
import torch
import torch.nn as nn

pytestmark = pytest.mark.gpu

STEM = "backbone.stem.conv"

KERNEL_CASES = [
    # cin, cout, k, stride, H, W, output ("s8" | "round" = int8 of the bf16-rounded value | "bf16" | "f32"), residual, slices, route
    (256, 256, 3, 1, 40, 24, "s8", False, False, "big-halo"),
    (128, 256, 3, 2, 40, 40, "bf16", False, False, "big-pertap"),
    (256, 256, 1, 1, 20, 20, "f32", False, False, "big-flat"),
    (512, 256, 1, 1, 40, 24, "round", False, False, "big-flat"),
    (256, 256, 3, 1, 20, 20, "bf16", True, True, "big-halo"),
    (256, 256, 1, 1, 40, 24, "s8", True, True, "big-flat"),
    (128, 256, 3, 2, 40, 24, "round", False, True, "big-pertap"),
    (256, 128, 3, 1, 20, 20, "s8", False, False, "big-halo"),    # cout <= 128, but 288 KB of weights
]


def _run_conv(qx, qw, mult, bias, k, stride, okind, out_scale, res=None, slices=False):
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200._lib import IMPL_TC, UYD_BF16, UYD_F32, UYD_S8

    B, cin, H, W = qx.shape
    cout = qw.shape[0]
    oh, ow = (H - 1) // stride + 1, (W - 1) // stride + 1
    dt = {"s8": UYD_S8, "round": UYD_S8, "f32": UYD_F32, "bf16": UYD_BF16}[okind]
    p = uyd.Plan(0, B)
    src = p.buffer(H, W, cin + 128, UYD_S8).sub(128, cin) if slices else p.buffer(H, W, cin, UYD_S8)
    dst = p.buffer(oh, ow, cout + 32, dt).sub(16, cout) if slices else p.buffer(oh, ow, cout, dt)
    rs = None
    if res is not None:
        rs = p.buffer(oh, ow, cout + 16).sub(8, cout) if slices else p.buffer(oh, ow, cout)
    p.conv_s8(src, dst, qw, mult, bias, k, stride, relu=res is not None or okind != "f32", out_scale=out_scale, impl=IMPL_TC,
              res=rs, out_round_bf16=okind == "round")
    p.finalize()
    p.write(src, torch.from_numpy(qx))
    if rs is not None:
        p.write(rs, res)
    p.run_no_input(B)
    torch.cuda.synchronize()
    return p.read(dst, B).cpu(), p.op_info(0)[0]


@pytest.mark.parametrize("case", KERNEL_CASES, ids=lambda c: f"{c[0]}-{c[1]}-k{c[2]}s{c[3]}-{c[4]}x{c[5]}-{c[6]}"
                         + ("-res" if c[7] else "") + ("-slices" if c[8] else ""))
def test_streamed_int8_conv_is_byte_exact(case):
    from oracle import quant as oq
    from oracle.quant_graph import bf16

    cin, cout, k, stride, H, W, okind, use_res, slices, route = case
    rng = np.random.default_rng(cin + cout + k + H)
    B = 3
    x = rng.normal(0, 1.0, (B, cin, H, W)).astype(np.float32)
    w = (rng.normal(0, 1.0, (cout, cin, k, k)) / np.sqrt(cin * k * k)).astype(np.float32)
    ax, aw = float(np.abs(x).max()), float(np.abs(w).max())
    qx, qw = oq.quantize(x, ax), oq.quantize(w, aw)
    mult, bias = oq.fold_multiplier(ax, aw, rng.uniform(0.8, 1.2, cout), rng.uniform(-0.1, 0.1, cout),
                                    rng.normal(0, 0.2, cout), rng.uniform(0.8, 1.2, cout), eps=1e-5)
    out_scale = float(oq.scale_of(3.0))
    relu = use_res or okind != "f32"
    acc, y, qy = oq.conv_int8(qx, qw, mult, bias, stride, relu=relu, out_scale=out_scale)
    oh, ow = acc.shape[2:]
    res = bf16(torch.from_numpy(rng.normal(0, 1, (B, cout, oh, ow)).astype(np.float32))) if use_res else None
    yt = torch.from_numpy(y) + res if use_res else torch.from_numpy(y)
    got, info = _run_conv(qx, qw, mult, bias, k, stride, okind, out_scale, res, slices)
    assert f"tc:{route}" in info, info
    if okind == "s8":
        want = np.clip(np.rint(yt.numpy() * np.float32(out_scale)), -127, 127).astype(np.int8)
        np.testing.assert_array_equal(got.numpy(), want if use_res else qy)
    elif okind == "round":
        want = np.clip(np.rint(bf16(yt).numpy() * np.float32(out_scale)), -127, 127).astype(np.int8)
        np.testing.assert_array_equal(got.numpy(), want)
    elif okind == "f32":
        assert got.numpy().tobytes() == yt.numpy().tobytes()
    else:
        assert torch.equal(got, bf16(yt))
    assert np.abs(acc).max() > 1000


def test_streamed_int8_accumulator_beyond_2_pow_24():
    """256 -> 256 3x3: |acc| reaches 2304 * 127^2; the int32 -> fp32 conversion rounds to nearest-even."""
    from oracle import quant as oq

    cin, cout, k, B, H, W = 256, 256, 3, 1, 16, 24
    rng = np.random.default_rng(5)
    qx = np.full((B, cin, H, W), 127, np.int8)
    qx[:, ::7] = 126
    qw = rng.integers(120, 128, (cout, cin, k, k)).astype(np.int8)
    qw[::3] *= -1
    mult = np.full(cout, 1.0000001, np.float32)
    bias = rng.normal(0, 1, cout).astype(np.float32)
    acc, y, _ = oq.conv_int8(qx, qw, mult, bias, 1, relu=False)
    assert np.abs(acc).max() > 2 ** 25
    got, info = _run_conv(qx, qw, mult, bias, k, 1, "f32", 0.0)
    assert "tc:big-halo" in info
    assert got.numpy().tobytes() == y.tobytes()


# ---- the network --------------------------------------------------------------------------------------------------
def _model(bc=32, seed=1):
    import unina_yolo_dla_b200 as uyd

    return uyd.UninaCustomB200(4, bc).init_synthetic(seed=seed).cuda()


def _frames(n, size, seed=11):
    from oracle import init as oi

    return oi.seeded_frames(n, size, seed=seed).cuda()


def _heads_bytes(outs):
    return [(c.cpu().numpy().tobytes(), r.cpu().numpy().tobytes()) for c, r in outs]


def _oracle_heads(m, amax, p, B):
    from oracle import custom_graph as cg
    from oracle.custom_quant_graph import CustomInt8Graph

    net = cg.CustomNet(m.num_classes, m.backbone.out_channels[0] // 2, m.backbone.lite_p2)
    net.load_state_dict({k: v.cpu() for k, v in m.state_dict().items()})
    net.eval()
    return CustomInt8Graph(net, amax).forward_from(p.read(p.feature_slices["stem"], B).cpu())


def _op_texts(p):
    return [p.op_info(i)[0] for i in range(p.launches)]


@pytest.mark.parametrize("bc,size,B", [(32, 320, 2), (32, 640, 1), (8, 320, 2)])
def test_int8_network_is_byte_exact_from_the_stem(bc, size, B):
    m = _model(bc)
    x = _frames(B, size)
    amax = m.calibrate_int8(x, float_layers=("stem",))
    convs = [n for n, mod in m.named_modules() if isinstance(mod, nn.Conv2d)]
    assert set(amax) == set(convs) - {STEM} and len(amax) == 66
    outs = m(x)
    torch.cuda.synchronize()
    p = m.plan_for(x)
    texts = _op_texts(p)
    s8 = [t for t in texts if t.startswith("conv_s8")]
    assert len(s8) == 66
    want = _oracle_heads(m, amax, p, B)
    for (c, r), (wc, wr) in zip(outs, want):
        assert c.shape == wc.shape and c.cpu().numpy().tobytes() == wc.numpy().tobytes()
        assert r.shape == wr.shape and r.cpu().numpy().tobytes() == wr.numpy().tobytes()
    if bc == 32 and size == 640:
        assert not any("direct" in t for t in s8), [t for t in s8 if "direct" in t]
        big = [t for t in s8 if "->256 " in t]
        assert len(big) == 8 and all("tc:big-" in t for t in big), big   # stage3_conv, stage3_c3k2.cv3, sppf.cv2,
        #                                                                   pan_c3k2_2.cv3, head_p4's four 3x3s
        # the default float layers (stem, head_p2): 60 quantised convs, the P3 / P4 heads unchanged
        m.set_quantization(amax)
        outs2 = m(x)
        assert sum(1 for t in _op_texts(m.plan_for(x)) if t.startswith("conv_s8")) == 60
        assert _heads_bytes(outs2)[1:] == _heads_bytes(outs)[1:]
        assert _heads_bytes(outs2)[0] != _heads_bytes(outs)[0]


@pytest.fixture(scope="module")
def int8_model():
    """bc32 at 320², max-calibrated on 8 seeded frames with the default float layers."""
    m = _model()
    amax = m.calibrate_int8(_frames(8, 320, seed=21))
    return m, amax


@pytest.mark.parametrize("method", ["max", "histogram"])
def test_calibrate_int8_names_every_quantised_conv(method):
    m = _model(seed=2)
    amax = m.calibrate_int8(_frames(4, 320, seed=3), float_layers=("stem",), method=method, batch_size=2)
    convs = [n for n, mod in m.named_modules() if isinstance(mod, nn.Conv2d)]
    assert set(amax) == {n for n in convs if m.quant.covers(n)} == set(convs) - {STEM}
    assert all(a > 0 and w > 0 for a, w in amax.values())
    if method == "histogram":
        mx = m.calibrate_int8(_frames(4, 320, seed=3), method="max", batch_size=2, enable=False)
        assert all(amax[n][0] <= mx[n][0] * 1.001 for n in amax)   # the entropy threshold never exceeds the maximum


def test_qat_checkpoint_and_set_quantization_none(int8_model):
    import unina_yolo_dla_b200 as uyd

    m, amax = int8_model
    x = _frames(2, 320, seed=5)
    q_out = _heads_bytes(m(x))
    fresh = uyd.UninaCustomB200(4, 32).cuda()
    fresh.load_state_dict(dict(m.state_dict(), **m.quant_state_dict()))
    assert fresh.quant is not None and fresh.quant.amax.keys() == amax.keys()
    assert _heads_bytes(fresh(x)) == q_out
    plain = uyd.UninaCustomB200(4, 32).cuda()
    plain.load_state_dict(m.state_dict())
    assert plain.quant is None
    f_out = _heads_bytes(plain(x))
    assert f_out != q_out
    m.set_quantization(None)
    try:
        assert _heads_bytes(m(x)) == f_out
    finally:
        m.set_quantization(amax)


def test_int8_predict_paths_agree(int8_model):
    from unina_yolo_dla_b200 import preprocess

    m, _ = int8_model
    g = torch.Generator().manual_seed(9)
    frames = torch.randint(0, 256, (12, 320, 320, 4), generator=g, dtype=torch.uint8).cuda()
    x = preprocess.bgra(frames, preprocess.norm_params())
    outs = m(x)
    best = torch.stack([c.flatten(1).max(1).values for c, _ in outs], 1).max(1).values
    conf = float(torch.sigmoid(best.min()) * 0.9)
    d12, c12 = m.predict_batched(x, conf=conf)                 # stream
    d2, c2 = m.predict_batched(x[:2], conf=conf)               # graph
    assert int(c12.min()) > 0
    assert torch.equal(c2, c12[:2]) and torch.equal(d2, d12[:2])
    for b, rows in enumerate(m.predict(x[:2], conf=conf)):
        assert torch.equal(rows, d2[b, :int(c2[b])])
    # camera bytes into the float stem, then the INT8 graph
    assert _heads_bytes(m.forward_camera(frames[:3])) == _heads_bytes(m(x[:3]))
    for graph in (True, False):
        d, c = m.predict_camera(frames[:3], conf=conf, graph=graph)
        assert torch.equal(c, c12[:3]) and torch.equal(d, d12[:3])


def test_int8_class_scores_stay_near_bf16(int8_model):
    """Sanity of the scales, not a parity claim."""
    m, amax = int8_model
    x = _frames(2, 320, seed=7)
    q = m(x)
    m.set_quantization(None)
    try:
        f = m(x)
    finally:
        m.set_quantization(amax)
    for (cq, _), (cf, _) in zip(q, f):
        assert float((torch.sigmoid(cq) - torch.sigmoid(cf)).abs().max()) < 0.25
