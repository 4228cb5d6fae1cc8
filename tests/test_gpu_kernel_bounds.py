"""Every bf16 kernel instance, at the smallest shape that selects it, against the fp64 reference and its per-element
bound (fp64ref.py), on canary-filled plans; each case asserts which instance it ran.  KERNELS maps every kernel
instance in libuyd.so to the case that runs it or to the reason it is tested elsewhere; the host suite checks the
table against the library's symbols and test_every_table_entry_was_launched checks it against what ran here."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

_C = "case: "
KERNELS = {
    **{f"conv_direct_kernel<{co},{iv},{ws}>": _C + "test_direct_conv_instances"
       for co in (4, 8, 16) for iv in (4, 8) for ws in (0, 1)},
    **{f"conv_dw_col_kernel<{r}>": _C + "test_depthwise_instances" for r in (8, 10, 20)},
    "conv_dw4_kernel": _C + "test_depthwise_instances",
    "conv_dw_kernel": _C + "test_depthwise_instances",
    **{f"conv_stem_tiled_kernel<{t},{c}>": _C + "test_stem_conv_instances" for t in ("float", "uint8") for c in (16, 32)},
    **{f"conv_stem_nchw_kernel<{c},{t}>": _C + "test_stem_conv_instances" for t in ("float", "uint8") for c in (4, 16)},
    "conv_stem_mma_kernel<float,1>": _C + "test_stem_conv_instances",
    "conv_stem_mma_kernel<uint8,1>": _C + "test_stem_conv_instances",
    "conv_stem_mma_kernel<float,0>": _C + "test_stem_mma_without_the_lo_plane",
    "conv_stem_mma_kernel<uint8,0>": _C + "test_stem_mma_without_the_lo_plane",
    "conv_stem_mma_kernel<CamIn,1>": "excluded: camera frames, tested in test_gpu_custom_camera.py",
    "conv_stem_mma_kernel<CamLetterboxIn,1>": "excluded: letterboxed camera frames, tested in test_gpu_letterbox.py",
    **{f"stem_v2_kernel<{t},{pw},{pe}>": _C + "test_fused_stem_instances"
       for t in ("float", "uint8") for pw in (0, 1) for pe in (0, 1)},
    **{f"stem_v2_kernel<{t},{pw},{pe}>": "excluded: camera frames, tested in test_gpu_custom_camera.py / test_gpu_letterbox.py"
       for t in ("CamIn", "CamLetterboxIn") for pw in (0, 1) for pe in (0, 1)},
    **{f"conv_tc_kernel<0,{ks}>": _C + "test_tensor_core_conv_instances" for ks in (1, 2, 4)},
    "conv_tc_big_kernel<0>": _C + "test_tensor_core_conv_instances",
    **{f"conv_chain_kernel<{a},{b},{d}>": _C + "test_chain_instances"
       for a, b, d in ((2, 2, 1), (4, 4, 1), (2, 2, 0), (2, 4, 0), (4, 2, 0), (4, 4, 0))},
    **{f"c3k_flat_kernel<{a},{b}>": _C + "test_c3k_instances" for a, b in ((4, 8), (8, 8), (16, 16))},
    "c3k_tc_kernel<1>": _C + "test_c3k_instances",
    "c3k_tc_kernel<2>": _C + "test_c3k_instances",
    "cls_branch_fused_kernel<32>": _C + "test_cls_branch_instances",
    "cls_branch_fused_kernel<64>": _C + "test_cls_branch_instances",
    "sppf_plane_kernel": _C + "test_sppf_and_upsample_instances_are_exact",
    "sppf_pool_kernel": _C + "test_sppf_and_upsample_instances_are_exact",
    "upsample2x_kernel": _C + "test_sppf_and_upsample_instances_are_exact",
    # exact elsewhere
    **{f"conv_tc_kernel<1,{ks}>": "excluded: INT8, bit-exact in test_gpu_int8.py" for ks in (1, 2, 4)},
    "conv_tc_big_kernel<1>": "excluded: INT8, bit-exact in test_gpu_int8.py / test_gpu_custom_int8.py",
    **{f"c3k_flat_q_kernel<{a},{b}>": "excluded: INT8 C3k, bit-exact in test_gpu_int8.py" for a, b in ((4, 8), (8, 8), (16, 16))},
    "conv_s8_c4_kernel<0>": "excluded: INT8, bit-exact in test_gpu_int8.py",
    "conv_s8_c4_kernel<1>": "excluded: INT8, bit-exact in test_gpu_int8.py",
    "conv_s8_direct_kernel": "excluded: INT8, bit-exact in test_gpu_int8.py",
    "conv_s8_dw_kernel": "excluded: INT8, bit-exact in test_gpu_int8.py",
    "quantize_s8_kernel": "excluded: INT8 quantiser, bit-exact in test_gpu_int8.py",
    "quantize_s8_x16_kernel": "excluded: INT8 quantiser, bit-exact in test_gpu_int8.py",
    "absmax_kernel": "excluded: INT8 calibration statistics, test_gpu_int8.py",
    "abs_histogram_kernel": "excluded: INT8 calibration statistics, test_gpu_int8.py",
    "nms_image_kernel": "excluded: NMS, bit-exact in test_gpu_parity.py",
    "compact_valid_kernel": "excluded: NMS, bit-exact in test_gpu_custom_predict.py",
    **{f"nms_records_kernel<{s}>": "excluded: NMS, bit-exact in test_gpu_custom_predict.py"
       for s in ("RecordSource<0>", "RecordSource<1>", "TlbrSource")},
    "decode_dfl_kernel<16>": "excluded: DFL decode, test_dfl_decode_matches_oracle",
    "decode_tlbr_kernel": "excluded: TLBR decode, bit-exact in test_gpu_custom_predict.py",
    "nhwc_to_nchw_kernel": _C + "test_head_export_is_exact",
    "bgra_vec4_kernel": "excluded: camera pre-process, exact in test_gpu_preprocess.py",
    "bgra_scalar_kernel": "excluded: camera pre-process, exact in test_gpu_preprocess.py",
    "bgra_resize_kernel<1>": "excluded: camera pre-process, exact in test_gpu_preprocess.py",
    "bgra_resize_kernel<4>": "excluded: camera pre-process, exact in test_gpu_preprocess.py",
    "nv12_kernel": "excluded: camera pre-process, exact in test_gpu_preprocess.py",
    "letterbox_boxes_kernel": "excluded: letterbox, exact in test_gpu_letterbox.py",
    "eval_update_kernel": "excluded: evaluation, exact in test_gpu_eval.py",
    "small_object_metric_kernel": "excluded: evaluation, exact in test_gpu_eval.py",
    "map_match_kernel": "excluded: mAP, exact in test_gpu_map.py",
    "ap_per_class_kernel": "excluded: mAP, exact in test_gpu_map.py",
}

SEEN = set()   # kernel ids every case of this module launched


@pytest.fixture(scope="module")
def T():
    import uyd_testlib
    return uyd_testlib


@pytest.fixture(scope="module")
def R():
    import fp64ref
    return fp64ref


@pytest.fixture(scope="module")
def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _conv(T, R, want, cin, cout, k, s, H, W, what, **kw):
    names = set()
    got, ref, slack = T.run_single_conv(cin, cout, k, s, H, W, kernels=names, **kw)
    SEEN.update(names)
    assert want in names, (what, sorted(names))
    R.assert_within(got, ref, slack, f"{want} {what}")
    return names


DIRECT = [
    # CO_T, IN_VEC, W_SMEM: cout % 16 / 8 / 4; cin % 8 == 0 and an 8-aligned slice; k^2 cin cout 2 B <= 96 KB
    ((16, 8, 1), (16, 16, 3, 1, 9, 9, dict(residual=True))),
    ((16, 8, 0), (128, 128, 3, 1, 9, 9, dict(out_f32=True, relu=False, out_total=136, out_coff=8))),
    ((16, 4, 1), (12, 16, 3, 2, 17, 17, dict())),
    ((16, 4, 0), (108, 128, 3, 1, 9, 9, dict(residual=True))),
    ((8, 8, 1), (16, 8, 1, 1, 9, 9, dict(out_f32=True, relu=False, out_total=12, out_coff=4))),
    ((8, 8, 0), (256, 24, 3, 1, 9, 9, dict())),
    ((8, 4, 1), (4, 8, 3, 1, 9, 11, dict(residual=True, in_total=12, in_coff=4, batch=3, max_batch=5))),
    ((8, 4, 0), (228, 24, 3, 1, 9, 9, dict(in_total=232, in_coff=4))),
    ((4, 8, 1), (8, 4, 1, 1, 9, 9, dict(out_total=12, out_coff=8))),
    ((4, 8, 0), (1376, 4, 3, 1, 9, 9, dict(out_f32=True))),
    ((4, 4, 1), (4, 4, 3, 1, 24, 40, dict(residual=True, in_total=8, in_coff=4, out_total=8, out_coff=4))),
    ((4, 4, 0), (1372, 4, 3, 2, 11, 11, dict(residual=True))),
]


@pytest.mark.parametrize("inst,case", DIRECT, ids=[f"{a}-{b}-{c}" for (a, b, c), _ in DIRECT])
def test_direct_conv_instances(T, R, inst, case):
    cin, cout, k, s, H, W, kw = case
    _conv(T, R, "conv_direct_kernel<{},{},{}>".format(*inst), cin, cout, k, s, H, W, str(case), impl=T.IMPL_DIRECT, **kw)


def test_depthwise_instances(T, R, sms, monkeypatch):
    """conv_dw_col_kernel<R> takes the tallest strip R in (20, 10) that still leaves 1024 threads per SM:
    n * ow * (c / 4) * (oh / R) >= 1024 * SMs; otherwise R = 8 (ragged at 20 rows)."""
    want = 1024 * sms
    dw = dict(impl=T.IMPL_DIRECT, depthwise=True)
    _conv(T, R, "conv_dw_col_kernel<8>", 32, 32, 3, 1, 20, 28, "20x28", **dw)
    n20 = -(-want // (20 * 32))                        # 20 x 20 x 128: one strip of 20 per column
    _conv(T, R, "conv_dw_col_kernel<20>", 128, 128, 3, 1, 20, 20, f"b{n20}", batch=n20, **dw)
    n10 = -(-want // (30 * 32 * 3))                    # 30 x 30: 30 % 20 != 0, three strips of 10
    _conv(T, R, "conv_dw_col_kernel<10>", 128, 128, 3, 1, 30, 30, f"b{n10}", batch=n10, **dw)
    _conv(T, R, "conv_dw_kernel", 64, 64, 3, 2, 20, 28, "stride 2", **dw)
    monkeypatch.setenv("UYD_DW_OLD", "1")
    _conv(T, R, "conv_dw4_kernel", 64, 64, 3, 1, 12, 20, "UYD_DW_OLD", **dw)
    _conv(T, R, "conv_dw_kernel", 16, 16, 3, 1, 12, 18, "UYD_DW_OLD, ow % 4 != 0", **dw)


def _stem_run(T, cout, stride, H, W, u8, B):
    """One stem conv reading the network input on a canary-filled plan: (got, launched ids, frame, weight, bias)."""
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200.plan import NETWORK_INPUT

    g = torch.Generator().manual_seed(H * 7 + W + cout)
    r = T.bf16_round
    w, b = torch.randn(cout, 3, 3, 3, generator=g) / 27 ** 0.5, torch.randn(cout, generator=g) * 0.1
    xin = (torch.rand(B, 3, H, W, generator=g) * 255).to(torch.uint8) if u8 else torch.rand(B, 3, H, W, generator=g)
    xf = xin.float() / 255 if u8 else xin
    assert H % stride == 0 and W % stride == 0      # the plan derives the frame extent from the output's
    oh, ow = H // stride, W // stride
    p = uyd.Plan(0, B + 1)
    dst = p.buffer(oh, ow, cout + 16).sub(8, cout)
    p.conv(NETWORK_INPUT, dst, w.numpy(), b.numpy(), 3, stride, relu=True)
    p.finalize()
    names = set()
    xc = xin.cuda()
    got, = T.run_canaried(p, [], [dst], B, run=lambda: p.run(xc), kernels=names)
    return got, names, xf, r(w), b


def _stem_check(R, want, got, names, xf, w, b, stride, frame_rel, what):
    SEEN.update(names)
    assert want in names, sorted(names)
    ref, slack = R.conv(xf, w, b, stride=stride, bf16_out=True, slack_in=frame_rel * xf.double().abs())
    R.assert_within(got, ref, slack, f"{want} {what}")


def _stem(T, R, want, cout, stride, H, W, u8, B=2, frame_rel=0.0, env=None, monkeypatch=None):
    if env:
        monkeypatch.setenv(*env)
    _stem_check(R, want, *_stem_run(T, cout, stride, H, W, u8, B), stride, frame_rel, f"{H}x{W} s{stride} u8={u8}")


@pytest.mark.parametrize("u8", [False, True], ids=["float", "uint8"])
def test_stem_conv_instances(T, R, u8, monkeypatch):
    t = "uint8" if u8 else "float"
    _stem(T, R, f"conv_stem_mma_kernel<{t},1>", 32, 2, 34, 70, u8, frame_rel=R.FRAME_HILO)
    _stem(T, R, f"conv_stem_tiled_kernel<{t},16>", 16, 2, 34, 70, u8)
    _stem(T, R, f"conv_stem_nchw_kernel<16,{t}>", 48, 2, 22, 30, u8)
    _stem(T, R, f"conv_stem_nchw_kernel<4,{t}>", 8, 1, 17, 19, u8)
    _stem(T, R, f"conv_stem_tiled_kernel<{t},32>", 32, 2, 34, 70, u8, env=("UYD_STEM_TILED", "1"), monkeypatch=monkeypatch)


NO_SPLIT_CASE = (32, 2, 34, 70, 2)   # cout, stride, H, W, B


def test_stem_mma_without_the_lo_plane(R, tmp_path):
    """conv_stem_mma_kernel<TIn, false> stages only the hi bf16 plane of the frame (2^-9 relative).  UYD_STEM_NO_SPLIT
    is read once per process, so the runs happen in a child process (this file run as a script)."""
    out = tmp_path / "no_split.pt"
    env = dict(os.environ, UYD_STEM_NO_SPLIT="1")
    subprocess.run([sys.executable, *(["-s"] if sys.flags.no_user_site else []), __file__, str(out)], env=env, check=True,
                   timeout=600)
    cout, stride, H, W, _ = NO_SPLIT_CASE
    for u8, res in torch.load(out, weights_only=False).items():
        _stem_check(R, f"conv_stem_mma_kernel<{'uint8' if u8 else 'float'},0>", *res, stride, R.FRAME_BF16,
                    f"{H}x{W} u8={u8} hi plane only")


def test_head_export_is_exact(T):
    """export_head (nhwc_to_nchw_kernel): an fp32 head buffer copied out as NCHW, bit for bit."""
    import unina_yolo_dla_b200 as uyd

    B, H, W = 3, 12, 20
    p = uyd.Plan(0, B + 1)
    src, up = p.buffer(H // 2, W // 2, 8), p.buffer(H, W, 8)
    head = p.buffer(H, W, 68, T.UYD_F32)
    p.upsample2x(src, up)
    p.set_heads([head], [8], 16, 4)
    p.finalize()
    can = T.Canary(p)
    out = torch.full((B, 68, H, W), float("nan"), device="cuda")
    names = T.launched(lambda: p.export_head(0, out, B))
    SEEN.update(names)
    assert "nhwc_to_nchw_kernel" in names, sorted(names)
    assert torch.equal(out.cpu(), can.raw(head.buf)[:B].permute(0, 3, 1, 2))


@pytest.mark.parametrize("u8", [False, True], ids=["float", "uint8"])
@pytest.mark.parametrize("pw", [False, True], ids=["no1x1", "1x1"])
@pytest.mark.parametrize("persist", [False, True], ids=["grid", "persistent"])
def test_fused_stem_instances(T, R, sms, u8, pw, persist):
    """stem_v2_kernel<TIn, PW, PERSIST>: persistent CTAs once there are 8 tiles (16 x 8 outputs) per SM."""
    import unina_yolo_dla_b200 as uyd

    H, W = (64, 128) if persist else (36, 100)
    tiles = -(-(W // 4) // 16) * -(-(H // 4) // 8)
    B = -(-8 * sms // tiles) if persist else 2
    g = torch.Generator().manual_seed(H + W + pw)
    r = T.bf16_round
    w0, w1 = torch.randn(16, 3, 3, 3, generator=g) / 27 ** 0.5, torch.randn(32, 16, 3, 3, generator=g) / 144 ** 0.5
    w2 = torch.randn(16, 32, 1, 1, generator=g) / 32 ** 0.5
    b0, b1, b2 = (torch.randn(n, generator=g) * 0.1 for n in (16, 32, 16))
    xin = (torch.rand(B, 3, H, W, generator=g) * 255).to(torch.uint8) if u8 else torch.rand(B, 3, H, W, generator=g)
    xf = xin.float() / 255 if u8 else xin
    p = uyd.Plan(0, B)
    dst = p.buffer(H // 4, W // 4, 56).sub(16, 16 if pw else 32)
    p.stem2(dst, w0.numpy(), b0.numpy(), w1.numpy(), b1.numpy(), *((w2.numpy(), b2.numpy()) if pw else ()))
    p.finalize()
    names = set()
    xc = xin.cuda()
    got, = T.run_canaried(p, [], [dst], B, run=lambda: p.run(xc), kernels=names)
    SEEN.update(names)
    want = f"stem_v2_kernel<{'uint8' if u8 else 'float'},{int(pw)},{int(persist)}>"
    assert want in names, sorted(names)
    R.assert_within(got, *R.stem2(xf, r(w0), b0, r(w1), b1, *((r(w2), b2) if pw else ())), f"{want} b{B}")


TC = [
    # kernel instance, op_info mode, case; KS = input channels per 64-byte block / 16 (min(cin, 64) / 16)
    ("conv_tc_kernel<0,1>", "flat", (16, 32, 1, 1, 20, 20, dict(in_total=48, in_coff=16, out_total=64, out_coff=32))),
    ("conv_tc_kernel<0,2>", "flat", (32, 16, 1, 1, 20, 36, dict(relu=False, out_f32=True, out_total=20, out_coff=4))),
    ("conv_tc_kernel<0,4>", "flat", (192, 32, 1, 1, 17, 23, dict(in_total=256, in_coff=64, max_batch=5))),
    ("conv_tc_kernel<0,1>", "halo", (16, 16, 3, 1, 40, 40, dict(residual=True))),
    ("conv_tc_kernel<0,2>", "halo", (32, 64, 3, 1, 33, 47, dict(out_total=96, out_coff=32))),
    ("conv_tc_kernel<0,4>", "halo", (64, 64, 3, 1, 40, 40, dict(residual=True, max_batch=5))),
    ("conv_tc_kernel<0,1>", "pertap", (16, 32, 3, 2, 64, 64, dict())),
    ("conv_tc_kernel<0,4>", "pertap", (64, 128, 3, 2, 34, 46, dict(in_total=128, in_coff=64))),
    ("conv_tc_kernel<0,2>", "pairs", (32, 32, 3, 2, 36, 52, dict(out_total=48, out_coff=16, max_batch=5))),  # dense input
    ("conv_tc_big_kernel<0>", "big-flat", (512, 256, 1, 1, 20, 20, dict(out_total=512, out_coff=256))),
    ("conv_tc_big_kernel<0>", "big-halo", (128, 128, 3, 1, 40, 56, dict(residual=True, max_batch=5))),
    ("conv_tc_big_kernel<0>", "big-pertap", (128, 128, 3, 2, 40, 72, dict(in_total=192, in_coff=64))),
]


@pytest.mark.parametrize("inst,mode,case", TC, ids=[f"{m}-{c[0]}-{c[1]}" for _, m, c in TC])
def test_tensor_core_conv_instances(T, R, inst, mode, case):
    cin, cout, k, s, H, W, kw = case
    names = _conv(T, R, inst, cin, cout, k, s, H, W, str(case), impl=T.IMPL_TC, batch=3, **kw)
    info = [n for n in names if n.startswith("op_info:")]
    assert any(f"tc:{mode} " in n or n.endswith(f"tc:{mode}") for n in info), info


CHAIN = [  # cin, n1, n2, dw1, final -> conv_chain_kernel<cin / 16, n1 / 16, dw1>
    (32, 32, 32, True, "pw3"), (64, 64, 48, True, "store_bf16"), (32, 32, 64, False, "dfl"),
    (32, 64, 16, False, "store_f32"), (64, 32, 32, False, "store_bf16"), (64, 64, 64, False, "dfl"),
]


@pytest.mark.parametrize("case", CHAIN, ids=lambda c: f"{c[0]}-{c[1]}-{c[2]}-{'dw' if c[3] else 'dense'}-{c[4]}")
def test_chain_instances(T, R, case):
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200._lib import CHAIN_DFL, CHAIN_PW3, CHAIN_STORE, UYD_F32

    cin, n1, n2, dw1, final = case
    H, W, B, nc = 24, 36, 3, 4
    g = torch.Generator().manual_seed(cin + n1 + n2)
    r = T.bf16_round
    x = torch.randn(B, cin, H, W, generator=g)
    w1 = torch.randn(n1, 1 if dw1 else cin, 3, 3, generator=g) / (9 * (1 if dw1 else cin)) ** 0.5
    w2 = torch.randn(n2, n1, generator=g) / n1 ** 0.5
    w3 = torch.randn(nc, n2, generator=g) / n2 ** 0.5
    b1, b2, b3 = (torch.randn(n, generator=g) * 0.1 for n in (n1, n2, nc))
    p = uyd.Plan(0, B + 1)
    src = p.buffer(H, W, cin + 16).sub(8, cin)
    geo = dict(a_total=H * W, a_off=0, no=4 + nc, stride=8.0)
    args = (src, w1.numpy(), b1.numpy(), w2.numpy(), b2.numpy())
    if final == "store_f32":
        out = p.buffer(H, W, n2 + 4, UYD_F32).sub(4, n2)
        p.chain(*args, dw1=dw1, final=CHAIN_STORE, out=out)
        ref = R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1)
    elif final == "store_bf16":
        out = p.buffer(H, W, n2 + 16).sub(8, n2)
        p.chain(*args, dw1=dw1, relu2=True, final=CHAIN_STORE, out=out)
        ref = R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1, relu2=True, bf16_2=True)
    elif final == "dfl":
        out = p.buffer(H, W, 68, UYD_F32).sub(0, 64)
        p.chain(*args, dw1=dw1, final=CHAIN_DFL, out=out, y_ch0=0, **geo)
        ref = R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1)
    else:
        out = p.buffer(H, W, 68, UYD_F32).sub(64, nc)
        p.chain(*args, dw1=dw1, relu2=True, final=CHAIN_PW3, w3=w3.numpy(), b3=b3.numpy(), out=out, y_ch0=4, **geo)
        ref = R.chain(r(x), r(w1), b1, r(w2), b2, dw1=dw1, relu2=True, w3=r(w3), b3=b3)
    p.finalize()
    names = set()
    got, = T.run_canaried(p, [(src, x)], [out], B, kernels=names)
    SEEN.update(names)
    want = f"conv_chain_kernel<{cin // 16},{n1 // 16},{int(dw1)}>"
    assert want in names, sorted(names)
    R.assert_within(got, *ref, f"{want} {final}")


def _c3k(T, R, c, H, W, B, env, monkeypatch):
    import unina_yolo_dla_b200 as uyd

    import torch.nn.functional as F

    for k, v in env.items():
        monkeypatch.setenv(k, v)
    x, ws, bs = R.c3k_operands(c, H, W, B)       # 3x3 weights at gain 0.4: see fp64ref.C3K_GAIN3
    p = uyd.Plan(0, B + 1)
    s_in, s_out = p.buffer(H, W, 3 * c).sub(c, c), p.buffer(H, W, 2 * c).sub(c, c)
    p.c3k(s_in, s_out, [w.numpy() for w in ws], [b.numpy() for b in bs])
    p.finalize()
    names = set()
    got, = T.run_canaried(p, [(s_in, x)], [s_out], B, kernels=names)
    SEEN.update(names)
    r = T.bf16_round
    R.assert_within(got, *R.c3k(r(x), [r(w) for w in ws], bs), f"c3k {c} {H}x{W} b{B} {env}")
    cb = lambda t, i: r(F.conv2d(t, r(ws[i]), bs[i], padding=ws[i].shape[2] // 2).relu())
    a_, b_ = cb(r(x), 0), cb(r(x), 1)
    u = r(a_ + F.conv2d(cb(a_, 2), r(ws[3]), bs[3], padding=1).relu())
    v = r(u + F.conv2d(cb(u, 4), r(ws[5]), bs[5], padding=1).relu())
    assert T.rel_err(got, cb(torch.cat((v, b_), 1), 6)) < 1e-2     # the whole-tensor check the bound replaces elsewhere
    return names


@pytest.mark.parametrize("c,th", [(c, th) for c in (8, 16, 32) for th in (32, 20, 16, 8, 4) if (c, th) != (32, 32)])
def test_c3k_instances(T, R, c, th, monkeypatch):
    """c3k_flat_kernel at every tile height c3k_launch_th can return (160 rows divide by all of them; c = 32 fits
    shared memory only up to TH = 20, so it runs at 80 rows), then the tcgen05 generation for the widths it serves."""
    want = {8: "c3k_flat_kernel<4,8>", 16: "c3k_flat_kernel<8,8>", 32: "c3k_flat_kernel<16,16>"}[c]
    H, W, B = (80 if c == 32 else 160), 40, 2
    names = _c3k(T, R, c, H, W, B, {"UYD_C3K_TC": "0", "UYD_C3K_TH": str(th)}, monkeypatch)
    assert want in names, sorted(names)
    # UYD_C3K_TH falls back silently when a height does not apply: the grid (one CTA per 40 x TH tile) shows what ran
    assert f"grid:{want}:{B * (W // 40) * (H // th)},1,1" in names, sorted(names)
    if c != 8 and th == 20:
        names = _c3k(T, R, c, 40, 80 if c == 16 else 40, 4, {"UYD_C3K_TC": "1"}, monkeypatch)
        assert f"c3k_tc_kernel<{c // 16}>" in names, sorted(names)


@pytest.mark.parametrize("cin", [32, 64])
def test_cls_branch_instances(T, R, cin):
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200._lib import UYD_F32

    g = torch.Generator().manual_seed(cin)
    B, H, W, mid, nc = 3, 16, 40, 32, 4
    ws = [torch.randn(cin, 1, 3, 3, generator=g) / 3, torch.randn(mid, cin, 1, 1, generator=g) / cin ** 0.5,
          torch.randn(mid, 1, 3, 3, generator=g) / 3, torch.randn(mid, mid, 1, 1, generator=g) / mid ** 0.5,
          torch.randn(nc, mid, 1, 1, generator=g) / mid ** 0.5]
    bs = [torch.randn(w.shape[0], generator=g) * 0.1 for w in ws]
    x = torch.randn(B, cin, H, W, generator=g)
    p = uyd.Plan(0, B + 1)
    src = p.buffer(H, W, cin + 8).sub(8, cin)
    dst = p.buffer(H, W, 68, UYD_F32).sub(64, nc)
    p.cls_branch(src, dst, mid, [w.numpy() for w in ws], [b.numpy() for b in bs])
    p.finalize()
    names = set()
    got, = T.run_canaried(p, [(src, x)], [dst], B, kernels=names)
    SEEN.update(names)
    assert f"cls_branch_fused_kernel<{cin}>" in names, sorted(names)
    r = T.bf16_round
    R.assert_within(got, *R.cls_branch(r(x), [r(w) for w in ws], bs), f"cls {cin}")


@pytest.mark.parametrize("c,H,W,want", [(64, 20, 20, "sppf_plane_kernel"), (24, 20, 20, "sppf_plane_kernel"),
                                        (64, 40, 48, "sppf_pool_kernel")], ids=["plane-gp2", "plane-gp1", "rows"])
def test_sppf_and_upsample_instances_are_exact(T, R, c, H, W, want):
    """sppf_plane_kernel pools two 8-channel groups per plane when c / 8 is even (gp = 2), one otherwise; a plane
    over 110 KB (2 * h * w * gp * 16 B) goes to the row kernel."""
    import unina_yolo_dla_b200 as uyd

    B = 3
    x = T.bf16_round(torch.randn(B, c, H, W, generator=torch.Generator().manual_seed(c + H)))
    p = uyd.Plan(0, B + 1)
    cat = p.buffer(H, W, 4 * c + 8).sub(8, 4 * c)
    up = p.buffer(2 * H, 2 * W, c + 16)
    p.sppf_pool(cat, c)
    p.upsample2x(cat.sub(0, c), up.sub(8, c))
    p.finalize()
    names = set()
    got, got_up = T.run_canaried(p, [(cat.sub(0, c), x)], [cat, up.sub(8, c)], B, kernels=names)
    SEEN.update(names)
    assert want in names and "upsample2x_kernel" in names, sorted(names)
    if want == "sppf_plane_kernel":      # one CTA per image and group of gp 8-channel planes
        gp = 2 if (c // 8) % 2 == 0 else 1
        assert f"grid:sppf_plane_kernel:{B * (c // 8) // gp},1,1" in names, sorted(names)
    assert torch.equal(got, R.max_pool_cascade(x))
    assert torch.equal(got_up, R.upsample2x(x))


def test_every_table_entry_was_launched(request):
    """Runs last in this module: every case named in KERNELS launched its instance.  Only meaningful when every
    case of the module was selected in this session."""
    selected = {it.originalname for it in request.session.items if it.module is request.module}
    if not {v[len(_C):] for v in KERNELS.values() if v.startswith(_C)} <= selected:
        pytest.skip("a subset of this module was selected")
    cases = {k for k, v in KERNELS.items() if v.startswith(_C)}
    assert not sorted(cases - SEEN), "table entries no case launched"


if __name__ == "__main__":   # child process of test_stem_mma_without_the_lo_plane
    from pathlib import Path

    _here = Path(__file__).resolve().parent
    sys.path[:0] = [str(_here), str(_here.parent)]
    import uyd_testlib

    torch.save({u8: _stem_run(uyd_testlib, *NO_SPLIT_CASE[:4], u8, NO_SPLIT_CASE[4]) for u8 in (False, True)}, sys.argv[1])
