"""The per-element bound of tests/fp64ref.py, checked on the CPU: it accepts fp32 arithmetic in any summation order
and rejects realistic kernel faults that the old whole-tensor metric (max|err| / max|ref| < 6e-3) lets through."""
import re
import shutil
import subprocess
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

import fp64ref as R

LIB = Path(__file__).resolve().parents[1] / "unina-yolo-dla_b200" / "libuyd.so"


def bf(t):
    return t.to(torch.bfloat16).float()


def operands(cin, cout, k, H, W, B=2, seed=0, groups=1):
    """Seeded operands as the GPU tests draw them: bf16 activations and weights, fp32 biases."""
    g = torch.Generator().manual_seed(seed)
    x = bf(torch.randn(B, cin, H, W, generator=g))
    w = torch.randn(cout, cin // groups, k, k, generator=g) / (cin // groups * k * k) ** 0.5
    b = torch.randn(cout, generator=g) * 0.1
    return x, w, b


def fp32_conv(x, w, b, relu=True, bf16_out=True, **kw):
    y = F.conv2d(x, w, b, padding=w.shape[-1] // 2, **kw)
    y = y.relu() if relu else y
    return bf(y) if bf16_out else y


def violations(got, ref, slack):
    return int((~((got.double() - ref).abs() <= slack)).sum())


def rel_err(got, ref):
    return float((got.double() - ref).abs().max() / ref.abs().max())


def truncate_bf16(t):
    return (t.contiguous().view(torch.int32) & -65536).view(torch.float32)


# ---- the bound accepts correct arithmetic -----------------------------------------------------------------------

@pytest.mark.parametrize("cin,cout,k", [(256, 256, 3), (16, 16, 3), (64, 64, 1), (32, 8, 3)])
def test_bound_accepts_fp32_in_several_orders(cin, cout, k):
    x, w, b = operands(cin, cout, k, 12, 12)
    wb = bf(w)
    ref, slack = R.conv(x, wb, b, bf16_out=True)
    assert violations(fp32_conv(x, wb, b), ref, slack) == 0                       # torch's own order
    perm = torch.randperm(cin, generator=torch.Generator().manual_seed(1))
    assert violations(fp32_conv(x[:, perm], wb[:, perm], b), ref, slack) == 0     # permuted input channels
    split = sum(F.conv2d(x[:, c:c + 8], wb[:, c:c + 8], None, padding=k // 2) for c in range(0, cin, 8))
    assert violations(bf((split + b.view(1, -1, 1, 1)).relu()), ref, slack) == 0  # split-K, fp32 partials
    f32ref, f32slack = R.conv(x, wb, b, bf16_out=False)
    assert violations(fp32_conv(x, wb, b, bf16_out=False), f32ref, f32slack) == 0


def test_bound_accepts_residual_groups_stride_and_prefold():
    x, w, b = operands(32, 32, 3, 16, 16, groups=32)
    r = bf(torch.randn(2, 32, 8, 8, generator=torch.Generator().manual_seed(3)))
    ref, slack = R.conv(x, bf(w), b, stride=2, groups=32, res=r, bf16_out=True)
    got = bf(F.conv2d(x, bf(w), b, stride=2, padding=1, groups=32).relu() + r)
    assert violations(got, ref, slack) == 0
    lo, wa, _ = operands(24, 16, 1, 6, 6, seed=4)
    sk, wb_, bb = operands(8, 16, 1, 12, 12, seed=5)
    part, ps = R.conv(lo, bf(wa), torch.zeros(16), relu=False)
    ref, slack = R.conv(sk, bf(wb_), bb, pre=part, pre_slack=ps, bf16_out=True)
    p32 = F.conv2d(lo, bf(wa))
    got = bf((F.conv2d(sk, bf(wb_), bb) + R.upsample2x(p32.double()).float()).relu())
    assert violations(got, ref, slack) == 0


def test_bound_accepts_a_two_stage_chain_with_a_bf16_intermediate():
    x, w1, b1 = operands(64, 64, 3, 12, 12, seed=6)
    _, w2, b2 = operands(64, 32, 1, 1, 1, seed=7)
    w3, b3 = torch.randn(4, 32, 1, 1, generator=torch.Generator().manual_seed(8)) / 32 ** 0.5, b2[:4]
    t = fp32_conv(x, bf(w1), b1)
    z = fp32_conv(t, bf(w2), b2)
    lg = fp32_conv(z, bf(w3), b3, relu=False, bf16_out=False)
    ref, slack = R.chain(x, bf(w1), b1, bf(w2), b2, relu2=True, w3=bf(w3), b3=b3)
    assert violations(lg, ref, slack) == 0
    ref, slack = R.chain(x, bf(w1), b1, bf(w2), b2)
    assert violations(fp32_conv(t, bf(w2), b2, relu=False, bf16_out=False), ref, slack) == 0


def c3k_operands(c, seed=9):
    g = torch.Generator().manual_seed(seed)
    h = c // 2
    shapes = [(h, c, 1), (h, c, 1), (h, h, 3), (h, h, 3), (h, h, 3), (h, h, 3), (c, c, 1)]
    ws = [bf(torch.randn(co, ci, k, k, generator=g) / (ci * k * k) ** 0.5) for co, ci, k in shapes]
    bs = [torch.randn(co, generator=g) * 0.1 for co, _, _ in shapes]
    return ws, bs


def c3k_fp32(x, ws, bs):
    cb = lambda t, i: fp32_conv(t, ws[i], bs[i])
    a, b = cb(x, 0), cb(x, 1)
    u = bf(a + fp32_conv(cb(a, 2), ws[3], bs[3], bf16_out=False))
    v = bf(u + fp32_conv(cb(u, 4), ws[5], bs[5], bf16_out=False))
    return cb(torch.cat((v, b), 1), 6)


def test_bound_accepts_the_c3k_block():
    ws, bs = c3k_operands(32)
    x = bf(torch.randn(2, 32, 16, 16, generator=torch.Generator().manual_seed(10)))
    ref, slack = R.c3k(x, ws, bs)
    assert violations(c3k_fp32(x, ws, bs), ref, slack) == 0
    # seven stages of worst-case carry: the bound stays finite but loose, so the GPU tests keep the whole-tensor
    # check of the C3k block next to it
    assert 0 < R.assert_within(c3k_fp32(x, ws, bs), ref, slack, "c3k") < 1


def c3k_emulation(x, ws, bs, pack=bf, out=bf):
    """The C3k block in fp32 with bf16 weights (``pack``) and bf16 stage outputs (``out``), as the kernels run it."""
    w = [pack(t) for t in ws]
    cv = lambda t, i: F.conv2d(t, w[i], bs[i], padding=w[i].shape[-1] // 2).relu()
    a, b = out(cv(x, 0)), out(cv(x, 1))
    u = out(a + cv(out(cv(a, 2)), 3))
    v = out(u + cv(out(cv(u, 4)), 5))
    return out(cv(torch.cat((v, b), 1), 6))


def _bias_missing(i):
    def fault(x, ws, bs):
        bs = [b.clone() for b in bs]
        bs[i][3] = 0
        return c3k_emulation(x, ws, bs)
    return fault


C3K_FAULTS = {"truncated-pack": lambda x, ws, bs: c3k_emulation(x, ws, bs, pack=truncate_bf16),
              "truncated-stage-outputs": lambda x, ws, bs: c3k_emulation(x, ws, bs, out=truncate_bf16),
              "m0.cv1-bias-missing": _bias_missing(2), "m1.cv1-bias-missing": _bias_missing(4)}
C3K_GPU_SHAPES = [(32, 80, 40, 2), (32, 40, 40, 4), (16, 160, 40, 2), (16, 40, 80, 4), (8, 160, 40, 2)]


@pytest.mark.parametrize("c,H,W,B", C3K_GPU_SHAPES, ids=[f"c{c}-{H}x{W}-b{B}" for c, H, W, B in C3K_GPU_SHAPES])
def test_c3k_bound_rejects_faults_at_the_gpu_cases_shapes(c, H, W, B):
    """The C3k bound at the operands of test_gpu_kernel_bounds.py's C3k cases (fp64ref.c3k_operands, 3x3 weights at
    gain 0.4) accepts the fp32 block and rejects each fault in many elements."""
    x, ws, bs = R.c3k_operands(c, H, W, B)
    x = bf(x)
    ref, slack = R.c3k(x, [bf(w) for w in ws], bs)
    assert violations(c3k_emulation(x, ws, bs), ref, slack) == 0
    for name, fault in C3K_FAULTS.items():
        assert violations(fault(x, ws, bs), ref, slack) >= 100, name


def test_c3k_bound_at_unit_gain_misses_the_truncated_pack():
    """Why the C3k bound cases use gain 0.4: at unit gain the carried slack at c = 32 lets truncated weights pass."""
    x, ws, bs = R.c3k_operands(32, 80, 40, 2, gain3=1.0)
    x = bf(x)
    ref, slack = R.c3k(x, [bf(w) for w in ws], bs)
    assert violations(C3K_FAULTS["truncated-pack"](x, ws, bs), ref, slack) == 0


def test_assert_within_reports_the_worst_element_and_fails_on_nan():
    ref = torch.ones(1, 2, 3, 4, dtype=torch.float64)
    slack = torch.full_like(ref, 1e-3)
    got = ref.clone().float()
    assert R.assert_within(got, ref, slack) == pytest.approx(1e-3)
    got[0, 1, 2, 3] = 1.5
    with pytest.raises(AssertionError, match=r"1 of 24 .*\(0, 1, 2, 3\)"):
        R.assert_within(got, ref, slack, "x")
    got[0, 1, 2, 3] = float("nan")
    with pytest.raises(AssertionError):
        R.assert_within(got, ref, slack, "x")


# ---- the bound rejects kernel faults ----------------------------------------------------------------------------

def _faults():
    def truncated_pack(x, w, b):
        return fp32_conv(x, truncate_bf16(w), b)

    def bf16_partials(x, w, b):
        acc = torch.zeros(x.shape[0], w.shape[0], x.shape[2], x.shape[3])
        for c in range(0, x.shape[1], 64):
            acc = bf(acc + F.conv2d(x[:, c:c + 64], bf(w[:, c:c + 64]), None, padding=w.shape[-1] // 2))
        return bf((acc + b.view(1, -1, 1, 1)).relu())

    def bias_missing(x, w, b):
        b = b.clone()
        b[5] = 0
        return fp32_conv(x, bf(w), b)

    def last_channel_ignored(x, w, b):
        return fp32_conv(x[:, :-1], bf(w)[:, :-1], b)

    def right_border_term_dropped(x, w, b):
        y = F.conv2d(x, bf(w), b, padding=1)
        # channel 3, tap (ky, kx) = (1, 0) of the last output column reads input column W - 2
        y[:, :, :, -1] -= x[:, 3, :, -2].unsqueeze(1) * bf(w)[:, 3, 1, 0].view(1, -1, 1)
        return bf(y.relu())

    def neighbour_image_row(x, w, b):
        xp = F.pad(x, (1, 1, 1, 1))
        xp[:-1, :, -1, 1:-1] = x[1:, :, 0]             # the padding row below image n read from image n + 1
        return bf((F.conv2d(xp, bf(w)) + b.view(1, -1, 1, 1)).relu())

    return [("truncated-pack", (256, 256, 3), truncated_pack), ("truncated-pack", (16, 16, 3), truncated_pack),
            ("bf16-partials", (256, 256, 3), bf16_partials), ("bias-missing", (64, 64, 1), bias_missing),
            ("last-channel-ignored", (64, 64, 3), last_channel_ignored),
            ("right-border-term-dropped", (16, 16, 3), right_border_term_dropped),
            ("neighbour-image-row", (32, 32, 3), neighbour_image_row)]


FAULTS = _faults()


@pytest.mark.parametrize("name,shape,fault", FAULTS, ids=[f"{n}-{s[0]}x{s[1]}k{s[2]}" for n, s, _ in FAULTS])
def test_bound_rejects_kernel_faults(name, shape, fault):
    cin, cout, k = shape
    x, w, b = operands(cin, cout, k, 12, 12)
    ref, slack = R.conv(x, bf(w), b, bf16_out=True)
    assert violations(fault(x, w, b), ref, slack) > 0
    assert violations(fp32_conv(x, bf(w), b), ref, slack) == 0


def test_bound_rejects_a_lost_stage1_column_in_a_chain():
    x, w1, b1 = operands(32, 32, 3, 12, 12, seed=11)
    _, w2, b2 = operands(32, 32, 1, 1, 1, seed=12)
    t = fp32_conv(x, bf(w1), b1)
    t[:, :, :, 7] = 0
    got = fp32_conv(t, bf(w2), b2, relu=False, bf16_out=False)
    ref, slack = R.chain(x, bf(w1), b1, bf(w2), b2)
    assert violations(got, ref, slack) > 0


def test_whole_tensor_metric_misses_the_truncated_pack_and_bf16_partials():
    """The weakness of max|err| / max|ref| < 6e-3, kept on record: both faults pass it."""
    x, w, b = operands(256, 256, 3, 12, 12)
    ref, _ = R.conv(x, bf(w), b)
    for name, shape, fault in FAULTS[:3]:
        if shape == (256, 256, 3):
            assert rel_err(fault(x, w, b), ref) < 6e-3, name


# ---- census: every bf16 kernel instance in the library has a case -------------------------------------------------

def library_kernels():
    tools = [shutil.which(t) or f"/usr/local/cuda/bin/{t}" for t in ("cuobjdump", "cu++filt")]
    if not LIB.exists() or not all(Path(t).exists() for t in tools):
        pytest.skip("libuyd.so or the CUDA binary utilities are not available")
    out = subprocess.run([tools[0], "-symbols", str(LIB)], capture_output=True, text=True, check=True).stdout
    mangled = sorted({ln.split()[-1] for ln in out.splitlines() if "STO_ENTRY" in ln})
    names = subprocess.run([tools[1]], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    return {R.kernel_id(n) for n in names.splitlines() if n.strip()}


def test_kernel_id_reads_both_demanglers_alike():
    assert R.kernel_id("void uyd::<unnamed>::conv_direct_kernel<(int)16, (int)4, (bool)0>(uyd::ConvArgs)") == \
        R.kernel_id("void uyd::(anonymous namespace)::conv_direct_kernel<16, 4, false>(uyd::ConvArgs)") == \
        "conv_direct_kernel<16,4,0>"
    assert R.kernel_id("void uyd::stemv2::stem_v2_kernel<uyd::CamIn, (bool)1, (bool)0>(uyd::StemArgs)") == \
        "stem_v2_kernel<CamIn,1,0>"
    assert R.kernel_id("uyd::<unnamed>::sppf_pool_kernel(__nv_bfloat16 *, int, int, int, int)") == "sppf_pool_kernel"


def test_every_kernel_instance_has_a_case_or_a_stated_exclusion():
    from test_gpu_kernel_bounds import KERNELS

    have = library_kernels()
    assert not sorted(have - set(KERNELS)), "kernel instances without a bound case or an exclusion"
    assert not sorted(set(KERNELS) - have), "table entries that name no kernel in libuyd.so"
    assert all(re.fullmatch(r"(case|excluded): .+", v) for v in KERNELS.values())
