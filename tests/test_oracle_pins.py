"""Pins the CPU oracle against real reference outputs (SURVEY.md 8c):
the reference's own model.py (live import when mounted + committed golden vectors),
its postprocess.hpp compiled from where it lies, and torchvision.ops.nms."""
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, REFERENCE
from oracle import custom_graph as cg
from oracle import init as oi
from oracle import postproc as pp
from oracle import yolo_graph as yg

sys.path.insert(0, str(GOLDEN))
import make_golden  # noqa: E402  (only its pure-python case table and GOLDEN_THREADS are used)


@pytest.mark.parametrize("bc", [8, 32])
def test_custom_graph_matches_golden_from_real_model_py(bc):
    g = np.load(GOLDEN / f"custom_bc{bc}.npz")
    saved = torch.get_num_threads()
    torch.set_num_threads(make_golden.GOLDEN_THREADS)   # the count custom_bc*.npz were computed with
    try:
        net = oi.build_custom(seed=7, base_channels=bc, calib_batch=2, size=int(g["size"]))
        assert oi.state_dict_sha256(net.state_dict()) == str(g["sha256"]), "seeded weights drifted from the fixture"
        with torch.no_grad():
            outs = net(oi.seeded_frames(1, int(g["size"]), seed=11))
    finally:
        torch.set_num_threads(saved)
    for lvl, (c, r) in zip((2, 3, 4), outs):
        np.testing.assert_array_equal(c.numpy(), g[f"p{lvl}_cls"])
        np.testing.assert_array_equal(r.numpy(), g[f"p{lvl}_reg"])


@pytest.mark.skipif(not REFERENCE.exists(), reason="/root/reference not mounted")
def test_custom_graph_matches_live_model_py():
    sys.path.insert(0, str(REFERENCE))
    import model as refmodel

    ref = oi.build_custom(seed=3, base_channels=16, calib_batch=2, size=128, cls=refmodel.UNINA_YOLO_DLA)
    mine = cg.CustomNet(4, 16)
    assert list(mine.state_dict().keys()) == list(ref.state_dict().keys())
    assert len(ref.state_dict()) == 378
    mine.load_state_dict(ref.state_dict(), strict=True)
    mine.eval()
    x = oi.seeded_frames(2, 128, seed=4)
    with torch.no_grad():
        a, b = ref(x), mine(x)
    for (ac, ar), (bc_, br) in zip(a, b):
        assert torch.equal(ac, bc_) and torch.equal(ar, br)
    # parameter count of the full-width network (SURVEY.md section 6)
    assert sum(p.numel() for p in cg.CustomNet(4, 32).parameters()) == 5_004_344


def test_yolo_graph_schema_and_census():
    m = yg.DetectionModel(yg.default_yaml_path())
    sd = m.state_dict()
    assert len(sd) == 925
    assert sum(p.numel() for p in m.parameters()) == 621_548
    assert sum(isinstance(x, torch.nn.Conv2d) for x in m.modules()) == 159  # 158 + DFL
    for k, shape in {
        "model.0.conv.weight": (16, 3, 3, 3),
        "model.2.m.1.m.0.cv2.conv.weight": (4, 4, 3, 3),
        "model.7.cv2.conv.weight": (128, 256, 1, 1),
        "model.20.cv2.0.1.conv.weight": (64, 64, 3, 3),
        "model.20.cv2.2.2.bias": (64,),
        "model.20.cv3.0.0.0.conv.weight": (32, 1, 3, 3),
        "model.20.cv3.1.1.1.bn.running_var": (32,),
        "model.20.cv3.2.2.weight": (4, 32, 1, 1),
        "model.20.dfl.conv.weight": (1, 16, 1, 1),
    }.items():
        assert tuple(sd[k].shape) == shape, k
    m.eval()
    with torch.no_grad():
        y, raw = m(torch.zeros(1, 3, 64, 64))
    assert y.shape == (1, 8, 16 * 16 + 8 * 8 + 4 * 4)
    assert [tuple(r.shape) for r in raw] == [(1, 68, 16, 16), (1, 68, 8, 8), (1, 68, 4, 4)]


def test_yolo_graph_reference_yaml_is_the_same_graph():
    import yaml

    ref = REFERENCE / "unina-yolo-dla-m.yaml"
    if not ref.exists():
        pytest.skip("/root/reference not mounted")
    assert yaml.safe_load(ref.read_text()) == yaml.safe_load(yg.default_yaml_path().read_text())


def test_nms_matches_torchvision_golden_and_live():
    import torchvision

    g = np.load(GOLDEN / "tv_nms.npz")
    for name, (b, s, thr) in make_golden.tv_cases().items():
        np.testing.assert_array_equal(b, g[f"{name}__boxes"])
        keep = pp.nms_torchvision_semantics(b, s, float(thr))
        np.testing.assert_array_equal(keep, g[f"{name}__keep"], err_msg=name)
        live = torchvision.ops.nms(torch.from_numpy(b), torch.from_numpy(s), float(thr)).numpy()
        np.testing.assert_array_equal(keep, live, err_msg=name)
    # known answers (SURVEY.md 8c): ties keep the lower index; IoU == thr is kept; the
    # fp32 IoU is compared against the *double* threshold (1/3 case suppresses).
    assert list(g["ties__keep"]) == [0, 3]
    assert list(g["iou_eq_half__keep"]) == [0, 1]
    assert list(g["iou_eq_third__keep"]) == [0]
    assert list(g["cross_class__keep"]) == [0, 2]


def test_postprocess_hpp_golden_and_live():
    g = np.load(GOLDEN / "postprocess_hpp.npz")
    cls, reg, stride = g["cls"], g["reg"], int(g["stride"])
    for thr, q, dk, kk in ((0.5, 0.0, "d0", "k0"), (0.3, 0.1, "d1", "k1")):
        d = pp.decode_tlbr(cls, reg, stride, thr, q)
        assert d.tobytes() == g[dk].tobytes()
        k = pp.greedy_nms_hpp(d, 0.45)
        assert k.tobytes() == g[kk].tobytes()
        if pp.ref_lib() is not None:  # the reference header itself, compiled
            assert pp.decode_tlbr(cls, reg, stride, thr, q, use_ref=True).tobytes() == d.tobytes()
            assert pp.greedy_nms_hpp(d, 0.45, use_ref=True).tobytes() == k.tobytes()


def test_non_max_suppression_pipeline_matches_torchvision_composition():
    """The restated Ultralytics pipeline == the same steps composed from torch + torchvision."""
    import torchvision

    rng = np.random.default_rng(0)
    B, nc, A = 2, 4, 5000
    pred = np.zeros((B, 4 + nc, A), np.float32)
    pred[:, 0:2] = rng.uniform(0, 640, (B, 2, A))
    pred[:, 2:4] = rng.uniform(4, 120, (B, 2, A))
    pred[:, 4:] = rng.uniform(0, 1, (B, nc, A)) ** 3
    outs, idx = pp.non_max_suppression(pred, 0.25, 0.7, max_det=300, max_nms=1500, return_index=True)
    for b in range(B):
        x = torch.from_numpy(pred[b].T.copy())
        xc = x[:, 4:].amax(1) > 0.25
        anchor = torch.nonzero(xc)[:, 0]
        x = x[xc]
        box = torch.cat((x[:, :2] - x[:, 2:4] / 2, x[:, :2] + x[:, 2:4] / 2), 1)
        conf, j = x[:, 4:].max(1, keepdim=True)
        x = torch.cat((box, conf, j.float()), 1)
        order = x[:, 4].argsort(descending=True, stable=True)[:1500]
        x, anchor = x[order], anchor[order]
        i = torchvision.ops.nms(x[:, :4] + x[:, 5:6] * 7680, x[:, 4], 0.7)[:300]
        np.testing.assert_array_equal(outs[b], x[i].numpy())
        np.testing.assert_array_equal(idx[b], anchor[i].numpy())
        assert len(outs[b]) == 300
    empty = pp.non_max_suppression(np.zeros((1, 8, 100), np.float32), 0.25, 0.7)
    assert empty[0].shape == (0, 6)


def test_int8_reference_is_the_fake_quant_graph():
    """oracle/quant.py: the integer statement equals conv(fake_quant(x), fake_quant(w)) -> BN -> ReLU
    (pytorch-quantization semantics as configured at qat.py:109-124) up to fp32 rounding."""
    import torch.nn.functional as F
    from oracle import quant as oq

    rng = np.random.default_rng(0)
    x = rng.normal(0, 1, (2, 16, 12, 12)).astype(np.float32)
    w = rng.normal(0, 0.1, (8, 16, 3, 3)).astype(np.float32)
    ax, aw = float(np.abs(x).max()), float(np.abs(w).max())
    qx, qw = oq.quantize(x, ax), oq.quantize(w, aw)
    assert qx.min() >= -127 and qx.max() == 127 or qx.min() == -127
    g, b, mu, var = rng.uniform(0.8, 1.2, 8), rng.uniform(-0.1, 0.1, 8), rng.normal(0, 0.2, 8), rng.uniform(0.8, 1.2, 8)
    m, bb = oq.fold_multiplier(ax, aw, g, b, mu, var, eps=1e-3)
    acc, y, qy = oq.conv_int8(qx, qw, m, bb, 1, True, out_scale=float(oq.scale_of(2.0)))
    fx = torch.from_numpy(qx.astype(np.float64) * ax / 127)
    fw = torch.from_numpy(qw.astype(np.float64) * aw / 127)
    ref = F.conv2d(fx, fw, padding=1).numpy()
    ref = (ref - mu[None, :, None, None]) * (g / np.sqrt(var + 1e-3))[None, :, None, None] + b[None, :, None, None]
    ref = np.maximum(ref, 0)
    np.testing.assert_allclose(y, ref, rtol=2e-5, atol=2e-6)
    assert np.abs(qy.astype(np.int32) - np.clip(np.rint(ref * 127 / 2.0), -127, 127)).max() <= 1
    # half-to-even rounding and the narrow range
    assert list(oq.quantize(np.array([0.5, 1.5, 2.5, -300.0, 300.0], np.float32), 127.0)) == [0, 2, 2, -127, 127]
