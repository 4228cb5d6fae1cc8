"""uyd_nms_ex (multi-label, class filter, class-agnostic NMS) and the ``classes`` / ``agnostic`` / ``multi_label``
arguments of the YAML network's entry points, byte for byte against the restated Ultralytics non_max_suppression
(tests/nms_options_ref.py, pinned to torch + torchvision by tests/test_nms_options_host.py)."""
import ctypes as C

import numpy as np
import pytest
import torch

import nms_options_ref as nref
from uyd_testlib_cpu import synth_predictions

pytestmark = pytest.mark.gpu
E_ARG = 10001

# (multi_label, classes, agnostic)
OPTIONS = [(False, None, False), (True, None, False), (True, [0, 3, 99, -1], False), (False, [1], True), (True, [], False),
           (True, None, True), (False, [0, 2], False)]


def _opt(multi_label, classes):
    from unina_yolo_dla_b200 import _lib

    o = _lib.NmsOptions(multi_label=int(multi_label))
    if classes is not None:
        o.num_filter_classes = len(classes)
        o.filter_classes = (C.c_int * max(1, len(classes)))(*classes)
    return o


def _call(y, conf, iou, max_nms, max_det, max_wh, opt, fn="uyd_nms_ex", fill=True):
    """One uyd_nms / uyd_nms_ex call on pre-filled outputs; returns (code, det, idx, cnt) on the host."""
    from unina_yolo_dla_b200 import _lib

    B, no, A = y.shape
    det = torch.full((B, max_det, 6), 7.0 if fill else 0.0, device="cuda")
    idx = torch.full((B, max_det), -7, dtype=torch.int32, device="cuda")
    cnt = torch.full((B,), -7, dtype=torch.int32, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())
    L = _lib.lib()
    if fn == "uyd_nms":
        ws = torch.empty(max(1, int(L.uyd_nms_workspace_bytes(B, A))), dtype=torch.uint8, device="cuda")
        code = L.uyd_nms(_lib.context(0), p(y), B, no - 4, A, conf, iou, max_nms, max_det, max_wh, p(ws), ws.numel(), p(det),
                         p(idx), p(cnt), None)
    else:
        code = L.uyd_nms_ex(_lib.context(0), p(y), B, no - 4, A, conf, iou, max_nms, max_det, max_wh,
                            C.byref(opt) if opt is not None else None, p(det), p(idx), p(cnt), None)
    torch.cuda.synchronize()
    return code, det.cpu().numpy(), idx.cpu().numpy(), cnt.cpu().numpy()


def _assert_equal_oracle(y_np, det, idx, cnt, want, widx):
    for b in range(y_np.shape[0]):
        k = int(cnt[b])
        assert k == len(want[b]), (b, k, len(want[b]))
        assert det[b, :k].tobytes() == want[b].tobytes(), b
        assert np.array_equal(idx[b, :k], widx[b]), b
        assert not det[b, k:].any() and (idx[b, k:] == -1).all()


# (batch, nc, anchors, cluster, max_det): 33 600 = the 640x640 anchor count, 134 400 = 1280x1280
CASES = [(64, 4, 33600, True, 300), (64, 80, 33600, False, 300), (64, 1, 33600, True, 1024), (8, 256, 33600, True, 300),
         (4, 80, 134400, True, 1024)]


@pytest.mark.parametrize("B,nc,A,cluster,max_det", CASES, ids=[f"b{c[0]}-nc{c[1]}-a{c[2]}-md{c[4]}" for c in CASES])
@pytest.mark.parametrize("conf", [0.001, 0.25])
def test_uyd_nms_ex_equals_oracle(B, nc, A, cluster, max_det, conf):
    y_np = synth_predictions(B, nc, A, seed=nc + A + B, cluster=cluster)
    y = torch.from_numpy(y_np).cuda()
    # the slab cut (> 4096 candidates per image) runs in every case, the max_nms truncation at conf 0.001 with nc > 1
    n_multi = int((y_np[:, 4:] > conf).sum((1, 2)).min())
    assert n_multi > 4096 and (n_multi > 30000 or conf == 0.25 or nc == 1)
    for multi_label, classes, agnostic in OPTIONS:
        max_wh = 0.0 if agnostic else 7680.0
        code, det, idx, cnt = _call(y, conf, 0.7, 30000, max_det, max_wh, _opt(multi_label, classes))
        assert code == 0
        want, widx = nref.non_max_suppression(y_np, conf, 0.7, max_det, 30000, return_index=True, classes=classes,
                                            agnostic=agnostic, multi_label=multi_label)
        _assert_equal_oracle(y_np, det, idx, cnt, want, widx)
        if classes is None:
            assert int(cnt.min()) > 0


def test_defaults_are_uyd_nms():
    from unina_yolo_dla_b200 import _lib

    y = torch.from_numpy(synth_predictions(16, 80, 33600, seed=3, cluster=True)).cuda()
    a = _call(y, 0.25, 0.7, 30000, 300, 7680.0, None, fn="uyd_nms")
    b = _call(y, 0.25, 0.7, 30000, 300, 7680.0, None)
    c = _call(y, 0.25, 0.7, 30000, 300, 7680.0, _lib.NmsOptions(0, 0, None))
    assert a[0] == b[0] == c[0] == 0
    for u, v in zip(a[1:], b[1:]):
        assert u.tobytes() == v.tobytes()
    for u, v in zip(a[1:], c[1:]):
        assert u.tobytes() == v.tobytes()
    # multi_label on one class is single-label (Ultralytics: multi_label &= nc > 1)
    y1 = torch.from_numpy(synth_predictions(4, 1, 33600, seed=4, cluster=True)).cuda()
    s = _call(y1, 0.25, 0.7, 30000, 300, 7680.0, None)
    m = _call(y1, 0.25, 0.7, 30000, 300, 7680.0, _lib.NmsOptions(1, 0, None))
    for u, v in zip(s[1:], m[1:]):
        assert u.tobytes() == v.tobytes()


def test_argument_errors_launch_nothing():
    from unina_yolo_dla_b200 import _lib

    y = torch.from_numpy(synth_predictions(2, 4, 1000, seed=5)).cuda()
    ids = (C.c_int * 2)(0, 1)
    bad = [_lib.NmsOptions(0, -1, None), _lib.NmsOptions(1, -1, C.cast(ids, C.POINTER(C.c_int))), _lib.NmsOptions(0, 2, None),
           _lib.NmsOptions(1, 1, None)]
    for o in bad:
        code, det, idx, cnt = _call(y, 0.25, 0.7, 30000, 300, 7680.0, o)
        assert code == E_ARG
        assert (det == 7.0).all() and (idx == -7).all() and (cnt == -7).all()


def test_property_ties_across_classes_and_anchors():
    """Boxes on a coarse integer lattice (many IoUs exactly equal to each other and to the threshold), scores from a
    small set shared across the classes of one anchor and across anchors, multi-label and class filters on: rows and
    anchor indices equal the oracle's, whose (score, anchor, class) order is pinned to torch.where + a stable sort."""
    from hypothesis import HealthCheck, given, settings, strategies as st

    import unina_yolo_dla_b200 as uyd

    m = uyd.UninaYoloB200.from_yaml()

    @settings(max_examples=40, deadline=None, suppress_health_check=list(HealthCheck), derandomize=True)
    @given(seed=st.integers(0, 2 ** 31 - 1), n=st.integers(1, 400), levels=st.integers(1, 6),
           iou=st.sampled_from([0.0, 1 / 3, 0.25, 0.5, 0.7, 1.0, 2 / 3]), nc=st.integers(1, 6),
           conf=st.sampled_from([0.0, 0.25, 0.5]), multi_label=st.booleans(), agnostic=st.booleans(),
           classes=st.one_of(st.none(), st.lists(st.integers(-1, 7), max_size=4)), max_det=st.sampled_from([5, 300]))
    def check(seed, n, levels, iou, nc, conf, multi_label, agnostic, classes, max_det):
        rng = np.random.default_rng(seed)
        A = 512
        y = np.zeros((1, 4 + nc, A), np.float32)
        y[0, 0:2, :n] = rng.integers(2, 12, (2, n)) * 4.0
        y[0, 2:4, :n] = rng.integers(1, 5, (2, n)) * 4.0
        y[0, 4:, :n] = rng.integers(1, levels + 1, (nc, n)).astype(np.float32) / (levels + 1)
        kw = dict(classes=classes, agnostic=agnostic, multi_label=multi_label)
        want, widx = nref.non_max_suppression(y, conf, iou, max_det, 30000, return_index=True, **kw)
        det, cnt, idx = m.nms(torch.from_numpy(y).cuda(), conf, iou, max_det, 30000, return_index=True, **kw)
        k = int(cnt[0])
        assert k == len(want[0])
        assert np.array_equal(idx[0, :k].cpu().numpy(), widx[0])
        assert det[0, :k].cpu().numpy().tobytes() == want[0].tobytes()

    check()


ENTRY_OPTIONS = [dict(), dict(multi_label=True), dict(classes=[0, 2]), dict(agnostic=True),
                 dict(multi_label=True, classes=[1], agnostic=True), dict(classes=[])]


def _yaml():
    import unina_yolo_dla_b200 as uyd

    return uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0).cuda()


def test_entry_points_equal_nms_of_forward():
    from unina_yolo_dla_b200 import preprocess as P

    m = _yaml()
    B, conf = 4, 0.01
    x = torch.rand(B, 3, 320, 320, generator=torch.Generator().manual_seed(11)).cuda()
    y = m.forward(x, raw_heads=False)
    frames = torch.randint(0, 256, (B, 300, 500, 4), dtype=torch.uint8, generator=torch.Generator().manual_seed(12)).cuda()
    yc = m.forward_camera(frames, letterbox=True)
    H, W = frames.shape[1:3]
    ref, ref_cam = [], []
    for kw in ENTRY_OPTIONS:
        d, c = m.nms(y, conf, **kw)
        ref.append((d, c))
        dc, cc = m.nms(yc, conf, **kw)
        P.letterbox_boxes(dc, cc, H, W, *P.camera_extent(H, W, None, True))
        ref_cam.append((dc, cc))
        if kw == dict(classes=[]):
            assert int(c.max()) == 0
        else:
            assert int(c.sum()) > 0
    assert not torch.equal(ref[0][0], ref[1][0])   # the multi-label rows differ from the single-label ones
    # alternate the option sets twice, so a graph captured for one set is replayed only for that set
    for _ in range(2):
        for kw, (d, c) in zip(ENTRY_OPTIONS, ref):
            for graph in (True, False):
                dg, cg = m.predict_batched(x, conf, graph=graph, **kw)
                assert torch.equal(cg, c) and torch.equal(dg, d), (kw, graph)
    for kw, (d, c), (dc, cc) in zip(ENTRY_OPTIONS, ref, ref_cam):
        rows = m.predict(x, conf, **kw)
        for b in range(B):
            assert torch.equal(rows[b], d[b, : int(c[b])])
        for to_host in (True, False):
            outs = list(m.predict_stream([x.cpu(), x.cpu()], conf, to_host=to_host, **kw))
            for ds, cs in outs:
                assert torch.equal(cs.cuda(), c) and torch.equal(ds.cuda(), d), (kw, to_host)
        dp, cp = m.predict_camera(frames, conf=conf, letterbox=True, **kw)
        assert torch.equal(cp, cc) and torch.equal(dp, dc), kw


def test_validator_path_multi_label_map_equals_oracle():
    """``model.val``'s NMS (conf 0.001, iou 0.7, multi_label) on the YAML network, then mAP on the device, against the
    oracle's multi-label NMS of the same predictions and the restated Ultralytics metrics on its rows."""
    import map_scenes as S
    from oracle import mapref as er
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    m = _yaml()
    B = 8
    x = torch.rand(B, 3, 320, 320, generator=torch.Generator().manual_seed(5)).cuda()
    det, cnt = m.predict_batched(x, conf=0.001, iou=0.7, multi_label=True)
    single, scnt = m.predict_batched(x, conf=0.001, iou=0.7)
    y = m.forward(x, raw_heads=False).cpu().numpy()
    want = nref.non_max_suppression(y, 0.001, 0.7, 300, 30000, multi_label=True)
    det_h, cnt_h = det.cpu().numpy(), cnt.cpu().numpy()
    for b in range(B):
        assert int(cnt_h[b]) == len(want[b]) and det_h[b, : cnt_h[b]].tobytes() == want[b].tobytes()
    assert not (torch.equal(det, single) and torch.equal(cnt, scnt))
    dets = [torch.from_numpy(w) for w in want]
    assert sum(len(d) for d in dets) > 100
    g = torch.Generator().manual_seed(6)
    gts = []
    for d in dets:   # labels near a sample of the detections plus unmatched ones
        pick = d[torch.randperm(len(d), generator=g)[:12]]
        box = pick[:, :4] + torch.randn(len(pick), 4, generator=g) * 3
        cls = torch.where(torch.rand(len(pick), generator=g) < 0.8, pick[:, 5], torch.randint(0, 4, (len(pick),), generator=g).float())
        extra = torch.rand(4, 2, generator=g) * 280
        gts.append(torch.cat((torch.cat((cls[:, None], box), 1),
                              torch.cat((torch.randint(0, 4, (4, 1), generator=g).float(), extra, extra + 30), 1))))
    gt, gcnt = S.pack(dets, gts, det.shape[1])[2:]
    ev = DetectionEvaluator(nc=4)
    ev.update(det, cnt, gt.cuda(), gcnt.cuda())
    got, ref = ev.map_metrics(), er.map_eval(dets, gts)
    for k in er.RESULT_KEYS + ("fitness",):
        assert got[k] == ref[k], (k, got[k], ref[k])
    for k in ("ap50", "ap", "ap_class_index"):
        assert np.array_equal(got[k], ref[k]), k
    assert got["metrics/mAP50(B)"] > 0
