"""The restated Ultralytics ``non_max_suppression`` with its ``classes`` / ``agnostic`` / ``multi_label`` options
(tests/nms_options_ref.py) against a literal torch + torchvision composition of the Ultralytics statements, live against
``ultralytics`` when it imports, on known answers, and at its defaults against oracle/postproc.py."""
import numpy as np
import pytest
import torch

import nms_options_ref as nref

CLASSES = [None, [], [1], [0, 3, 99, -1]]


def composed(pred, conf, iou, classes=None, agnostic=False, multi_label=False, max_det=300, max_nms=30000, max_wh=7680):
    """Ultralytics 8.3.x non_max_suppression, statement by statement, in torch + torchvision (stable argsort)."""
    import torchvision

    pred = torch.from_numpy(pred)
    nc = pred.shape[1] - 4
    multi_label &= nc > 1
    cls_t = torch.tensor(classes) if classes is not None else None
    xc = pred[:, 4:].amax(1) > conf
    outs, idxs = [], []
    for b in range(pred.shape[0]):
        x = pred[b].T
        xk = torch.arange(x.shape[0])
        x, xk = x[xc[b]], xk[xc[b]]
        box = torch.cat((x[:, :2] - x[:, 2:4] / 2, x[:, :2] + x[:, 2:4] / 2), 1)
        cls = x[:, 4:]
        if multi_label:
            i, j = torch.where(cls > conf)
            x = torch.cat((box[i], x[i, 4 + j, None], j[:, None].float()), 1)
            xk = xk[i]
        else:
            c, j = cls.max(1, keepdim=True)
            filt = c.view(-1) > conf
            x = torch.cat((box, c, j.float()), 1)[filt]
            xk = xk[filt]
        if cls_t is not None:
            filt = (x[:, 5:6] == cls_t).any(1)
            x, xk = x[filt], xk[filt]
        if x.shape[0] > max_nms:
            filt = x[:, 4].argsort(descending=True, stable=True)[:max_nms]
            x, xk = x[filt], xk[filt]
        c = x[:, 5:6] * (0 if agnostic else max_wh)
        i = torchvision.ops.nms(x[:, :4] + c, x[:, 4], iou)[:max_det]
        outs.append(x[i].numpy())
        idxs.append(xk[i].numpy())
    return outs, idxs


def scene(nc, seed, B=2, A=6000, ties=False):
    rng = np.random.default_rng(seed)
    pred = np.zeros((B, 4 + nc, A), np.float32)
    pred[:, 0:2] = rng.uniform(0, 640, (B, 2, A))
    pred[:, 2:4] = rng.uniform(4, 120, (B, 2, A))
    sc = rng.uniform(0, 1, (B, nc, A)) ** 3
    pred[:, 4:] = np.round(sc * 16) / 16 if ties else sc   # ties: equal scores across anchors and across classes
    return pred


@pytest.mark.parametrize("nc", [1, 4, 80])
@pytest.mark.parametrize("classes", CLASSES, ids=str)
@pytest.mark.parametrize("agnostic", [False, True])
@pytest.mark.parametrize("multi_label", [False, True])
def test_oracle_equals_torch_torchvision_composition(nc, classes, agnostic, multi_label):
    max_nms = 1000
    for seed, ties in ((nc, False), (nc + 100, True)):
        pred = scene(nc, seed, ties=ties)
        kw = dict(classes=classes, agnostic=agnostic, multi_label=multi_label)
        # more candidates than max_nms (whenever the filter leaves enough), so the truncation is exercised
        n_cand = (pred[:, 4:] > 0.25).sum((1, 2)) if multi_label else (pred[:, 4:].max(1) > 0.25).sum(1)
        assert n_cand.min() > 2 * max_nms
        got, gidx = nref.non_max_suppression(pred, 0.25, 0.7, 300, max_nms, return_index=True, **kw)
        want, widx = composed(pred, 0.25, 0.7, max_det=300, max_nms=max_nms, **kw)
        for b in range(pred.shape[0]):
            assert got[b].tobytes() == want[b].tobytes(), (seed, b)
            np.testing.assert_array_equal(gidx[b], widx[b])
        if classes == []:
            assert all(len(g) == 0 for g in got)
        elif classes is None:
            assert all(len(g) == 300 for g in got)


def test_live_ultralytics():
    ops = pytest.importorskip("ultralytics.utils.ops")
    for nc in (1, 4, 80):
        pred = scene(nc, 7 + nc)   # continuous scores: Ultralytics' unstable argsort meets no ties
        for classes in CLASSES:
            for agnostic in (False, True):
                for multi_label in (False, True):
                    want, widx = nref.non_max_suppression(pred, 0.25, 0.7, 300, 1500, return_index=True, classes=classes,
                                                        agnostic=agnostic, multi_label=multi_label)
                    live, lidx = ops.non_max_suppression(torch.from_numpy(pred.copy()), 0.25, 0.7, classes=classes,
                                                         agnostic=agnostic, multi_label=multi_label, max_det=300,
                                                         max_nms=1500, max_time_img=1e9, in_place=False, return_idxs=True)
                    for b in range(pred.shape[0]):
                        assert live[b].numpy().tobytes() == want[b].tobytes()
                        np.testing.assert_array_equal(lidx[b].numpy(), widx[b])


def one(boxes_scores, conf=0.25, iou=0.7, **kw):
    """One image from rows (cx, cy, w, h, score_0, ..., score_{nc-1})."""
    pred = np.asarray(boxes_scores, np.float32).T[None].copy()
    out, idx = nref.non_max_suppression(pred, conf, iou, 300, 30000, return_index=True, **kw)
    return out[0], idx[0]


def test_multi_label_gives_one_row_per_class_above_conf():
    rows = [[50, 50, 20, 20, 0.6, 0.8]]
    out, idx = one(rows, multi_label=True)
    assert out[:, 5].tolist() == [1.0, 0.0] and out[:, 4].tolist() == [np.float32(0.8), np.float32(0.6)]
    assert idx.tolist() == [0, 0]
    out, idx = one(rows)
    assert out[:, 5].tolist() == [1.0] and idx.tolist() == [0]


def test_multi_label_agnostic_keeps_the_higher_pair_unless_iou_1():
    out, _ = one([[50, 50, 20, 20, 0.6, 0.8]], multi_label=True, agnostic=True)
    assert out[:, 5].tolist() == [1.0]
    out, _ = one([[50, 50, 20, 20, 0.7, 0.7]], multi_label=True, agnostic=True)   # a tie: class 0 comes first
    assert out[:, 5].tolist() == [0.0]
    out, _ = one([[50, 50, 20, 20, 0.6, 0.8]], iou=1.0, multi_label=True, agnostic=True)   # IoU 1 is not > 1
    assert out[:, 5].tolist() == [1.0, 0.0]


def test_overlapping_boxes_of_two_classes():
    rows = [[50, 50, 20, 20, 0.9, 0.1], [51, 50, 20, 20, 0.1, 0.8]]
    out, idx = one(rows)
    assert idx.tolist() == [0, 1] and out[:, 5].tolist() == [0.0, 1.0]
    out, idx = one(rows, agnostic=True)
    assert idx.tolist() == [0] and out[:, 5].tolist() == [0.0]


def test_single_label_filter_applies_to_the_best_class():
    rows = [[50, 50, 20, 20, 0.9, 0.5], [200, 200, 20, 20, 0.1, 0.6]]
    out, idx = one(rows, classes=[1])
    assert idx.tolist() == [1] and out[:, 5].tolist() == [1.0]   # anchor 0's best class is 0: dropped, no fallback
    out, idx = one(rows, classes=[1], multi_label=True)
    assert idx.tolist() == [1, 0] and out[:, 4].tolist() == [np.float32(0.6), np.float32(0.5)]


def test_empty_class_list_keeps_nothing():
    rows = [[50, 50, 20, 20, 0.9, 0.5], [200, 200, 20, 20, 0.1, 0.6]]
    for ml in (False, True):
        out, idx = one(rows, classes=[], multi_label=ml)
        assert out.shape == (0, 6) and len(idx) == 0


def test_one_class_multi_label_is_single_label():
    pred = scene(1, 3)
    for classes in (None, [0]):
        a = nref.non_max_suppression(pred, 0.25, 0.7, 300, 1500, return_index=True, classes=classes, multi_label=True)
        b = nref.non_max_suppression(pred, 0.25, 0.7, 300, 1500, return_index=True, classes=classes)
        for b_ in range(pred.shape[0]):
            assert a[0][b_].tobytes() == b[0][b_].tobytes() and np.array_equal(a[1][b_], b[1][b_])


@pytest.mark.parametrize("nc", [1, 4, 80])
def test_defaults_equal_the_oracle(nc):
    from oracle import postproc as pp

    for ties in (False, True):
        pred = scene(nc, 200 + nc, ties=ties)
        a = nref.non_max_suppression(pred, 0.25, 0.7, 300, 1000, return_index=True)
        b = pp.non_max_suppression(pred, 0.25, 0.7, 300, 1000, return_index=True)
        for i in range(pred.shape[0]):
            assert a[0][i].tobytes() == b[0][i].tobytes() and np.array_equal(a[1][i], b[1][i])
