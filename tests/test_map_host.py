"""mAP50 / mAP50-95 semantics on the host: known answers of the restated Ultralytics DetectionValidator /
ap_per_class (oracle/mapref.py), the one-pass (m(p), v*(p)] matching form the CUDA matcher uses against the literal
match_predictions, and the library's numpy tail (evaluate.map_results) against the restatement."""
import numpy as np
import pytest
import torch

import map_scenes as S
from oracle import mapref as er

THR = er.IOUV.numpy()


def _tp(det, gt):
    det, gt = torch.tensor(det, dtype=torch.float32).reshape(-1, 6), torch.tensor(gt, dtype=torch.float32).reshape(-1, 5)
    iou = er.box_iou(gt[:, 1:], det[:, :4])
    lit = er.match_predictions(det[:, 5], gt[:, 0], iou)
    assert np.array_equal(lit, er.match_one_pass(det[:, 5], gt[:, 0], iou))
    return lit


def test_perfect_detector_is_0995():
    gts = [torch.tensor([[0, 10, 10, 50, 50], [1, 100, 100, 150, 160.0], [1, 300, 20, 340, 90]])]
    dets = [torch.tensor([[10, 10, 50, 50, 0.9, 0], [100, 100, 150, 160, 0.8, 1], [300, 20, 340, 90, 0.7, 1.0]])]
    r = er.map_eval(dets, gts)
    assert r["metrics/mAP50(B)"] == 0.995 and r["ap50"].tolist() == [0.995, 0.995]
    assert abs(r["metrics/mAP50-95(B)"] - 0.995) < 1e-15
    assert r["metrics/precision(B)"] == 1.0 and r["metrics/recall(B)"] == 1.0


def test_iou_072_is_tp_up_to_070():
    tp = _tp([[0, 0, 72, 100, 0.9, 0]], [[0, 0, 0, 100, 100]])
    assert tp[0].tolist() == [True] * 5 + [False] * 5


def test_higher_confidence_wins_over_higher_iou():
    # row 0 (higher confidence) IoU 0.8, row 1 IoU 0.95: row 0 takes the label wherever it qualifies
    tp = _tp([[0, 0, 80, 100, 0.9, 0], [0, 0, 95, 100, 0.8, 0]], [[0, 0, 0, 100, 100]])
    assert tp[0].tolist() == (THR <= np.float32(0.8)).tolist()
    assert tp[1].tolist() == (THR > np.float32(0.8)).tolist()


def test_taken_best_label_makes_fp_despite_other_overlap():
    # row 1's best label (0) is taken by row 0; it also overlaps label 1 at IoU 0.54, which stays unmatched
    gt = [[0, 0, 0, 100, 100], [0, 40, 0, 140, 100]]
    tp = _tp([[0, 0, 100, 100, 0.9, 0], [10, 0, 110, 100, 0.8, 0]], gt)
    iou = er.box_iou(torch.tensor(gt)[:, 1:], torch.tensor([[10.0, 0, 110, 100]]))
    assert float(iou[1, 0]) >= 0.5 and float(iou[0, 0]) > float(iou[1, 0])
    assert tp[0].all() and not tp[1].any()


def test_cross_class_never_matches():
    assert not _tp([[0, 0, 100, 100, 0.9, 1]], [[0, 0, 0, 100, 100]]).any()


def test_equal_iou_goes_to_the_higher_label_index():
    # row 0 has the same IoU (90 / 110) with labels 0 and 1 and takes label 1; so row 1, exactly on label 0, is a TP
    gt = [[0, 0, 0, 10, 10], [0, 2, 0, 12, 10]]
    det = [[1, 0, 11, 10, 0.9, 0], [0, 0, 10, 10, 0.8, 0]]
    iou = er.box_iou(torch.tensor(gt)[:, 1:], torch.tensor(det)[:, :4])
    assert float(iou[0, 0]) == float(iou[1, 0])
    tp = _tp(det, gt)
    assert tp[0, :4].all() and tp[1].all()


def test_equal_confidence_ranks_in_record_order():
    gt = torch.tensor([[0, 0, 0, 100, 100], [0, 200, 0, 300, 100]])
    hit, miss = [0, 0, 100, 100, 0.5, 0], [400, 0, 500, 100, 0.5, 0]
    a = er.map_eval([torch.tensor([hit, miss])], [gt])
    b = er.map_eval([torch.tensor([miss, hit])], [gt])
    assert a["metrics/mAP50(B)"] > b["metrics/mAP50(B)"]                    # the stable order decides
    c = er.map_eval([torch.tensor([miss]), torch.tensor([hit])], [gt[:0], gt])
    assert c["metrics/mAP50(B)"] == b["metrics/mAP50(B)"]                   # earlier image first


def test_images_without_detections_or_labels():
    gts = [torch.tensor([[0, 0, 0, 100, 100.0]]), torch.tensor([[0, 0, 0, 50, 50.0]]), torch.zeros(0, 5)]
    dets = [torch.tensor([[0, 0, 100, 100, 0.9, 0.0]]), torch.zeros(0, 6), torch.tensor([[0, 0, 30, 30, 0.5, 0.0]])]
    tp, conf, pcls, tcls = er.map_stats(dets, gts)
    assert tp.shape == (2, 10) and tp[:, 0].tolist() == [True, False] and tcls.tolist() == [0, 0]
    r = er.map_eval(dets, gts)
    # recall 0.5 at precision 1, then an FP: the 101-point curve is 1 on [0, 0.5), 0.5 at 0.5, then down to 0
    assert abs(r["metrics/mAP50(B)"] - 0.6225) < 0.01 and r["ap_class_index"].tolist() == [0]
    none = er.map_eval([torch.zeros(0, 6)], [gts[0]])
    assert none["metrics/mAP50(B)"] == 0.0 and len(none["ap_class_index"]) == 0   # no TP: nothing is reported


@pytest.mark.parametrize("lattice", [False, True])
def test_one_pass_equals_literal_match_predictions(lattice):
    ties = 0
    for seed in range(6):
        dets, gts = S.scene(12, 100 + seed, max_det=200, n_gt=24, lattice=lattice)
        for d, g in zip(dets, gts):
            if not len(d) or not len(g):
                continue
            iou = er.box_iou(g[:, 1:], d[:, :4])
            lit = er.match_predictions(d[:, 5], g[:, 0], iou)
            assert np.array_equal(lit, er.match_one_pass(d[:, 5], g[:, 0], iou))
            same = (iou * (g[:, 0:1] == d[:, 5])).numpy()
            top = np.sort(same, 0)[-2:] if len(g) > 1 else None
            ties += 0 if top is None else int(((top[0] == top[1]) & (top[1] >= 0.5)).sum())
    if lattice:
        assert ties > 3   # equal best IoUs of one detection were exercised


def test_library_tail_equals_restatement():
    from unina_yolo_dla_b200.evaluate import map_results

    for seed, lattice in ((3, False), (4, True)):
        dets, gts = S.scene(24, seed, nc=6, lattice=lattice)
        ref = er.map_eval(dets, gts)
        raw, nc = ref["raw"], 8
        ap, pc, rc, nl = np.zeros((nc, 10)), np.zeros((nc, 1000)), np.zeros((nc, 1000)), np.zeros(nc, np.int64)
        idx = raw["ap_class_index"]
        ap[idx], pc[idx], rc[idx], nl[idx] = raw["ap"], raw["p_curve"], raw["r_curve"], raw["nt"]
        got = map_results(ap, pc, rc, nl)
        for k in er.RESULT_KEYS + ("fitness",):
            assert got[k] == ref[k], k
        for k in ("ap50", "ap", "ap_class_index"):
            assert np.array_equal(got[k], ref[k]), k
    assert map_results(None, None, None, np.ones(3))["metrics/mAP50-95(B)"] == 0.0


def test_restatement_equals_ultralytics_when_installed():
    ul = pytest.importorskip("ultralytics")   # noqa: F841  PARITY UNPINNED otherwise
    from ultralytics.models.yolo.detect import DetectionValidator
    from ultralytics.utils.metrics import ap_per_class

    v = DetectionValidator()
    dets, gts = S.scene(8, 7, nc=4)   # continuous boxes and confidences: no ties
    for d, g in zip(dets, gts):
        if len(d) and len(g):
            iou = er.box_iou(g[:, 1:], d[:, :4])
            assert np.array_equal(v.match_predictions(d[:, 5], g[:, 0], iou).numpy(), er.match_predictions(d[:, 5], g[:, 0], iou))
    tp, conf, pcls, tcls = er.map_stats(dets, gts)
    up = ap_per_class(tp, conf, pcls, tcls)
    mine = er.ap_per_class(tp, conf, pcls, tcls)
    assert np.array_equal(up[5], mine["ap"]) and np.array_equal(up[7], mine["p_curve"]) and np.array_equal(up[8], mine["r_curve"])
