"""Oracle: mAP50 / mAP50-95 of Ultralytics ``model.val``, restated.  TEST INFRASTRUCTURE.

``match_predictions`` / ``smooth`` / ``compute_ap`` / ``ap_per_class`` / ``det_metrics`` / ``map_eval`` restate
Ultralytics 8.3.x DetectionValidator.match_predictions (the non-scipy branch), update_metrics / get_stats and
utils.metrics (ap_per_class, compute_ap with method "interp", smooth, Metric.mean_results / fitness,
DetMetrics.results_dict).  PARITY UNPINNED: ``ultralytics`` is not installable here; when it can be imported,
tests/test_map_host.py compares against it live.  Assumed behaviours:
  - iouv = torch.linspace(0.5, 0.95, 10) in fp32, compared ``iou >= thr`` in fp32 (NEP 50: the Python float
    threshold is weak, so numpy compares in the array's float32);
  - box_iou with eps = 1e-7 (``evalref.box_iou``, ``iou_ultra`` in csrc/evalmatch.cu), iou[L, D] = box_iou(gt, det);
  - recall = tpc / (n_l + 1e-16), precision = tpc / (tpc + fpc), both int64 counts divided in fp64;
  - the 1000-point curves np.interp(-x, -conf, ., left=0) (recall) and left=1 (precision) at IoU 0.5;
  - compute_ap: sentinels [0] + r + [1] / [1] + p + [0], the flipped maximum.accumulate envelope, np.interp at
    np.linspace(0, 1, 101) and np.trapezoid;
  - smooth(f=0.1) of the class-mean F1 curve (a 101-tap box filter), its argmax, tp = (r * nt).round(),
    fp = (tp / (p + 1e-16) - tp).round();
  - results keys metrics/precision(B), metrics/recall(B), metrics/mAP50(B), metrics/mAP50-95(B), fitness with
    fitness = 0.1 * mAP50 + 0.9 * mAP50-95 (np.nan_to_num of the four, weights [0, 0, 0.1, 0.9], summed);
  - get_stats runs ap_per_class only when some prediction is a TP at some threshold; otherwise every metric is 0
    and no class is reported.  Classes without labels are never reported.
Two tie orders are implementation-defined upstream (numpy's default argsort is unstable and dispatches to SIMD
sorts) and are fixed here with kind="stable"; they are the only inputs on which an Ultralytics run can differ:
  - one prediction with equal IoU to two same-class ground truths: the higher ground-truth index wins (what
    ``argsort()[::-1]`` does on short arrays, where numpy sorts by insertion);
  - equal confidences: predictions rank by (order of the update calls, image in the batch, row in the image).
Pure-Python loops per image: test sizes and the measurement in tools/map_bench.py only.
"""
from __future__ import annotations

import numpy as np
import torch

from .evalref import box_iou  # noqa: F401  (Ultralytics metrics.box_iou, eps = 1e-7)

IOUV = torch.linspace(0.5, 0.95, 10)
RESULT_KEYS = ("metrics/precision(B)", "metrics/recall(B)", "metrics/mAP50(B)", "metrics/mAP50-95(B)")


def match_predictions(pred_classes, true_classes, iou, iouv=IOUV):
    """DetectionValidator.match_predictions, non-scipy branch.  pred_classes [D], true_classes [L], iou [L, D]
    (box_iou(gt, det)); returns the [D, len(iouv)] bool TP matrix."""
    correct = np.zeros((pred_classes.shape[0], iouv.shape[0])).astype(bool)
    correct_class = true_classes[:, None] == pred_classes
    iou = (iou * correct_class).cpu().numpy()
    for i, threshold in enumerate(iouv.cpu().tolist()):
        matches = np.array(np.nonzero(iou >= threshold)).T
        if matches.shape[0]:
            if matches.shape[0] > 1:
                matches = matches[iou[matches[:, 0], matches[:, 1]].argsort(kind="stable")[::-1]]
                matches = matches[np.unique(matches[:, 1], return_index=True)[1]]
                matches = matches[np.unique(matches[:, 0], return_index=True)[1]]
            correct[matches[:, 1].astype(int), i] = True
    return correct


def match_one_pass(pred_classes, true_classes, iou, iouv=IOUV):
    """The same matrix in one pass over the predictions (the form csrc/evalmatch.cu uses): j*(p) is p's best
    same-class ground truth (highest index among equal IoUs), v*(p) that IoU, m(p) the largest v*(q) over earlier
    q with j*(q) = j*(p); p is a TP at t exactly when m(p) < t <= v*(p).  Thresholds must be positive."""
    iou = np.nan_to_num((iou * (true_classes[:, None] == pred_classes)).cpu().numpy(), nan=0.0)
    thr = iouv.cpu().numpy()
    correct = np.zeros((iou.shape[1], len(thr)), bool)
    if iou.shape[0] == 0:
        return correct
    taken = {}
    for p in range(iou.shape[1]):
        col = iou[:, p]
        j = len(col) - 1 - int(np.argmax(col[::-1]))
        v = col[j]
        m = taken.get(j, np.float32(0.0))
        correct[p] = (m < thr) & (thr <= v)
        taken[j] = max(m, v)
    return correct


def smooth(y, f=0.05):
    nf = round(len(y) * f * 2) // 2 + 1
    p = np.ones(nf // 2)
    yp = np.concatenate((p * y[0], y, p * y[-1]), 0)
    return np.convolve(yp, np.ones(nf) / nf, mode="valid")


def compute_ap(recall, precision):
    mrec = np.concatenate(([0.0], recall, [1.0]))
    mpre = np.concatenate(([1.0], precision, [0.0]))
    mpre = np.flip(np.maximum.accumulate(np.flip(mpre)))
    x = np.linspace(0, 1, 101)
    return np.trapezoid(np.interp(x, mrec, mpre), x), mpre, mrec


def ap_per_class(tp, conf, pred_cls, target_cls, eps=1e-16):
    """utils.metrics.ap_per_class without plots; the confidence sort is stable (see the header)."""
    i = np.argsort(-conf, kind="stable")
    tp, conf, pred_cls = tp[i], conf[i], pred_cls[i]
    unique_classes, nt = np.unique(target_cls, return_counts=True)
    nc = unique_classes.shape[0]
    x = np.linspace(0, 1, 1000)
    ap, p_curve, r_curve = np.zeros((nc, tp.shape[1])), np.zeros((nc, 1000)), np.zeros((nc, 1000))
    for ci, c in enumerate(unique_classes):
        i = pred_cls == c
        n_l = nt[ci]
        n_p = i.sum()
        if n_p == 0 or n_l == 0:
            continue
        fpc = (1 - tp[i]).cumsum(0)
        tpc = tp[i].cumsum(0)
        recall = tpc / (n_l + eps)
        r_curve[ci] = np.interp(-x, -conf[i], recall[:, 0], left=0)
        precision = tpc / (tpc + fpc)
        p_curve[ci] = np.interp(-x, -conf[i], precision[:, 0], left=1)
        for j in range(tp.shape[1]):
            ap[ci, j], _, _ = compute_ap(recall[:, j], precision[:, j])
    f1_curve = 2 * p_curve * r_curve / (p_curve + r_curve + eps)
    i = smooth(f1_curve.mean(0), 0.1).argmax()
    p, r, f1 = p_curve[:, i], r_curve[:, i], f1_curve[:, i]
    tp = (r * nt).round()
    fp = (tp / (p + eps) - tp).round()
    return dict(tp=tp, fp=fp, p=p, r=r, f1=f1, ap=ap, ap_class_index=unique_classes.astype(int), p_curve=p_curve,
                r_curve=r_curve, f1_curve=f1_curve, nt=nt)


def det_metrics(tp, conf, pred_cls, target_cls):
    """DetectionValidator.get_stats -> DetMetrics.process -> results_dict, plus the per-class ap50 / ap /
    ap_class_index (Metric.ap50, Metric.ap, ap_class_index) and the raw ap_per_class output under "raw"."""
    if len(tp) and tp.any():
        raw = ap_per_class(tp, conf, pred_cls, target_cls)
        p, r, all_ap, idx = raw["p"], raw["r"], raw["ap"], raw["ap_class_index"]
    else:
        raw, p, r, all_ap, idx = None, np.zeros(0), np.zeros(0), np.zeros((0, tp.shape[1] if tp.ndim == 2 else 10)), np.zeros(0, int)
    mean = [p.mean() if len(p) else 0.0, r.mean() if len(r) else 0.0, all_ap[:, 0].mean() if len(all_ap) else 0.0,
            all_ap.mean() if len(all_ap) else 0.0]
    fitness = (np.nan_to_num(np.array(mean)) * [0.0, 0.0, 0.1, 0.9]).sum()
    out = dict(zip(RESULT_KEYS + ("fitness",), mean + [fitness]))
    out.update(ap50=all_ap[:, 0] if len(all_ap) else np.zeros(0), ap=all_ap.mean(1) if len(all_ap) else np.zeros(0),
               ap_class_index=idx, raw=raw)
    return out


def map_stats(dets, gts, iouv=IOUV, one_pass=False):
    """DetectionValidator.update_metrics over images in processing order.  dets: [N, 6] tensors (x1,y1,x2,y2,conf,cls)
    in confidence order, gts: [G, 5] tensors (cls,x1,y1,x2,y2), both in the same pixel space.  Returns the
    concatenated (tp [P, T] bool, conf [P] fp32, pred_cls [P], target_cls [L])."""
    match = match_one_pass if one_pass else match_predictions
    tps, confs, pcls, tcls = [], [], [], []
    for det, gt in zip(dets, gts):
        det, gt = det.float().cpu(), gt.float().cpu()
        tcls.append(gt[:, 0].numpy())
        if len(det) == 0:
            continue
        tp = np.zeros((len(det), len(iouv)), bool)
        if len(gt):
            tp = match(det[:, 5], gt[:, 0], box_iou(gt[:, 1:5], det[:, :4]), iouv)
        tps.append(tp)
        confs.append(det[:, 4].numpy())
        pcls.append(det[:, 5].numpy())
    T = len(iouv)
    cat = lambda xs, shape, dt: np.concatenate(xs) if xs else np.zeros(shape, dt)   # noqa: E731
    return (cat(tps, (0, T), bool), cat(confs, (0,), np.float32), cat(pcls, (0,), np.float32), cat(tcls, (0,), np.float32))


def map_eval(dets, gts):
    """The model.val box metrics of a whole validation pass (results dict + per-class ap50 / ap / ap_class_index)."""
    return det_metrics(*map_stats(dets, gts))
