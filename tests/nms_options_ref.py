"""Ultralytics 8.3.x ``non_max_suppression`` with its ``classes``, ``agnostic`` and ``multi_label`` options, restated in
numpy on top of the oracle's torchvision-semantics greedy NMS (``oracle.postproc.nms_sorted``).  TEST INFRASTRUCTURE
for tests/test_nms_options_host.py and tests/test_gpu_nms_options.py.

With the options at their defaults the result is ``oracle.postproc.non_max_suppression``'s (checked by the host test).

PARITY UNPINNED: ``ultralytics`` is not installed where this is tested, so the host test pins the restatement to a
literal torch + torchvision composition of the Ultralytics statements and compares against
``ultralytics.utils.ops.non_max_suppression`` only when it imports.  Assumed behaviours:
  * ``multi_label &= nc > 1``; candidates are ``i, j = torch.where(cls > conf)`` over the rows with ``amax > conf``,
    in row-major order (anchor, then class), each row's conf the score of class j;
  * ``classes``: ``(x[:, 5:6] == classes).any(1)`` after the best class / the pairs are formed and before the
    ``max_nms`` truncation (single-label: an anchor whose best class is not listed is dropped, it does not fall back
    to its second class); ``[]`` keeps nothing;
  * ``c = cls * (0 if agnostic else max_wh)``.
Ties: the stable order, as in the oracle -- score descending, then anchor, then class ascending.
"""
from __future__ import annotations

import numpy as np

from oracle import postproc as pp


def stable_top(conf: np.ndarray, k: int) -> np.ndarray:
    """``argsort(-conf, kind="stable")[:k]`` without sorting every entry: the rows scoring at least the k-th largest
    score, stably sorted (a subset keeps its relative order, so the first k are the same)."""
    if len(conf) <= k:
        return np.argsort(-conf, kind="stable")
    kth = np.partition(conf, len(conf) - k)[len(conf) - k]
    sub = np.nonzero(conf >= kth)[0]
    return sub[np.argsort(-conf[sub], kind="stable")[:k]]


def non_max_suppression(pred: np.ndarray, conf_thres=0.25, iou_thres=0.45, max_det=300, max_nms=30000, max_wh=7680.0,
                        return_index=False, classes=None, agnostic=False, multi_label=False):
    """``pred``: [B, 4+nc, A] fp32 (cx, cy, w, h, class scores).  Returns a list of [N_i, 6] fp32 rows
    (x1, y1, x2, y2, conf, cls) and, optionally, the anchor index of every kept row."""
    pred = np.asarray(pred, dtype=np.float32)
    B, no, A = pred.shape
    multi_label = multi_label and no - 4 > 1
    keep_cls = None if classes is None else np.asarray([classes] if np.isscalar(classes) else list(classes), np.float64)
    thr = np.float32(conf_thres)
    outs, idxs = [], []
    for b in range(B):
        p = pred[b].T  # [A, 4+nc]
        xc = p[:, 4:].max(1) > thr
        anchor = np.nonzero(xc)[0]
        x = p[xc]
        half = x[:, 2:4] / np.float32(2)
        box = np.concatenate((x[:, 0:2] - half, x[:, 0:2] + half), 1).astype(np.float32)
        if multi_label:
            i, j = np.nonzero(x[:, 4:] > thr)   # row-major, as torch.where
            box, conf, anchor = box[i], x[i, 4 + j], anchor[i]
        else:
            j = x[:, 4:].argmax(1)
            conf = x[:, 4:].max(1)
            m = conf > thr
            box, conf, j, anchor = box[m], conf[m], j[m], anchor[m]
        if keep_cls is not None:
            m = (j.astype(np.float32)[:, None] == keep_cls[None, :]).any(1)
            box, conf, j, anchor = box[m], conf[m], j[m], anchor[m]
        order = stable_top(conf, max_nms)
        box, conf, j, anchor = box[order], conf[order], j[order], anchor[order]
        off = (j.astype(np.float32) * np.float32(0.0 if agnostic else max_wh))[:, None]
        keep = pp.nms_sorted((box + off).astype(np.float32), iou_thres, max_det)
        outs.append(np.concatenate((box[keep], conf[keep, None], j[keep, None].astype(np.float32)), 1).astype(np.float32))
        idxs.append(anchor[keep].astype(np.int64))
    return (outs, idxs) if return_index else outs
