"""Batched evaluation consumer of the detections (reference: UninaValidator trainer.py:196-286, the
small-object metrics; calibrate_conformal_prediction train.py:299-520, the conformal quantile; with ``nc`` set,
the box metrics of Ultralytics ``model.val``: precision, recall, mAP50, mAP50-95 and fitness).  Everything
stays on the GPU; with several ranks the detections are gathered first (dp.gather_detections, the only
collective of the path) or the counters / scores / records are reduced at the end (``reduce``)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import check


# Ultralytics DetectionValidator.iouv and DetMetrics.keys
MAP_IOUV = torch.linspace(0.5, 0.95, 10)
MAP_KEYS = ("metrics/precision(B)", "metrics/recall(B)", "metrics/mAP50(B)", "metrics/mAP50-95(B)")
_PAD_KEY = torch.iinfo(torch.int64).max   # the key of a padding row: sorts behind every class


class DetectionEvaluator:
    """``nc`` (opt-in) also collects, per ``update``, the records ``map_metrics`` turns into mAP50 / mAP50-95 for
    classes 0 .. nc - 1; with ``nc=None`` nothing of that runs."""

    def __init__(self, size_threshold: float = 15.0, small_iou: float = 0.45, match_iou: float = 0.5, device=None, nc=None):
        self.size_threshold, self.small_iou, self.match_iou = float(size_threshold), float(small_iou), float(match_iou)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.nc = None if nc is None else int(nc)
        if self.nc is not None and self.nc <= 0:
            raise ValueError("nc must be positive")
        self.reset()

    def reset(self) -> None:
        self.counters = torch.zeros(3, dtype=torch.int64, device=self.device)   # small-object TP, FP, FN
        self._scores = []
        if self.nc is not None:
            self._n_labels = torch.zeros(self.nc, dtype=torch.int64, device=self.device)
            self._dropped = torch.zeros(1, dtype=torch.int64, device=self.device)
            self._keys, self._masks = [], []   # per update: sort keys [B * max_det] int64, TP masks (uint16 bits in int16)

    @torch.no_grad()
    def update(self, det: torch.Tensor, cnt: torch.Tensor, gt: torch.Tensor, gt_cnt: torch.Tensor) -> None:
        """det [B, max_det, 6] / cnt [B] as returned by ``predict_batched``; gt [B, G, 5] rows
        (cls, x1, y1, x2, y2) in pixels, gt_cnt [B] (int32).  No host synchronisation."""
        assert det.is_cuda and det.dtype == torch.float32 and det.is_contiguous() and det.shape[2] == 6
        assert gt.is_cuda and gt.dtype == torch.float32 and gt.is_contiguous() and gt.shape[2] == 5
        assert cnt.dtype == torch.int32 and gt_cnt.dtype == torch.int32 and cnt.is_cuda and gt_cnt.is_cuda
        B, max_det, _ = det.shape
        scores = torch.empty(B, max_det, dtype=torch.float32, device=det.device)
        dev = det.device.index if det.device.index is not None else torch.cuda.current_device()
        check(_lib.lib().uyd_eval_update(_lib.context(dev), C.c_void_p(det.data_ptr()), C.c_void_p(cnt.data_ptr()), B, max_det,
                                         C.c_void_p(gt.data_ptr()), C.c_void_p(gt_cnt.data_ptr()), gt.shape[1], self.size_threshold,
                                         self.small_iou, self.match_iou, C.c_void_p(self.counters.data_ptr()),
                                         C.c_void_p(scores.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
              "uyd_eval_update")
        self._scores.append(scores)
        if self.nc is not None:
            keys = torch.empty(B * max_det, dtype=torch.int64, device=det.device)
            masks = torch.empty(B * max_det, dtype=torch.int16, device=det.device)
            thr = (C.c_float * len(MAP_IOUV))(*MAP_IOUV.tolist())
            check(_lib.lib().uyd_eval_match(_lib.context(dev), C.c_void_p(det.data_ptr()), C.c_void_p(cnt.data_ptr()), B, max_det,
                                            C.c_void_p(gt.data_ptr()), C.c_void_p(gt_cnt.data_ptr()), gt.shape[1], self.nc, thr,
                                            len(MAP_IOUV), C.c_void_p(masks.data_ptr()), C.c_void_p(keys.data_ptr()),
                                            C.c_void_p(self._n_labels.data_ptr()), C.c_void_p(self._dropped.data_ptr()),
                                            C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
                  "uyd_eval_match")
            self._keys.append(keys)
            self._masks.append(masks)

    def reduce(self, group=None) -> None:
        """Sums the counters and concatenates the scores over the ranks (when every rank evaluated its own shard).
        With ``nc`` set it also sums the label counts and gathers the mAP records in rank order, so with contiguous
        ``dp.shard_bounds`` shards equal confidences rank as in one process."""
        import torch.distributed as dist

        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return
        dist.all_reduce(self.counters, group=group)
        s = torch.cat([t.flatten() for t in self._scores]) if self._scores else torch.empty(0, device=self.device)
        self._scores = [_all_gather_padded(s, -1.0, group)]
        if self.nc is not None:
            dist.all_reduce(self._n_labels, group=group)
            dist.all_reduce(self._dropped, group=group)
            keys = torch.cat(self._keys) if self._keys else torch.empty(0, dtype=torch.int64, device=self.device)
            masks = torch.cat(self._masks) if self._masks else torch.empty(0, dtype=torch.int16, device=self.device)
            self._keys = [_all_gather_padded(keys, _PAD_KEY, group)]
            self._masks = [_all_gather_padded(masks.int(), 0, group).short()]   # int32 on the wire: gloo has no int16

    @torch.no_grad()
    def map_metrics(self) -> dict:
        """The box metrics of Ultralytics ``model.val`` over everything ``update`` saw: the results dict (keys
        metrics/precision(B), metrics/recall(B), metrics/mAP50(B), metrics/mAP50-95(B), fitness) plus the per-class
        ``ap50``, ``ap`` (mean over IoU 0.5:0.95) and ``ap_class_index`` arrays, classes with labels only.
        One stable device sort of the records, one ap_per_class launch, then numpy on [classes, 1000] arrays."""
        return map_results(*self._ap_per_class())

    def _ap_per_class(self):
        """(ap [nc, 10], p_curve [nc, 1000], r_curve [nc, 1000]) as fp64 numpy, or Nones without any record, and
        the label counts [nc]."""
        if self.nc is None:
            raise RuntimeError("map_metrics needs DetectionEvaluator(nc=...)")
        dropped = int(self._dropped)
        if dropped:
            raise ValueError(f"{dropped} ground truths / detections had a class outside [0, {self.nc}) or a NaN confidence")
        T = len(MAP_IOUV)
        n_labels = self._n_labels.cpu().numpy()
        keys = torch.cat(self._keys) if self._keys else torch.empty(0, dtype=torch.int64, device=self.device)
        ap = p_curve = r_curve = None
        if keys.numel():
            masks = torch.cat(self._masks)
            # The one step left to torch: a stable device sort of all records by (class, confidence descending); the
            # stable order keeps (update call, image, row) among equal keys.  libuyd ships no radix sort of its own.
            skeys, order = torch.sort(keys, stable=True)
            ap = torch.empty(self.nc, T, dtype=torch.float64, device=self.device)
            p_curve = torch.empty(self.nc, 1000, dtype=torch.float64, device=self.device)
            r_curve = torch.empty(self.nc, 1000, dtype=torch.float64, device=self.device)
            dev = self.device.index if self.device.index is not None else torch.cuda.current_device()
            check(_lib.lib().uyd_eval_ap(_lib.context(dev), C.c_void_p(skeys.data_ptr()), C.c_void_p(order.data_ptr()),
                                         C.c_void_p(masks.data_ptr()), keys.numel(), C.c_void_p(self._n_labels.data_ptr()),
                                         self.nc, T, C.c_void_p(ap.data_ptr()), C.c_void_p(p_curve.data_ptr()),
                                         C.c_void_p(r_curve.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
                  "uyd_eval_ap")
            ap, p_curve, r_curve = ap.cpu().numpy(), p_curve.cpu().numpy(), r_curve.cpu().numpy()
        return ap, p_curve, r_curve, n_labels

    def small_object_metrics(self) -> dict:
        """trainer.py:267-285 (the 1e-7 guards included)."""
        tp, fp, fn = (int(v) for v in self.counters.tolist())
        precision = tp / (tp + fp + 1e-7)
        recall = tp / (tp + fn + 1e-7)
        f1 = 2 * (precision * recall) / (precision + recall + 1e-7)
        return {"metrics/small_precision": precision, "metrics/small_recall": recall, "metrics/small_f1": f1,
                "tp": tp, "fp": fp, "fn": fn}

    def nonconformity_scores(self) -> torch.Tensor:
        if not self._scores:
            return torch.empty(0, device=self.device)
        s = torch.cat([t.flatten() for t in self._scores])
        return s[s >= 0]

    def conformal(self, alpha: float = 0.10) -> dict:
        """train.py:491-512: q_hat = the (1 - alpha) quantile (linear interpolation, numpy's default) of 1 - IoU."""
        s = self.nonconformity_scores().double()
        if s.numel() == 0:
            raise ValueError("Conformal Prediction Calibration failed: No matched predictions found.")
        srt, _ = torch.sort(s)
        pos = (srt.numel() - 1) * (1 - alpha)
        lo = int(pos // 1)
        hi = min(lo + 1, srt.numel() - 1)
        q_hat = float(srt[lo] + (srt[hi] - srt[lo]) * (pos - lo))
        return {"alpha": alpha, "coverage_target": 1 - alpha, "q_hat": q_hat, "dilation_factor": q_hat,
                "num_calibration_samples": int(srt.numel()), "mean_nonconformity": float(s.mean()),
                "std_nonconformity": float(s.std(unbiased=False))}


def _all_gather_padded(x: torch.Tensor, pad_value, group) -> torch.Tensor:
    """Concatenation in rank order of every rank's 1-D ``x``, each padded to the longest with ``pad_value``."""
    import torch.distributed as dist

    n = torch.tensor([x.numel()], device=x.device)
    sizes = [torch.zeros_like(n) for _ in range(dist.get_world_size(group))]
    dist.all_gather(sizes, n, group=group)
    m = int(max(int(v) for v in sizes))
    pad = torch.full((m,), pad_value, dtype=x.dtype, device=x.device)
    pad[: x.numel()] = x
    out = [torch.empty_like(pad) for _ in sizes]
    dist.all_gather(out, pad, group=group)
    return torch.cat(out)


def _smooth(y: np.ndarray, f: float = 0.05) -> np.ndarray:
    """Ultralytics utils.metrics.smooth: box filter of odd width round(len * 2f) // 2 + 1, edges padded."""
    nf = round(len(y) * f * 2) // 2 + 1
    p = np.ones(nf // 2)
    yp = np.concatenate((p * y[0], y, p * y[-1]), 0)
    return np.convolve(yp, np.ones(nf) / nf, mode="valid")


def map_results(ap, p_curve, r_curve, n_labels, eps: float = 1e-16) -> dict:
    """The host tail of Ultralytics ap_per_class and DetMetrics.results_dict over the per-class outputs of
    ``uyd_eval_ap`` (ap [nc, 10], p_curve / r_curve [nc, 1000] fp64, n_labels [nc]): keep the classes with labels,
    F1 = 2pr / (p + r + eps), the argmax of its smoothed class mean picks one confidence for P and R.  Like
    DetectionValidator.get_stats, when no prediction is a TP at any threshold (then every ap is 0; any TP makes its
    class's ap positive) nothing is reported and every metric is 0."""
    sel = np.flatnonzero(np.asarray(n_labels) > 0)
    if ap is None or not (ap[sel] > 0).any():
        p = r = np.zeros(0)
        all_ap = np.zeros((0, len(MAP_IOUV)))
        sel = np.zeros(0, dtype=int)
    else:
        all_ap, pc, rc = ap[sel], p_curve[sel], r_curve[sel]
        f1 = 2 * pc * rc / (pc + rc + eps)
        i = _smooth(f1.mean(0), 0.1).argmax()
        p, r = pc[:, i], rc[:, i]
    mean = [p.mean() if len(p) else 0.0, r.mean() if len(r) else 0.0, all_ap[:, 0].mean() if len(all_ap) else 0.0,
            all_ap.mean() if len(all_ap) else 0.0]
    fitness = (np.nan_to_num(np.array(mean)) * [0.0, 0.0, 0.1, 0.9]).sum()
    out = dict(zip(MAP_KEYS + ("fitness",), mean + [fitness]))
    out.update(ap50=all_ap[:, 0].copy(), ap=all_ap.mean(1), ap_class_index=sel.astype(int))
    return out


class SmallObjectMetric:
    """Drop-in for ``data_loader.SmallObjectMetric`` (data_loader.py:249-414): same constructor, ``reset`` /
    ``update(predictions, ground_truths)`` / ``compute``, same keys; the matching runs on the GPU, one CTA per
    image (csrc/evalmatch.cu ``small_object_metric_kernel``).  ``update`` takes the reference's lists
    (``[N,6]`` rows x_c,y_c,w,h,conf,cls and ``[G,5]`` rows cls,x_c,y_c,w,h, normalised) or already padded device
    tensors through ``update_batched``; ``from_xyxy_pixels`` converts ``predict`` rows."""

    def __init__(self, size_threshold: int = 15, iou_threshold: float = 0.5, image_size: int = 640, device=None) -> None:
        self.size_threshold, self.iou_threshold, self.image_size = size_threshold, iou_threshold, image_size
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.reset()

    def reset(self) -> None:
        self._counters = torch.zeros(3, dtype=torch.int64, device=self.device)

    @property
    def true_positives(self) -> int:
        return int(self._counters[0])

    @property
    def false_positives(self) -> int:
        return int(self._counters[1])

    @property
    def false_negatives(self) -> int:
        return int(self._counters[2])

    @staticmethod
    def from_xyxy_pixels(det: torch.Tensor, image_size: float) -> torch.Tensor:
        """[..., 6] rows (x1,y1,x2,y2,conf,cls) in pixels -> (x_c,y_c,w,h,conf,cls) normalised."""
        out = det.clone()
        out[..., 0] = (det[..., 0] + det[..., 2]) / 2 / image_size
        out[..., 1] = (det[..., 1] + det[..., 3]) / 2 / image_size
        out[..., 2] = (det[..., 2] - det[..., 0]) / image_size
        out[..., 3] = (det[..., 3] - det[..., 1]) / image_size
        return out

    @torch.no_grad()
    def update_batched(self, pred: torch.Tensor, cnt: torch.Tensor, gt: torch.Tensor, gt_cnt: torch.Tensor) -> None:
        """pred [B, max_det, 6] in confidence order, cnt [B] int32, gt [B, G, 5], gt_cnt [B] int32: device tensors."""
        assert pred.is_cuda and pred.dtype == torch.float32 and pred.is_contiguous() and pred.shape[2] == 6
        assert gt.is_cuda and gt.dtype == torch.float32 and gt.is_contiguous() and gt.shape[2] == 5
        assert cnt.dtype == torch.int32 and gt_cnt.dtype == torch.int32
        dev = pred.device.index if pred.device.index is not None else torch.cuda.current_device()
        check(_lib.lib().uyd_small_object_metric_update(
            _lib.context(dev), C.c_void_p(pred.data_ptr()), C.c_void_p(cnt.data_ptr()), pred.shape[0], pred.shape[1],
            C.c_void_p(gt.data_ptr()), C.c_void_p(gt_cnt.data_ptr()), gt.shape[1], float(self.size_threshold), float(self.iou_threshold),
            float(self.image_size), C.c_void_p(self._counters.data_ptr()), C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)),
            "uyd_small_object_metric_update")

    @torch.no_grad()
    def update(self, predictions, ground_truths) -> None:
        B = len(predictions)
        if B == 0:
            return
        md = max(1, max(int(p.shape[0]) if p.numel() else 0 for p in predictions))
        gm = max(1, max(int(g.shape[0]) if g.numel() else 0 for g in ground_truths))
        pred = torch.zeros(B, md, 6, device=self.device)
        gt = torch.zeros(B, gm, 5, device=self.device)
        cnt = torch.zeros(B, dtype=torch.int32, device=self.device)
        gcnt = torch.zeros(B, dtype=torch.int32, device=self.device)
        for i, (p, g) in enumerate(zip(predictions, ground_truths)):
            if p.numel():
                p = p.to(self.device, torch.float32)
                order = torch.sort(p[:, 4], descending=True, stable=True).indices   # data_loader.py:349-350
                pred[i, : p.shape[0]] = p[order]
                cnt[i] = p.shape[0]
            if g.numel():
                gt[i, : g.shape[0]] = g.to(self.device, torch.float32)
                gcnt[i] = g.shape[0]
        self.update_batched(pred, cnt, gt, gcnt)

    def compute(self) -> dict:
        tp, fp, fn = (int(v) for v in self._counters.tolist())
        precision = tp / (tp + fp) if (tp + fp) > 0 else 0.0
        recall = tp / (tp + fn) if (tp + fn) > 0 else 0.0
        f1 = 2 * (precision * recall) / (precision + recall) if (precision + recall) > 0 else 0.0
        return {"small_object_precision": precision, "small_object_recall": recall, "small_object_f1": f1,
                "small_object_tp": tp, "small_object_fp": fp, "small_object_fn": fn}
