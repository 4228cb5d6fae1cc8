"""Seeded detection / label scenes for the mAP tests (tests/test_map_host.py, tests/test_gpu_map.py)."""
import torch


def scene(B, seed, max_det=300, n_gt=20, nc=4, lattice=False, empty=True):
    """B images: ground truths [G, 5] (cls, x1, y1, x2, y2) and detections [N, 6] (x1, y1, x2, y2, conf, cls) in
    confidence order (stable), at most max_det.  Detections are jittered label copies (mostly the right class), second
    copies competing for the same label, and clutter.  ``lattice``: integer corners on a coarse grid and confidences
    in eighths, so equal IoUs and equal confidences are common.  ``empty``: image 1 has no detections, image 2 no
    labels (when B > 2)."""
    g = torch.Generator().manual_seed(seed)
    dets, gts = [], []
    for b in range(B):
        k = int(torch.randint(0, n_gt + 1, (1,), generator=g)) if b else n_gt
        if lattice:
            xy = torch.randint(0, 12, (k, 2), generator=g).float() * 4
            wh = torch.randint(2, 6, (k, 2), generator=g).float() * 4
        else:
            xy = torch.rand(k, 2, generator=g) * 580
            wh = torch.rand(k, 2, generator=g) * 60 + 4
        gt = torch.cat((torch.randint(0, nc, (k, 1), generator=g).float(), xy, xy + wh), 1)
        n_copy = min(k * 2, max_det)
        src = torch.randint(0, max(k, 1), (n_copy,), generator=g)
        if k:
            box = gt[src, 1:]
            box = box + (torch.randint(-1, 2, box.shape, generator=g).float() * 4 if lattice else torch.randn(box.shape, generator=g) * wh[src].repeat(1, 2) * 0.08)
            cls = torch.where(torch.rand(n_copy, generator=g) < 0.85, gt[src, 0], torch.randint(0, nc, (n_copy,), generator=g).float())
        else:
            box, cls = torch.zeros(0, 4), torch.zeros(0)
        m = int(torch.randint(0, max_det - len(box) + 1, (1,), generator=g))
        cxy = torch.rand(m, 2, generator=g) * 600
        cbox = torch.cat((cxy, cxy + torch.rand(m, 2, generator=g) * 40 + 2), 1)
        if lattice:
            cbox = (cbox / 4).round() * 4
        boxes = torch.cat((box, cbox))
        cls = torch.cat((cls, torch.randint(0, nc, (m,), generator=g).float()))
        conf = (torch.randint(1, 9, (len(boxes),), generator=g).float() / 8) if lattice else torch.rand(len(boxes), generator=g) * 0.999 + 0.001
        order = torch.argsort(conf, descending=True, stable=True)
        d = torch.cat((boxes, conf[:, None], cls[:, None]), 1)[order][:max_det]
        if empty and B > 2 and b == 1:
            d = d[:0]
        if empty and B > 2 and b == 2:
            gt = gt[:0]
        dets.append(d.contiguous())
        gts.append(gt.contiguous())
    return dets, gts


def pack(dets, gts, max_det, gmax=None):
    """Padded tensors det [B, max_det, 6], cnt [B] int32, gt [B, gmax, 5], gcnt [B] int32 (CPU)."""
    B = len(dets)
    gmax = gmax or max(1, max(len(x) for x in gts))
    det, gt = torch.zeros(B, max_det, 6), torch.zeros(B, gmax, 5)
    cnt, gcnt = torch.zeros(B, dtype=torch.int32), torch.zeros(B, dtype=torch.int32)
    for b, (d, t) in enumerate(zip(dets, gts)):
        det[b, : len(d)] = d
        gt[b, : len(t)] = t
        cnt[b], gcnt[b] = len(d), len(t)
    return det, cnt, gt, gcnt
