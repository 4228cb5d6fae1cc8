"""Generates tests/golden/*.npz by running the REAL reference in this container.

Run from the repo root:  python tests/golden/make_golden.py
Needs /root/reference (read-only mount).  The vectors are committed; the GPU box and CI
only read them.

* custom_bc{8,32}.npz   : outputs of the reference's own ``model.py`` ``UNINA_YOLO_DLA``
                          (imported from /root/reference/unina_yolo_dla) on a seeded
                          frame, with the seeded/calibrated weights of
                          ``oracle.init.build_custom`` (weights are reproduced from the
                          seed; their sha256 is stored to catch RNG drift).
* postprocess_hpp.npz   : outputs of the reference's ``postprocess.hpp`` (decode_head with
                          and without conformal dilation, nms) compiled from where it lies.
* tv_nms.npz            : ``torchvision.ops.nms`` results on the known-answer cases of
                          SURVEY.md 8c (ties, IoU == thr, cross-class, many survivors).
"""
from __future__ import annotations

import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, "/root/reference/unina_yolo_dla")

from oracle import init as oi  # noqa: E402
from oracle import postproc as pp  # noqa: E402

OUT = Path(__file__).resolve().parent
# custom_bc*.npz are computed with this many intra-op threads: oneDNN splits the reduction of an fp32 convolution by
# thread count, so the BN calibration pass and the forward reproduce bit for bit only at the same count.
GOLDEN_THREADS = 8


def custom(bc: int, size: int):
    import model as refmodel  # the real reference module

    torch.set_num_threads(GOLDEN_THREADS)
    net = oi.build_custom(seed=7, base_channels=bc, calib_batch=2, size=size, cls=refmodel.UNINA_YOLO_DLA)
    x = oi.seeded_frames(1, size, seed=11)
    with torch.no_grad():
        outs = net(x)
    d = {"sha256": np.array(oi.state_dict_sha256(net.state_dict())), "size": np.array(size), "bc": np.array(bc)}
    for lvl, (c, r) in zip((2, 3, 4), outs):
        d[f"p{lvl}_cls"] = c.numpy()
        d[f"p{lvl}_reg"] = r.numpy()
    np.savez_compressed(OUT / f"custom_bc{bc}.npz", **d)
    print("custom", bc, {k: v.shape for k, v in d.items() if k.startswith("p")})


def postprocess_hpp():
    assert pp.ref_lib() is not None, "reference header not compiled"
    rng = np.random.default_rng(3)
    w, h, nc, stride = 24, 20, 4, 8
    cls = rng.normal(-0.5, 1.5, (nc, h, w)).astype(np.float32)
    reg = rng.uniform(0.5, 4.0, (4, h, w)).astype(np.float32)
    d0 = pp.decode_tlbr(cls, reg, stride, 0.5, 0.0, use_ref=True)
    d1 = pp.decode_tlbr(cls, reg, stride, 0.3, 0.1, use_ref=True)
    # distinct confidences so the header's unstable std::sort is deterministic
    assert len(np.unique(d1["conf"])) == len(d1)
    k1 = pp.greedy_nms_hpp(d1, 0.45, use_ref=True)
    k0 = pp.greedy_nms_hpp(d0, 0.45, use_ref=True)
    np.savez_compressed(OUT / "postprocess_hpp.npz", cls=cls, reg=reg, stride=stride,
                        d0=d0, d1=d1, k0=k0, k1=k1)
    print("postprocess.hpp", len(d0), len(d1), len(k0), len(k1))


def tv_cases():
    """name -> (boxes[n,4], scores[n], thr)."""
    rng = np.random.default_rng(5)
    cases = {}
    # equal scores: ties -> lower index first
    cases["ties"] = (np.array([[0, 0, 10, 10], [1, 1, 11, 11], [0, 0, 10, 10], [50, 50, 60, 60]], np.float32),
                     np.array([0.9, 0.9, 0.9, 0.9], np.float32), 0.5)
    # IoU exactly == thr must be KEPT: two 2x1 boxes overlapping by half -> IoU 1/3; and 0.5
    cases["iou_eq_third"] = (np.array([[0, 0, 2, 1], [1, 0, 3, 1]], np.float32), np.array([0.8, 0.7], np.float32), 1.0 / 3.0)
    cases["iou_eq_half"] = (np.array([[0, 0, 2, 2], [0, 0, 2, 1]], np.float32), np.array([0.8, 0.7], np.float32), 0.5)
    # cross-class overlap via the +cls*7680 offset trick
    b = np.array([[10, 10, 50, 50], [12, 12, 52, 52], [10, 10, 50, 50]], np.float32)
    c = np.array([0, 0, 1], np.float32)[:, None] * 7680.0
    cases["cross_class"] = ((b + c).astype(np.float32), np.array([0.9, 0.8, 0.7], np.float32), 0.45)
    # dense random
    n = 3000
    xy = rng.uniform(0, 600, (n, 2)).astype(np.float32)
    wh = rng.uniform(4, 80, (n, 2)).astype(np.float32)
    cl = rng.integers(0, 4, n).astype(np.float32)[:, None] * np.float32(7680.0)
    bb = np.concatenate((xy, xy + wh), 1).astype(np.float32) + cl
    cases["dense3000"] = (bb.astype(np.float32), rng.uniform(0.01, 1, n).astype(np.float32), 0.7)
    # many survivors (> 300): a grid of disjoint boxes
    g = np.stack(np.meshgrid(np.arange(25), np.arange(25)), -1).reshape(-1, 2).astype(np.float32) * 20
    cases["disjoint625"] = (np.concatenate((g, g + 10), 1), rng.uniform(0.3, 1, 625).astype(np.float32), 0.45)
    # degenerate zero-area boxes (0/0 -> NaN -> never suppressed)
    cases["degenerate"] = (np.array([[5, 5, 5, 5], [5, 5, 5, 5], [0, 0, 10, 10]], np.float32),
                           np.array([0.9, 0.8, 0.7], np.float32), 0.1)
    cases["empty"] = (np.zeros((0, 4), np.float32), np.zeros((0,), np.float32), 0.5)
    return cases


def tv_nms():
    import torchvision

    d = {}
    for name, (b, s, thr) in tv_cases().items():
        keep = torchvision.ops.nms(torch.from_numpy(b), torch.from_numpy(s), float(thr)).numpy()
        d[f"{name}__boxes"], d[f"{name}__scores"], d[f"{name}__thr"], d[f"{name}__keep"] = b, s, np.float32(thr), keep
        print("tv_nms", name, len(b), "->", len(keep))
    np.savez_compressed(OUT / "tv_nms.npz", **d)


if __name__ == "__main__":
    custom(8, 64)
    custom(32, 64)
    postprocess_hpp()
    tv_nms()
