"""mAP50 / mAP50-95 on the device (uyd_eval_match, uyd_eval_ap, DetectionEvaluator(nc=...).map_metrics) against the
restated Ultralytics DetectionValidator.match_predictions / ap_per_class (oracle/mapref.py), byte for byte."""
import ctypes as C
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import map_scenes as S
from oracle import mapref as er

pytestmark = pytest.mark.gpu
E_ARG, E_UNSUPPORTED = 10001, 10003
PAD = torch.iinfo(torch.int64).max


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _match(det, cnt, gt, gcnt, nc, thr=None, gmax=None):
    from unina_yolo_dla_b200 import _lib

    thr = er.IOUV.tolist() if thr is None else list(thr)
    B, md = det.shape[:2] if det is not None else (cnt.shape[0], 16)   # det=None: a NULL pointer, shapes of the test scene
    masks = torch.full((B * md,), 0x5a5a, dtype=torch.int16, device="cuda")
    keys = torch.full((B * md,), -5, dtype=torch.int64, device="cuda")
    nl = torch.zeros(nc if nc > 0 else 1, dtype=torch.int64, device="cuda")
    dropped = torch.zeros(1, dtype=torch.int64, device="cuda")
    code = _lib.lib().uyd_eval_match(_lib.context(0), _ptr(det), _ptr(cnt), B, md, _ptr(gt), _ptr(gcnt),
                                     gt.shape[1] if gmax is None else gmax, nc, (C.c_float * max(1, len(thr)))(*thr), len(thr),
                                     _ptr(masks), _ptr(keys), _ptr(nl), _ptr(dropped), None)
    torch.cuda.synchronize()
    return code, masks.view(B, md), keys.view(B, md), nl, dropped


def _desc_bits(conf):
    u = conf.astype(np.float32).view(np.uint32).astype(np.int64)
    u = np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000)
    return ~u & 0xFFFFFFFF


@pytest.mark.parametrize("B,max_det,n_gt,lattice,seed", [(64, 300, 40, False, 1), (64, 300, 40, True, 2), (3, 1024, 1024, False, 3),
                                                         (4, 1024, 1024, True, 4)])
def test_tp_masks_and_keys_equal_match_predictions(B, max_det, n_gt, lattice, seed):
    dets, gts = S.scene(B, seed, max_det=max_det, n_gt=n_gt, lattice=lattice)
    det, cnt, gt, gcnt = S.pack(dets, gts, max_det, gmax=n_gt)
    code, masks, keys, nl, dropped = _match(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda(), 4)
    assert code == 0 and int(dropped) == 0
    masks, keys = masks.cpu().numpy().view(np.uint16), keys.cpu().numpy()
    n_tp = 0
    for b, (d, g) in enumerate(zip(dets, gts)):
        n = len(d)
        want = np.zeros((n, 10), bool)
        if n and len(g):
            want = er.match_predictions(d[:, 5], g[:, 0], er.box_iou(g[:, 1:], d[:, :4]))
        got = (masks[b, :n, None] >> np.arange(10)) & 1
        assert np.array_equal(got.astype(bool), want), b
        assert np.array_equal(keys[b, :n] >> 32, d[:, 5].numpy().astype(np.int64))
        assert np.array_equal(keys[b, :n] & 0xFFFFFFFF, _desc_bits(d[:, 4].numpy()))
        assert (keys[b, n:] == PAD).all() and (masks[b, n:] == 0).all()
        n_tp += int(want.sum())
    assert n_tp > 50
    want_nl = np.bincount(torch.cat(gts)[:, 0].long().numpy(), minlength=4)
    assert np.array_equal(nl.cpu().numpy(), want_nl)


def test_sixteen_thresholds_and_dropped_rows():
    thr = torch.linspace(0.3, 0.95, 16)
    dets, gts = S.scene(8, 5, max_det=300, n_gt=30, lattice=True)
    det, cnt, gt, gcnt = S.pack(dets, gts, 300)
    det[0, 0, 5], det[0, 1, 5], det[0, 2, 4] = 4.0, 1.5, float("nan")   # class == nc, non-integer class, NaN confidence
    gt[3, 0, 0] = -1.0
    code, masks, keys, nl, dropped = _match(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda(), 4, thr.tolist())
    assert code == 0 and int(dropped) == 4
    masks, keys = masks.cpu().numpy().view(np.uint16), keys.cpu().numpy()
    assert (keys[0, :3] == PAD).all() and (masks[0, :3] == 0).all()
    for b in range(1, 8):
        d, g = dets[b], gt[b, : int(gcnt[b])]
        if b == 3:
            g = g[1:]   # the dropped label takes part in nothing
        if not len(d):
            continue
        want = er.match_predictions(d[:, 5], g[:, 0], er.box_iou(g[:, 1:], d[:, :4]), thr) if len(g) else np.zeros((len(d), 16), bool)
        got = (masks[b, : len(d), None] >> np.arange(16)) & 1
        assert np.array_equal(got.astype(bool), want), b
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    ev = DetectionEvaluator(nc=4)
    ev.update(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda())
    with pytest.raises(ValueError):
        ev.map_metrics()


def _check(ev, dets, gts):
    ref = er.map_eval(dets, gts)
    raw = ref["raw"]
    ap, pc, rc, nl = ev._ap_per_class()
    idx = raw["ap_class_index"]
    assert np.array_equal(np.flatnonzero(nl > 0), idx) and np.array_equal(nl[idx], raw["nt"])
    assert ap[idx].tobytes() == raw["ap"].tobytes()
    assert pc[idx].tobytes() == raw["p_curve"].tobytes() and rc[idx].tobytes() == raw["r_curve"].tobytes()
    got = ev.map_metrics()
    for k in er.RESULT_KEYS + ("fitness",):
        assert got[k] == ref[k], (k, got[k], ref[k])
    for k in ("ap50", "ap", "ap_class_index"):
        assert np.array_equal(got[k], ref[k]), k
    return got


@pytest.mark.parametrize("lattice", [False, True])
def test_map_metrics_equal_restatement_over_several_updates(lattice):
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    ev, one = DetectionEvaluator(nc=6), DetectionEvaluator(nc=6)
    all_d, all_g = [], []
    for seed in range(3):
        dets, gts = S.scene(64, 10 + seed, max_det=300, n_gt=30, nc=5, lattice=lattice)
        det, cnt, gt, gcnt = S.pack(dets, gts, 300, gmax=30)
        ev.update(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda())
        all_d += dets
        all_g += gts
    got = _check(ev, all_d, all_g)
    assert got["metrics/mAP50(B)"] > 0.01 and len(got["ap_class_index"]) == 5
    det, cnt, gt, gcnt = S.pack(all_d, all_g, 300, gmax=30)
    one.update(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda())   # one concatenated update: the same records in order
    a, b = ev._ap_per_class(), one._ap_per_class()
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))
    assert one.map_metrics()["fitness"] == got["fitness"]


def test_large_class_spans_several_chunks():
    """One class with ~40 k records: the AP walk crosses chunk boundaries (4096 positions each)."""
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    dets, gts = S.scene(160, 21, max_det=300, n_gt=60, nc=1)
    ev = DetectionEvaluator(nc=1)
    for i in range(0, 160, 64):
        det, cnt, gt, gcnt = S.pack(dets[i:i + 64], gts[i:i + 64], 300, gmax=60)
        ev.update(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda())
    assert sum(len(d) for d in dets) > 4 * 4096
    _check(ev, dets, gts)


@pytest.mark.parametrize("net", ["yaml", "custom"])
def test_whole_path_on_predict_batched_rows(net):
    import unina_yolo_dla_b200 as uyd
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    m = (uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0) if net == "yaml" else uyd.UninaCustomB200(4, 32).init_synthetic(seed=1)).cuda()
    B = 8
    x = torch.rand(B, 3, 320, 320, generator=torch.Generator().manual_seed(5)).cuda()
    det, cnt = m.predict_batched(x, conf=0.001, iou=0.7)
    torch.cuda.synchronize()
    dets = [det[b, : int(cnt[b])].cpu() for b in range(B)]
    assert sum(len(d) for d in dets) > 100
    g = torch.Generator().manual_seed(6)
    gts = []
    for d in dets:   # labels near a sample of the detections (TPs at various IoUs) plus unmatched ones
        pick = d[torch.randperm(len(d), generator=g)[:12]]
        box = pick[:, :4] + torch.randn(len(pick), 4, generator=g) * 3
        cls = torch.where(torch.rand(len(pick), generator=g) < 0.8, pick[:, 5], torch.randint(0, 4, (len(pick),), generator=g).float())
        extra = torch.rand(4, 2, generator=g) * 280
        gts.append(torch.cat((torch.cat((cls[:, None], box), 1),
                              torch.cat((torch.randint(0, 4, (4, 1), generator=g).float(), extra, extra + 30), 1))))
    gt, gcnt = S.pack(dets, gts, det.shape[1])[2:]
    ev = DetectionEvaluator(nc=4)
    ev.update(det, cnt, gt.cuda(), gcnt.cuda())
    got = _check(ev, dets, gts)
    assert got["metrics/mAP50(B)"] > 0


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _reduce_worker(rank, world, port, out_path):
    from unina_yolo_dla_b200.dp import shard_bounds
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    dets, gts = S.scene(37, 31, max_det=300, n_gt=20, nc=3, lattice=True)
    b, e = shard_bounds(len(dets), world, rank)
    ev = DetectionEvaluator(nc=3)
    det, cnt, gt, gcnt = S.pack(dets[b:e], gts[b:e], 300, gmax=20)
    ev.update(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda())
    ev.reduce()
    if rank == 0:
        torch.save((ev._ap_per_class(), ev.map_metrics()), out_path)
    dist.destroy_process_group()


def test_reduce_over_two_gloo_ranks_equals_one_process(tmp_path):
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    out = tmp_path / "map.pt"
    mp.spawn(_reduce_worker, args=(2, _free_port(), str(out)), nprocs=2, join=True)
    arrays, got = torch.load(out, weights_only=False)
    dets, gts = S.scene(37, 31, max_det=300, n_gt=20, nc=3, lattice=True)
    ev = DetectionEvaluator(nc=3)
    det, cnt, gt, gcnt = S.pack(dets, gts, 300, gmax=20)
    ev.update(det.cuda(), cnt.cuda(), gt.cuda(), gcnt.cuda())
    assert all(x.tobytes() == y.tobytes() for x, y in zip(arrays, ev._ap_per_class()))
    want = _check(ev, dets, gts)
    for k in er.RESULT_KEYS + ("fitness",):
        assert got[k] == want[k]


def test_rejected_arguments_launch_nothing():
    from unina_yolo_dla_b200 import _lib

    dets, gts = S.scene(2, 9, max_det=16, n_gt=4, empty=False)
    det, cnt, gt, gcnt = (t.cuda() for t in S.pack(dets, gts, 16))

    def match(**kw):
        a = dict(det=det, cnt=cnt, gt=gt, gcnt=gcnt, nc=4, thr=None, gmax=None)
        a.update(kw)
        code, masks, keys, nl, dropped = _match(**a)
        assert (masks == 0x5a5a).all() and (keys == -5).all() and not nl.any() and not dropped.any()   # untouched
        return code

    assert match(det=None) == E_ARG and match(gcnt=None) == E_ARG and match(nc=0) == E_ARG
    assert match(thr=[]) == E_ARG and match(thr=[0.5] * 17) == E_ARG
    assert match(thr=[0.5, 0.0]) == E_ARG and match(thr=[math.nan]) == E_ARG and match(gmax=0) == E_ARG
    assert match(gmax=1025) == E_UNSUPPORTED and match(nc=(1 << 20) + 1) == E_UNSUPPORTED
    big = torch.zeros(1, 1025, 6, device="cuda")
    assert match(det=big, cnt=cnt[:1], gt=gt[:1], gcnt=gcnt[:1]) == E_UNSUPPORTED
    empty = torch.zeros(0, 16, 6, device="cuda")
    assert match(det=empty) == E_ARG

    keys = torch.zeros(8, dtype=torch.int64, device="cuda")
    order = torch.arange(8, device="cuda")
    masks = torch.zeros(8, dtype=torch.int16, device="cuda")
    nl = torch.ones(4, dtype=torch.int64, device="cuda")
    out = [torch.full((4, n), -7.0, dtype=torch.float64, device="cuda") for n in (10, 1000, 1000)]

    def ap(**kw):
        a = dict(k=keys, o=order, m=masks, n=8, nl=nl, nc=4, T=10)
        a.update(kw)
        code = _lib.lib().uyd_eval_ap(_lib.context(0), _ptr(a["k"]), _ptr(a["o"]), _ptr(a["m"]), a["n"], _ptr(a["nl"]), a["nc"], a["T"],
                                      *(_ptr(t) for t in out), None)
        torch.cuda.synchronize()
        assert all((t == -7.0).all() for t in out)
        return code

    assert ap(k=None) == E_ARG and ap(o=None) == E_ARG and ap(nl=None) == E_ARG and ap(n=0) == E_ARG
    assert ap(nc=0) == E_ARG and ap(T=0) == E_ARG and ap(T=17) == E_ARG and ap(nc=(1 << 20) + 1) == E_UNSUPPORTED


def test_without_nc_update_is_unchanged():
    from unina_yolo_dla_b200.evaluate import DetectionEvaluator

    dets, gts = S.scene(16, 12, max_det=300, n_gt=30)
    det, cnt, gt, gcnt = (t.cuda() for t in S.pack(dets, gts, 300))
    plain, withmap = DetectionEvaluator(), DetectionEvaluator(nc=4)
    plain.update(det, cnt, gt, gcnt)
    withmap.update(det, cnt, gt, gcnt)
    assert torch.equal(plain.counters, withmap.counters)
    assert torch.equal(plain._scores[0], withmap._scores[0])
    assert not hasattr(plain, "_keys")
    with pytest.raises(RuntimeError):
        plain.map_metrics()
    from oracle import evalref

    tot = np.asarray(evalref.small_object_counts(dets, gts, 15, 0.45))
    assert plain.counters.cpu().tolist() == tot.tolist()
