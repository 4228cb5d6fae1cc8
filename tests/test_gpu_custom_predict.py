"""Batched TLBR decode + NMS of the model.py network (uyd_nms_tlbr, UninaCustomB200.predict_batched) against the
per-image composition it replaces (uyd_decode_tlbr per level + uyd_nms_detections) and the postprocess.hpp oracle.
Every comparison is byte for byte."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

STRIDES = (4, 8, 16)
UYD_E_ARG, UYD_E_UNSUPPORTED = 10001, 10003


def _model(bc, seed=1):
    import unina_yolo_dla_b200 as uyd

    return uyd.UninaCustomB200(4, bc).init_synthetic(seed=seed).cuda()


def _frames(batch, size, seed, dtype=torch.float32):
    from oracle import init as oi

    x = oi.seeded_frames(batch, size, seed=seed)
    if dtype == torch.uint8:
        x = (x * 255).to(torch.uint8)
    return x.cuda()


def _nhwc_heads(outs):
    """forward()'s [(cls, reg)] NCHW pairs -> the [B, H, W, nc + 4] fp32 head layout of the plan."""
    return [torch.cat((c, r), 1).permute(0, 2, 3, 1).contiguous() for c, r in outs]


def _nms_tlbr(heads, nc, conf, iou, q=0.0, strict=True, max_nms=0, max_det=1024, strides=STRIDES, batch=None, nl=None,
              det=None, cnt=None):
    """Direct uyd_nms_tlbr call; returns (code, det, cnt) after a synchronise."""
    from unina_yolo_dla_b200 import _lib

    B = heads[0].shape[0] if batch is None else batch
    n = len(heads)
    ptrs = (C.c_void_p * max(n, 1))(*[h.data_ptr() if h is not None else None for h in heads])
    gh = (C.c_int * max(n, 1))(*[h.shape[1] if h is not None else 1 for h in heads])
    gw = (C.c_int * max(n, 1))(*[h.shape[2] if h is not None else 1 for h in heads])
    st = (C.c_int * max(n, 1))(*strides[:max(n, 1)])
    if det is None:
        det = torch.empty(B, max(max_det, 1), 6, dtype=torch.float32, device="cuda")
    if cnt is None:
        cnt = torch.empty(B, dtype=torch.int32, device="cuda")
    code = _lib.lib().uyd_nms_tlbr(_lib.context(0), ptrs, gh, gw, st, n if nl is None else nl, B, nc, conf, q, int(strict), iou,
                                   max_nms, max_det, C.c_void_p(det.data_ptr()), C.c_void_p(cnt.data_ptr()), None)
    torch.cuda.synchronize()
    return code, det, cnt


def _decode_records(heads, b, nc, conf, q, strict):
    """uyd_decode_tlbr per level on image b (CHW planes), cell_base = level offset: (dets[n, 8], cell[n]) on the device."""
    from unina_yolo_dla_b200 import _lib

    cells = sum(h.shape[1] * h.shape[2] for h in heads)
    dets = torch.zeros(cells, 8, dtype=torch.float32, device="cuda")
    cell = torch.zeros(cells, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    base = 0
    for h, s in zip(heads, STRIDES):
        gh, gw = h.shape[1], h.shape[2]
        cls = h[b, :, :, :nc].permute(2, 0, 1).contiguous()
        reg = h[b, :, :, nc:].permute(2, 0, 1).contiguous()
        _lib.check(_lib.lib().uyd_decode_tlbr(_lib.context(0), C.c_void_p(cls.data_ptr()), C.c_void_p(reg.data_ptr()),
                                              C.c_void_p(dets.data_ptr()), C.c_void_p(cell.data_ptr()), C.c_void_p(cnt.data_ptr()),
                                              cells, gw, gh, s, nc, conf, q, int(strict), base, None), "uyd_decode_tlbr")
        base += gh * gw
    torch.cuda.synchronize()
    n = int(cnt.item())
    return dets[:n].contiguous(), cell[:n].contiguous()


def _record_nms(dets, cell, iou):
    """uyd_nms_detections on device records -> [k, 6] rows (x1,y1,x2,y2,conf,cls) as numpy float32."""
    from unina_yolo_dla_b200 import _lib

    L = _lib.lib()
    n = max(len(dets), 1)
    d = torch.zeros(n, 8, dtype=torch.float32, device="cuda")
    c = torch.zeros(n, dtype=torch.int32, device="cuda")
    d[:len(dets)] = dets
    c[:len(dets)] = cell
    cnt = torch.tensor([len(dets), 0], dtype=torch.int32, device="cuda")
    ws_bytes = int(L.uyd_nms_detections_workspace_bytes(n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    kept = torch.zeros(1024, 8, dtype=torch.float32, device="cuda")
    _lib.check(L.uyd_nms_detections(_lib.context(0), C.c_void_p(d.data_ptr()), C.c_void_p(c.data_ptr()), C.c_void_p(cnt.data_ptr()), n,
                                    iou, C.c_void_p(ws.data_ptr()), ws_bytes, C.c_void_p(kept.data_ptr()),
                                    C.c_void_p(cnt[1:].data_ptr()), None), "uyd_nms_detections")
    torch.cuda.synchronize()
    k = kept[: int(cnt[1])]
    return torch.cat((k[:, :5], k[:, 5:6].view(torch.int32).float()), 1).cpu().numpy()


def _oracle_rows(dets, cell, iou):
    """oracle.postproc.greedy_nms_hpp on records ordered by cell index (its stable sort then breaks confidence ties
    by cell, as the device key does), first 1024 -> [k, 6] rows."""
    from oracle import postproc as pp

    a = dets.cpu().numpy()[np.argsort(cell.cpu().numpy(), kind="stable")]
    rec = np.zeros(len(a), dtype=pp.DET_DTYPE)
    for i, f in enumerate(("x1", "y1", "x2", "y2", "conf")):
        rec[f] = a[:, i]
    rec["cls"] = a[:, 5].view(np.int32)
    k = pp.greedy_nms_hpp(rec, iou)[:1024]
    out = np.zeros((len(k), 6), np.float32)
    for i, f in enumerate(("x1", "y1", "x2", "y2", "conf")):
        out[:, i] = k[f]
    out[:, 5] = k["cls"].astype(np.float32)
    return out


def _assert_image(det, cnt, b, want):
    n = int(cnt[b])
    got = det[b].cpu().numpy()
    assert n == len(want), (b, n, len(want))
    assert got[:n].tobytes() == np.ascontiguousarray(want, np.float32).tobytes(), b
    assert not got[n:].any(), b  # every row past the count is zeros


@pytest.mark.parametrize("bc,size,batch,dtype,conf,q,strict", [
    (32, 640, 64, torch.float32, 0.5, 0.0, True),
    (8, 320, 3, torch.uint8, 0.5, 0.0, True),
    (8, 320, 4, torch.float32, 0.5, 0.1, True),
    (8, 320, 4, torch.float32, 0.55, 0.0, False),
], ids=["bc32_640_b64", "bc8_320_b3_u8", "conformal_q", "not_strict"])
def test_predict_batched_matches_per_image_path(bc, size, batch, dtype, conf, q, strict):
    m = _model(bc)
    x = _frames(batch, size, seed=21, dtype=dtype)
    det, cnt = m.predict_batched(x, conf=conf, iou=0.45, conformal_q=q, strict=strict, graph=False)
    want = m._predict_per_image(x, conf=conf, iou=0.45, conformal_q=q, strict=strict)
    assert det.shape == (batch, 1024, 6) and cnt.shape == (batch,) and cnt.dtype == torch.int32
    assert int(cnt.sum()) > 0
    for b in range(batch):
        _assert_image(det, cnt, b, want[b].cpu().numpy())
    # predict is rebuilt on predict_batched: same rows, same order, same bytes
    rows = m.predict(x, conf=conf, iou=0.45, conformal_q=q, strict=strict)
    assert len(rows) == batch
    for r, w in zip(rows, want):
        assert r.shape == w.shape and r.cpu().numpy().tobytes() == w.cpu().numpy().tobytes()


def test_dense_scene_every_cell_is_a_candidate():
    """conf 0 with >=: all 8 400 cells of a 320 x 320 frame enter the NMS (more than one 4096-key slab)."""
    m = _model(8)
    x = _frames(2, 320, seed=5)
    det, cnt = m.predict_batched(x, conf=0.0, iou=0.45, strict=False, graph=False)
    want = m._predict_per_image(x, conf=0.0, iou=0.45, strict=False)
    heads = _nhwc_heads(m(x))
    for b in range(2):
        _assert_image(det, cnt, b, want[b].cpu().numpy())
        dets, cell = _decode_records(heads, b, 4, 0.0, 0.0, False)
        assert len(dets) == 8400
        _assert_image(det, cnt, b, _oracle_rows(dets, cell, 0.45))


def _tie_heads(nc=3):
    """Three levels (8x8, 4x4, 2x2) of 3 images, nc = 3 (rows of 7 floats): class logits from four values, so many
    cells share a confidence; level 1 has no candidate in any image, image 2 none at all."""
    g = torch.Generator().manual_seed(3)
    heads = []
    for h in (8, 4, 2):
        logit = torch.tensor([-1.0, 0.25, 0.75, 2.0])[torch.randint(0, 4, (3, h, h, nc), generator=g)]
        reg = torch.randint(2, 9, (3, h, h, 4), generator=g).float() * 0.5   # distances 1 .. 4 cells in half steps
        t = torch.cat((logit, reg), -1)
        if h == 4:
            t[..., :nc] = -30.0
        t[2, ..., :nc] = -30.0
        heads.append(t.cuda().contiguous())
    return heads


def test_direct_heads_with_ties_and_empty_level_and_image():
    heads = _tie_heads()
    code, det, cnt = _nms_tlbr(heads, 3, 0.5, 0.45)
    assert code == 0
    assert int(cnt[2]) == 0 and not det[2].cpu().numpy().any()
    for b in range(3):
        dets, cell = _decode_records(heads, b, 3, 0.5, 0.0, True)
        assert not ((cell >= 64) & (cell < 80)).any()   # level 1 produced nothing
        if b < 2:
            assert len(dets) > 0 and len(torch.unique(dets[:, 4])) < len(dets)   # confidence ties exist
        _assert_image(det, cnt, b, _record_nms(dets, cell, 0.45))
        _assert_image(det, cnt, b, _oracle_rows(dets, cell, 0.45))


def test_max_det_prefix_and_max_nms_top_k():
    m = _model(8)
    x = _frames(2, 320, seed=13)
    heads = _nhwc_heads(m(x))
    _, full, fcnt = _nms_tlbr(heads, 4, 0.5, 0.45)
    assert int(fcnt.min()) > 7
    for md in (1, 7, 300):
        code, det, cnt = _nms_tlbr(heads, 4, 0.5, 0.45, max_det=md)
        assert code == 0
        for b in range(2):
            n = min(int(fcnt[b]), md)
            assert int(cnt[b]) == n
            assert det[b].cpu().numpy().tobytes() == np.concatenate(
                (full[b, :n].cpu().numpy(), np.zeros((md - n, 6), np.float32))).tobytes()
    for k in (1, 50, 1000, 5000):
        code, det, cnt = _nms_tlbr(heads, 4, 0.5, 0.45, max_nms=k)
        assert code == 0
        for b in range(2):
            dets, cell = _decode_records(heads, b, 4, 0.5, 0.0, True)
            conf = dets[:, 4].cpu().numpy()
            top = np.lexsort((cell.cpu().numpy(), -conf))[:k]   # confidence descending, then cell ascending
            sel = torch.from_numpy(top).cuda()
            _assert_image(det, cnt, b, _record_nms(dets[sel].contiguous(), cell[sel].contiguous(), 0.45))


def test_batch_independence_and_graph_replay():
    m = _model(8)
    x = _frames(4, 320, seed=17)
    det, cnt = m.predict_batched(x, graph=False)
    for b in range(4):
        d1, c1 = m.predict_batched(x[b:b + 1], graph=False)
        assert int(c1[0]) == int(cnt[b])
        assert d1[0].cpu().numpy().tobytes() == det[b].cpu().numpy().tobytes()
    for dtype in (torch.float32, torch.uint8):
        xa, xb = _frames(2, 320, seed=31, dtype=dtype), _frames(2, 320, seed=32, dtype=dtype)
        for xi in (xa, xb, xa):
            de, ce = m.predict_batched(xi, conf=0.55, iou=0.5, graph=False)
            dg, cg = m.predict_batched(xi, conf=0.55, iou=0.5, graph=True)
            assert torch.equal(ce, cg) and dg.cpu().numpy().tobytes() == de.cpu().numpy().tobytes()
    # batch 1 predict replays a graph by default and still equals the per-image path
    x1 = x[:1]
    rows = m.predict(x1)
    want = m._predict_per_image(x1)
    assert rows[0].cpu().numpy().tobytes() == want[0].cpu().numpy().tobytes()


@pytest.mark.parametrize("case", ["max_det_0", "max_det_1025", "no_level", "null_head"])
def test_bad_arguments_are_rejected_without_writing(case):
    heads = _tie_heads()
    det = torch.full((3, 1025, 6), 7.0, device="cuda")
    cnt = torch.full((3,), -5, dtype=torch.int32, device="cuda")
    kw = {"max_det_0": dict(max_det=0), "max_det_1025": dict(max_det=1025), "no_level": dict(nl=0), "null_head": {}}[case]
    if case == "null_head":
        heads[1] = None
    code, det, cnt = _nms_tlbr(heads, 3, 0.5, 0.45, batch=3, det=det, cnt=cnt, **kw)
    assert code == (UYD_E_UNSUPPORTED if case.startswith("max_det") else UYD_E_ARG)
    assert bool((det == 7.0).all()) and bool((cnt == -5).all())
