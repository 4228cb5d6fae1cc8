"""Letterboxed camera frames (UYD_CAM_BGRA_LETTERBOX) in both networks' stems and uyd_letterbox_boxes, against the
path a user of the Ultralytics predictor takes by hand: the cv2-letterboxed frame (its numpy restatement,
oracle/letterbox.py, equal to cv2 byte for byte: tests/test_letterbox_host.py) as a tensor through forward /
predict_batched, then Ultralytics' scale_boxes + clip_boxes statements run with torch on the same device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import letterbox as lb

pytestmark = pytest.mark.gpu

UYD_E_ARG, UYD_E_UNSUPPORTED = 10001, 10003

# (frame width, frame height) -> (plan height, plan width)
PAIRS = [((1280, 720), (384, 640)), ((1280, 720), (640, 640)), ((1920, 1080), (384, 640)), ((320, 240), (480, 640)),
         ((641, 479), (480, 640)), ((1280, 725), (384, 640)), ((640, 384), (384, 640))]
CASES = [(3, f, p) for f, p in PAIRS] + [(64, (1280, 720), (384, 640))]
IDS = [f"b{b}-{f[0]}x{f[1]}-to-{p[0]}x{p[1]}" for b, f, p in CASES]


def _frames(B, w0, h0, seed):
    """Smooth content plus noise (uniform noise alone makes every anchor look alike) as BGRA bytes on the device."""
    g = torch.Generator().manual_seed(seed)
    low = torch.rand(B, 4, max(h0 // 32, 2), max(w0 // 32, 2), generator=g)
    img = torch.nn.functional.interpolate(low, size=(h0, w0), mode="bilinear", align_corners=False)
    img = 0.7 * img + 0.3 * torch.rand(B, 4, h0, w0, generator=g)
    return (img * 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous().cuda()


def _letterboxed(frames, H, W):
    """The cv2-letterboxed BGRA frames [B, H, W, 4] (device)."""
    host = frames.cpu().numpy()
    return torch.from_numpy(np.stack([lb.letterbox_bgra(f, H, W) for f in host])).cuda()


def _rgb_u8(bgra):
    return bgra[..., [2, 1, 0]].permute(0, 3, 1, 2).contiguous()


def _scale_boxes_torch(det, cnt, h0, w0, H, W):
    """Ultralytics ops.scale_boxes(img1_shape=(H, W), boxes, img0_shape=(h0, w0)) + clip_boxes, statement for statement,
    on each image's first count rows of a device copy."""
    out = det.clone()
    gain = min(H / h0, W / w0)
    pad = (round((W - w0 * gain) / 2 - 0.1), round((H - h0 * gain) / 2 - 0.1))
    for b, n in enumerate(cnt.tolist()):
        boxes = out[b, :n]
        boxes[..., 0] -= pad[0]
        boxes[..., 1] -= pad[1]
        boxes[..., 2] -= pad[0]
        boxes[..., 3] -= pad[1]
        boxes[..., :4] /= gain
        boxes[..., 0].clamp_(0, w0)
        boxes[..., 1].clamp_(0, h0)
        boxes[..., 2].clamp_(0, w0)
        boxes[..., 3].clamp_(0, h0)
    return out


def _yaml():
    import unina_yolo_dla_b200 as uyd

    return uyd.UninaYoloB200.from_yaml().init_synthetic(seed=0).cuda()


def _custom(bc=32):
    import unina_yolo_dla_b200 as uyd

    return uyd.UninaCustomB200(4, bc).init_synthetic(seed=1).cuda()


@pytest.mark.parametrize("B,frame,plan", CASES, ids=IDS)
def test_yaml_letterbox_equals_cv2_letterboxed_tensor(B, frame, plan):
    (w0, h0), (H, W) = frame, plan
    m = _yaml()
    frames = _frames(B, w0, h0, seed=w0 + h0 + B)
    x = _rgb_u8(_letterboxed(frames, H, W))
    assert torch.equal(m.forward_camera(frames, size=(H, W), letterbox=True), m(x, raw_heads=False))
    d0, c0 = m.predict_batched(x, conf=0.05, graph=False)
    assert int(c0.min()) > 0
    want = _scale_boxes_torch(d0, c0, h0, w0, H, W)
    d1, c1 = m.predict_camera(frames, size=(H, W), conf=0.05, letterbox=True)
    assert torch.equal(c1, c0) and torch.equal(d1, want)
    if (H, W) == lb.letterbox_shape(h0, w0):   # the default plan extent is the predictor's
        d2, c2 = m.predict_camera(frames, conf=0.05, letterbox=True)
        assert torch.equal(c2, c0) and torch.equal(d2, want)


def _conf_for(outs):
    best = torch.stack([c.flatten(1).max(1).values for c, _ in outs], 1).max(1).values
    return float(torch.sigmoid(best.min()) * 0.9)


@pytest.mark.parametrize("B,frame,plan", CASES, ids=IDS)
def test_custom_letterbox_equals_cv2_letterboxed_tensor(B, frame, plan):
    from unina_yolo_dla_b200 import preprocess

    (w0, h0), (H, W) = frame, plan
    m = _custom()
    frames = _frames(B, w0, h0, seed=w0 + h0 + B + 1)
    x = preprocess.bgra(_letterboxed(frames, H, W), preprocess.norm_params())   # ImageNet, uyd_preprocess_bgra_batch
    ref = m.forward(x)
    got = m.forward_camera(frames, size=(H, W), letterbox=True)
    for (ca, ra), (cb, rb) in zip(got, ref):
        assert torch.equal(ca, cb) and torch.equal(ra, rb)
    conf = _conf_for(ref)
    d0, c0 = m.predict_batched(x, conf=conf, graph=False)
    assert int(c0.min()) > 0
    want = _scale_boxes_torch(d0, c0, h0, w0, H, W)
    for graph in (False, True):
        if graph and B > m.GRAPH_MAX_BATCH:
            continue
        d1, c1 = m.predict_camera(frames, size=(H, W), conf=conf, graph=graph, letterbox=True)
        assert torch.equal(c1, c0) and torch.equal(d1, want), graph


def test_custom_letterbox_graph_replay_refreshes_frames():
    m = _custom()
    a, b = _frames(2, 1280, 720, seed=5), _frames(2, 1280, 720, seed=6)
    conf = _conf_for(m.forward_camera(a, letterbox=True))
    for frames in (a, b, a):
        d0, c0 = m.predict_camera(frames, conf=conf, graph=False, letterbox=True)
        d1, c1 = m.predict_camera(frames, conf=conf, graph=True, letterbox=True)
        assert torch.equal(c0, c1) and torch.equal(d0, d1)
    # the same frames without letterbox are a different graph (the cache key holds the mode)
    d2, _ = m.predict_camera(a[:, :384, :640].contiguous(), conf=conf, graph=True)
    d3, _ = m.predict_camera(a[:, :384, :640].contiguous(), conf=conf, graph=False)
    assert torch.equal(d2, d3)


def test_yaml_predict_stream_letterbox_equals_predict_camera():
    m = _yaml()
    batches = [_frames(n, 1280, 720, seed=30 + i).cpu().pin_memory() for i, n in enumerate((4, 4, 2))]
    got = [(d.clone(), c.clone()) for d, c in m.predict_stream(iter(batches), conf=0.05, camera="bgra", letterbox=True)]
    assert len(got) == 3
    for (d, c), b in zip(got, batches):
        wd, wc = m.predict_camera(b.cuda(), conf=0.05, letterbox=True)
        assert torch.equal(c, wc.cpu()) and torch.equal(d, wd.cpu())


# ---- uyd_letterbox_boxes alone ----

def _boxes_call(det, cnt, w0, h0, W, H, batch=None, max_det=None, det_ptr=None, cnt_ptr=None):
    from unina_yolo_dla_b200 import _lib

    code = _lib.lib().uyd_letterbox_boxes(None, det_ptr if det_ptr is not None else C.c_void_p(det.data_ptr()),
                                          cnt_ptr if cnt_ptr is not None else C.c_void_p(cnt.data_ptr()),
                                          det.shape[0] if batch is None else batch, det.shape[1] if max_det is None else max_det,
                                          w0, h0, W, H, None)
    torch.cuda.synchronize()
    return code


def test_box_kernel_hand_built_rows():
    """1280 x 720 in 384 x 640 (top pad 12, gain 0.5): a box crossing the top pad, one inside it (clamped to the top
    edge), one crossing the bottom pad and the right edge, an empty image, an image with count == max_det; rows past
    the count hold a sentinel that must survive."""
    from unina_yolo_dla_b200 import preprocess

    B, M = 4, 5
    det = torch.full((B, M, 6), -7.0, device="cuda")
    det[0, 0] = torch.tensor([10.0, 5.0, 100.0, 50.0, 0.9, 1.0])
    det[0, 1] = torch.tensor([200.0, 2.0, 260.0, 10.0, 0.8, 0.0])
    det[0, 2] = torch.tensor([600.5, 300.25, 650.0, 380.0, 0.7, 2.0])
    det[2] = torch.rand(M, 6, generator=torch.Generator().manual_seed(0)).cuda() * 700 - 30
    det[3, :2] = torch.tensor([[0.0, 12.0, 640.0, 372.0, 0.5, 3.0], [-3.0, 11.9, 641.0, 372.1, 0.4, 1.0]])
    cnt = torch.tensor([3, 0, M, 2], dtype=torch.int32, device="cuda")
    want = _scale_boxes_torch(det, cnt, 720, 1280, 384, 640)
    got = det.clone()
    preprocess.letterbox_boxes(got, cnt, 720, 1280, 384, 640)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert got[0, 1, :4].tolist() == [400.0, 0.0, 520.0, 0.0]       # inside the top pad: clamped to y = 0
    assert got[0, 2, :4].tolist() == [1201.0, 576.5, 1280.0, 720.0]   # clamped to the right / bottom edge
    assert torch.equal(got[0, 3:], det[0, 3:]) and torch.equal(got[1], det[1]) and torch.equal(got[3, 2:], det[3, 2:])
    assert torch.equal(got[3, 0, :4], torch.tensor([0.0, 0.0, 1280.0, 720.0], device="cuda"))
    np.testing.assert_array_equal(lb.scale_boxes(det[2].cpu().numpy(), 1280, 720, 640, 384), got[2].cpu().numpy())


@pytest.mark.parametrize("frame,plan", PAIRS, ids=[f"{f[0]}x{f[1]}-to-{p[0]}x{p[1]}" for f, p in PAIRS])
def test_box_kernel_random_rows(frame, plan):
    """Random rows over the whole plan and beyond it; 1920 x 1080 (gain 1/3) is where a true division and torch's
    multiply by the fp32 reciprocal differ in the last bit."""
    from unina_yolo_dla_b200 import preprocess

    (w0, h0), (H, W) = frame, plan
    g = torch.Generator().manual_seed(w0 + h0)
    B, M = 6, 300
    det = torch.zeros(B, M, 6)
    det[..., :4] = torch.rand(B, M, 4, generator=g) * torch.tensor([W + 40.0, H + 40.0, W + 40.0, H + 40.0]) - 20
    det[..., 4:] = torch.rand(B, M, 2, generator=g)
    det = det.cuda()
    cnt = torch.tensor([0, 1, 17, 299, 300, 150], dtype=torch.int32, device="cuda")
    for b, n in enumerate(cnt.tolist()):
        det[b, n:] = 0   # uyd_nms / uyd_nms_tlbr leave zeros past the count
    want = _scale_boxes_torch(det, cnt, h0, w0, H, W)
    got = det.clone()
    preprocess.letterbox_boxes(got, cnt, h0, w0, H, W)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    for b, n in enumerate(cnt.tolist()):
        assert not got[b, n:].any()
        np.testing.assert_array_equal(lb.scale_boxes(det[b, :n].cpu().numpy(), w0, h0, W, H), got[b, :n].cpu().numpy())


def test_box_kernel_rejects_bad_arguments_without_launch():
    det = torch.full((2, 4, 6), 3.0, device="cuda")
    cnt = torch.tensor([4, 4], dtype=torch.int32, device="cuda")
    snap = det.clone()
    assert _boxes_call(det, cnt, 1280, 720, 640, 384, det_ptr=C.c_void_p(0)) == UYD_E_ARG
    assert _boxes_call(det, cnt, 1280, 720, 640, 384, cnt_ptr=C.c_void_p(0)) == UYD_E_ARG
    assert _boxes_call(det, cnt, 1280, 720, 640, 384, det_ptr=C.c_void_p(det.data_ptr() + 2)) == UYD_E_ARG
    assert _boxes_call(det, cnt, 1280, 720, 640, 384, batch=0) == UYD_E_ARG
    assert _boxes_call(det, cnt, 1280, 720, 640, 384, max_det=0) == UYD_E_ARG
    assert _boxes_call(det, cnt, 0, 720, 640, 384) == UYD_E_ARG
    assert _boxes_call(det, cnt, 1280, 720, 640, -384) == UYD_E_ARG
    assert _boxes_call(det, cnt, 1, 4000, 640, 384) == UYD_E_ARG    # letterboxes to an empty frame
    assert torch.equal(det, snap)


# ---- rejections of the camera entry point ----

def _run_camera_code(p, frames, fmt, pitch=None, width=None, y=None):
    from unina_yolo_dla_b200 import _lib, preprocess

    f = _lib.CameraFrames()
    f.format = fmt
    f.width = width if width is not None else frames.shape[2]
    f.height = frames.shape[1]
    f.pitch = pitch if pitch is not None else frames.stride(1)
    f.frame_stride = frames.stride(0)
    f.data = frames.data_ptr()
    f.norm = preprocess.norm_params()
    code = _lib.lib().uyd_plan_run_camera(p.handle, C.byref(f), frames.shape[0], C.c_void_p(y.data_ptr()) if y is not None else None,
                                          None)
    torch.cuda.synchronize()
    return code


def _sentinel_plan(m, B, H, W):
    p = m.plan_for(torch.empty(B, 3, H, W, device="cuda"))
    stem = p.feature_slices["stem"]
    p.write(stem, torch.full((B, stem.c, H // 2, W // 2), 3.0, device="cuda"))
    return p, [stem, *p.heads], [p.read(s, B) for s in [stem, *p.heads]]


def _untouched(p, slices, snap, B):
    return all(torch.equal(p.read(s, B), v) for s, v in zip(slices, snap))


def test_camera_letterbox_rejected_without_launch():
    from unina_yolo_dla_b200 import _lib

    B, H, W = 2, 384, 640
    frames = _frames(B, 1280, 720, seed=9)
    m8 = _custom(8)
    p, sl, snap = _sentinel_plan(m8, B, H, W)
    assert _run_camera_code(p, frames, _lib.CAM_BGRA_LETTERBOX) == UYD_E_UNSUPPORTED   # base_channels 8: no camera loader
    assert _untouched(p, sl, snap, B)
    with pytest.raises(_lib.UydError):
        m8.forward_camera(frames, letterbox=True)
    with pytest.raises(_lib.UydError):
        m8.predict_camera(frames, graph=False, letterbox=True)
    m = _custom(32)
    p, sl, snap = _sentinel_plan(m, B, H, W)
    assert _run_camera_code(p, frames, _lib.CAM_BGRA_LETTERBOX, pitch=4 * 1280 + 2) == UYD_E_ARG   # pitch % 4 != 0
    assert _run_camera_code(p, frames, _lib.CAM_BGRA_LETTERBOX, pitch=4 * 1280 - 4) == UYD_E_ARG   # pitch < 4 width
    thin = torch.zeros(B, 4000, 1, 4, dtype=torch.uint8, device="cuda")
    assert _run_camera_code(p, thin, _lib.CAM_BGRA_LETTERBOX) == UYD_E_ARG   # 1 x 4000 letterboxes to an empty frame
    assert _untouched(p, sl, snap, B)
    y, uv = torch.zeros(B, 384, 640, dtype=torch.uint8, device="cuda"), torch.zeros(B, 192, 640, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError):
        m.forward_camera(y, uv=uv, letterbox=True)                                   # NV12 is not letterboxed
    with pytest.raises(ValueError):
        m.predict_camera(y, uv=uv, letterbox=True)
    my = _yaml()
    with pytest.raises(ValueError):
        my.predict_camera(y, uv=uv, letterbox=True)
    with pytest.raises(ValueError):
        next(my.predict_stream(iter([y.cpu()]), camera="nv12", letterbox=True))
    p = my.plan_for(torch.empty(B, 3, H, W, device="cuda"), fused=True)   # the YAML plan decodes into y
    assert p.fused
    y = torch.full((B, 4 + my.nc, my.num_anchors(H, W)), 5.0, device="cuda")
    assert _run_camera_code(p, frames, _lib.CAM_BGRA_LETTERBOX, pitch=4 * 1280 + 2, y=y) == UYD_E_ARG
    assert _run_camera_code(p, thin, _lib.CAM_BGRA_LETTERBOX, y=y) == UYD_E_ARG
    assert bool((y == 5.0).all())


# ---- non-square plans (the letterbox's rectangular extents) against the oracles ----

def _non_square(H, W, seed):
    from oracle import init as oi

    return oi.seeded_frames(2, 640, seed=seed)[:, :, :H, :W].contiguous()


@pytest.mark.parametrize("H,W", [(384, 640), (640, 384)])
def test_yaml_forward_non_square_matches_oracle(H, W):
    """The tolerance of tests/test_gpu_parity.py::test_full_forward_matches_oracle_bf16."""
    import unina_yolo_dla_b200 as uyd
    from oracle import yolo_graph as yg

    m = uyd.UninaYoloB200.from_yaml().init_synthetic(0)
    ref = yg.DetectionModel(yg.default_yaml_path())
    ref.load_state_dict(m.state_dict(), strict=True)
    ref.eval()
    m = m.cuda()
    x = _non_square(H, W, seed=5)
    with torch.no_grad():
        y_ref, raw_ref = ref(x)
    y, raws = m(x.cuda())
    torch.cuda.synchronize()
    rel = lambda a, b: float((a - b).abs().max() / b.abs().max().clamp_min(1e-12))
    for a, b in zip(raws, raw_ref):
        assert a.shape == b.shape
        assert rel(a.cpu()[:, :64], b[:, :64]) <= 1e-2 and rel(a.cpu()[:, 64:], b[:, 64:]) <= 1e-2
    assert rel(y.cpu()[:, :4], y_ref[:, :4]) <= 1e-2
    assert float((y.cpu()[:, 4:] - y_ref[:, 4:]).abs().max()) <= 1e-2


@pytest.mark.parametrize("bc", [8, 32])
@pytest.mark.parametrize("H,W", [(384, 640), (640, 384)])
def test_custom_forward_non_square_matches_oracle(bc, H, W):
    """The tolerance of tests/test_gpu_custom.py::test_custom_forward_640_matches_pinned_oracle (the stated one for this
    network at extents of 384 and more): regression <= 5e-3, class <= 2e-2 of range and <= 5e-3 rms."""
    import unina_yolo_dla_b200 as uyd
    from oracle import custom_graph as cg

    m = uyd.UninaCustomB200(4, bc).init_synthetic(seed=3)
    ref = cg.CustomNet(4, bc)
    ref.load_state_dict(m.state_dict(), strict=True)
    ref.eval()
    m = m.cuda()
    x = _non_square(H, W, seed=11)
    with torch.no_grad():
        want = ref(x)
    got = m(x.cuda())
    torch.cuda.synchronize()
    worst = {"cls": 0.0, "reg": 0.0, "cls_rms": 0.0}
    for pair_g, pair_w in zip(got, want):
        for name, g, w in zip(("cls", "reg"), pair_g, pair_w):
            assert g.shape == w.shape
            d = (g.cpu() - w).abs()
            rng = float(w.abs().max())
            worst[name] = max(worst[name], float(d.max()) / rng)
            if name == "cls":
                worst["cls_rms"] = max(worst["cls_rms"], float(d.pow(2).mean().sqrt()) / rng)
    print(f"model.py bc{bc} {H}x{W}: class {worst['cls']:.3e} (rms {worst['cls_rms']:.3e}), regression {worst['reg']:.3e}")
    assert worst["reg"] <= 5e-3 and worst["cls"] <= 2e-2 and worst["cls_rms"] <= 5e-3
