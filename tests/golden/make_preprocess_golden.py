"""Generates tests/golden/preprocess_ref.npz: the camera pre-processing output that tests/test_gpu_preprocess.py
compares with where the reference's own kernels (oracle/_ref/libref_preprocess.so) are not built.

Run on a GPU from the repo root:  python tests/golden/make_preprocess_golden.py [OUT]

Where that library is present, the stored values are its output.  The committed file was made without it, from this
project's kernels (unina-yolo-dla_b200/csrc/preprocess.cu) on a B200.  Those kernels are unchanged since
profiles/r03_pytest_gpu.log, the last suite run with the reference kernels present, in which every test of
tests/test_gpu_preprocess.py passed: our output equalled the reference's bit for bit for BGRA and within 1e-6 for
the bilinear resize and NV12, so the file holds the reference's output to that precision.

Per case (the seeded inputs of the tests): the sha256 of the whole fp32 output, and the output itself, whole up to
65536 elements, else a seeded sample of 4096 elements (stored_sample_index).
"""
from __future__ import annotations

import hashlib
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

import test_gpu_preprocess as t  # noqa: E402  (the tests' input generator, sampling rule and reference loader)
from unina_yolo_dla_b200 import preprocess as pre  # noqa: E402


def main(out: Path) -> None:
    ref = t.load_ref()
    norm, rnorm = pre.norm_params(), t.RefNorm(*t.IMAGENET)

    def bgra(x, size=None):
        if ref is None:
            return pre.bgra(x, norm, size=size)
        B, H, W = x.shape[:3]
        oh, ow = size or (H, W)
        y = torch.empty(B, 3, oh, ow, device="cuda")
        for b in range(B):
            if size is None:
                assert ref.preprocess_bgra(x[b].data_ptr(), y[b].data_ptr(), W, H, W * 4, rnorm, None) == 0
            else:
                assert ref.preprocess_bgra_resize(x[b].data_ptr(), y[b].data_ptr(), W, H, W * 4, ow, oh, rnorm, None) == 0
        return y

    def nv12(yp, uv):
        if ref is None:
            return pre.nv12(yp, uv, norm)
        H, W = yp.shape
        y = torch.empty(1, 3, H, W, device="cuda")
        assert ref.preprocess_nv12(yp.data_ptr(), uv.data_ptr(), y.data_ptr(), W, H, yp.stride(0), uv.stride(0), rnorm, None) == 0
        return y

    d = {}

    def put(name, y):
        torch.cuda.synchronize()
        flat = y.flatten().cpu()
        d[name] = flat[t.stored_sample_index(flat.numel())].numpy()
        d[name + "__sha256"] = np.array(hashlib.sha256(flat.numpy().tobytes()).hexdigest())

    for H, W in [(640, 640), (96, 132), (37, 50)]:
        put(f"bgra_{H}x{W}", bgra(t._frames(2, H, W, 1).cuda()))
    for (H, W), (oh, ow) in [((720, 1280), (640, 640)), ((480, 640), (640, 640)), ((100, 75), (64, 96))]:
        put(f"resize_{H}x{W}_{oh}x{ow}", bgra(t._frames(2, H, W, 2).cuda(), (oh, ow)))
    for H, W in [(64, 96), (50, 38)]:
        g = torch.Generator().manual_seed(3)
        yp = torch.randint(0, 256, (H, W), generator=g, dtype=torch.uint8).cuda()
        uv = torch.randint(0, 256, ((H + 1) // 2, W + (W % 2)), generator=g, dtype=torch.uint8).cuda()
        put(f"nv12_{H}x{W}", nv12(yp, uv))
    put("camera_bgra", bgra(t._frames(3, 320, 320, 7).cuda()))
    put("camera_resize", bgra(t._frames(2, 720, 1280, 8).cuda(), (640, 640)))
    g = torch.Generator().manual_seed(9)
    yp = torch.randint(0, 256, (2, 320, 320), generator=g, dtype=torch.uint8).cuda()
    uvp = torch.randint(0, 256, (2, 160, 320), generator=g, dtype=torch.uint8).cuda()
    put("camera_nv12", torch.cat([nv12(yp[b], uvp[b]) for b in range(2)]))
    np.savez_compressed(out, **d)
    print(out, "from the reference kernels" if ref is not None else "from this project's kernels",
          {k: v.shape for k, v in d.items() if not k.endswith("__sha256")})


if __name__ == "__main__":
    main(Path(sys.argv[1]) if len(sys.argv) > 1 else Path(__file__).resolve().parent / "preprocess_ref.npz")
