"""ctypes binding of libuyd.so (include/uyd.h).  No fallback: if the CUDA library is not
built or no sm_100 GPU is present, every use raises."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

HERE = Path(__file__).resolve().parent
LIB_PATH = HERE / "libuyd.so"

UYD_BF16, UYD_F32, UYD_S8, UYD_U8 = 0, 1, 2, 3
CHAIN_STORE, CHAIN_PW3, CHAIN_DFL = 0, 2, 3
IMPL_AUTO, IMPL_DIRECT, IMPL_TC = 0, 1, 2


class UydError(RuntimeError):
    pass


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in (
        "in_buf", "in_coff", "out_buf", "out_coff", "res_buf", "res_coff", "cin", "cout",
        "k", "stride", "depthwise", "relu", "impl", "pre_buf_p1")]


class ConvS8Desc(C.Structure):
    _fields_ = [("in_buf", C.c_int), ("in_coff", C.c_int), ("out_buf", C.c_int), ("out_coff", C.c_int), ("cin", C.c_int),
                ("cout", C.c_int), ("k", C.c_int), ("stride", C.c_int), ("relu", C.c_int), ("out_scale", C.c_float),
                ("impl", C.c_int), ("depthwise", C.c_int), ("res_buf", C.c_int), ("res_coff", C.c_int), ("out_round_bf16", C.c_int),
                ("pre_buf_p1", C.c_int)]


class C3kDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("in_buf", "in_coff", "out_buf", "out_coff", "c", "reserved")]


class ClsBranchDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("in_buf", "in_coff", "out_buf", "out_coff", "cin", "mid", "nc", "reserved")]


class ChainDesc(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("in_buf", "in_coff", "cin", "n1", "n2", "dw1", "relu2", "final_kind", "out_buf",
                                       "out_coff", "nc", "a_total", "a_off", "y_ch0", "no")] + [("stride_px", C.c_float)]


class NormParams(C.Structure):
    """Layout-identical to the reference NormParams (cuda_preprocess.h:38-45)."""
    _fields_ = [(n, C.c_float) for n in ("mean_r", "mean_g", "mean_b", "std_r", "std_g", "std_b")]


class CameraFrames(C.Structure):
    """uyd_camera_frames (include/uyd.h)."""
    _fields_ = [("format", C.c_int), ("width", C.c_int), ("height", C.c_int), ("pitch", C.c_int), ("uv_pitch", C.c_int),
                ("frame_stride", C.c_longlong), ("uv_frame_stride", C.c_longlong), ("data", C.c_void_p), ("uv", C.c_void_p),
                ("norm", NormParams)]


CAM_BGRA, CAM_NV12, CAM_BGRA_LETTERBOX = 1, 2, 3


class Detection(C.Structure):
    """Layout-identical to the reference GpuDetection (gpu_postprocess.h:27-33)."""
    _fields_ = [("x1", C.c_float), ("y1", C.c_float), ("x2", C.c_float), ("y2", C.c_float),
                ("confidence", C.c_float), ("class_id", C.c_int), ("valid", C.c_int), ("_pad", C.c_int)]


# name -> (restype, argtypes): every symbol include/uyd.h declares
SIGNATURES = {
    "uyd_version": (C.c_int, []),
    "uyd_last_error": (C.c_char_p, []),
    "uyd_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "uyd_destroy": (C.c_int, [C.c_void_p]),
    "uyd_sm_count": (C.c_int, [C.c_void_p]),
    "uyd_plan_create": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "uyd_plan_destroy": (C.c_int, [C.c_void_p]),
    "uyd_plan_add_buffer": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "uyd_plan_add_conv": (C.c_int, [C.c_void_p, C.POINTER(ConvDesc), C.c_void_p, C.c_void_p]),
    "uyd_plan_add_conv_s8": (C.c_int, [C.c_void_p, C.POINTER(ConvS8Desc), C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_plan_add_c3k": (C.c_int, [C.c_void_p, C.POINTER(C3kDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "uyd_plan_add_c3k_s8": (C.c_int, [C.c_void_p, C.POINTER(C3kDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                      C.POINTER(C.c_void_p), C.POINTER(C.c_float)]),
    "uyd_plan_add_cls_branch": (C.c_int, [C.c_void_p, C.POINTER(ClsBranchDesc), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]),
    "uyd_plan_add_quantize": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float]),
    "uyd_plan_slice_absmax": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "uyd_plan_slice_histogram": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p]),
    "uyd_plan_add_stem2": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_plan_add_stem2_pw": (C.c_int, [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 6),
    "uyd_plan_add_chain": (C.c_int, [C.c_void_p, C.POINTER(ChainDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "uyd_plan_run_decoded": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "uyd_plan_set_profile_output": (C.c_int, [C.c_void_p, C.c_void_p]),
    "uyd_plan_add_sppf_pool": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "uyd_plan_add_upsample2x": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "uyd_plan_set_heads": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int, C.c_int, C.c_int]),
    "uyd_plan_finalize": (C.c_int, [C.c_void_p]),
    "uyd_plan_bytes": (C.c_size_t, [C.c_void_p]),
    "uyd_plan_num_launches": (C.c_int, [C.c_void_p]),
    "uyd_plan_buffer_ptr": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "uyd_plan_run": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "uyd_plan_run_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "uyd_plan_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_float)]),
    "uyd_plan_set_timed_op": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "uyd_plan_timed_op_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "uyd_plan_op_info": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_size_t, C.POINTER(C.c_double),
                                   C.POINTER(C.c_double)]),
    "uyd_plan_run_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "uyd_plan_set_dfl_quant": (C.c_int, [C.c_void_p, C.c_float]),
    "uyd_plan_export_head_nchw": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "uyd_decode_dfl": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                 C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "uyd_decode_tlbr": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                  C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, C.c_void_p]),
    "uyd_nms_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "uyd_nms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_double, C.c_int, C.c_int,
                          C.c_float, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_nms_detections_workspace_bytes": (C.c_size_t, [C.c_int]),
    "uyd_nms_detections": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p,
                                     C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_nms_detections_inplace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_float, C.c_void_p, C.c_void_p]),
    "uyd_nms_tlbr": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int),
                               C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_float, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_compact_valid": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_norm_params_imagenet": (NormParams, []),
    "uyd_norm_params_unit": (NormParams, []),
    "uyd_preprocess_bgra_resize": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, NormParams, C.c_void_p]),
    "uyd_preprocess_bgra": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, NormParams, C.c_void_p]),
    "uyd_preprocess_nv12": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, NormParams, C.c_void_p]),
    "uyd_preprocess_bgra_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int, NormParams,
                                            C.c_void_p]),
    "uyd_preprocess_bgra_resize_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_int,
                                                   C.c_int, NormParams, C.c_void_p]),
    "uyd_eval_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_float,
                                  C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_small_object_metric_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                                 C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_void_p]),
    "uyd_eval_match": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                 C.POINTER(C.c_float), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_eval_ap": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_int,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "uyd_plan_run_camera": (C.c_int, [C.c_void_p, C.POINTER(CameraFrames), C.c_int, C.c_void_p, C.c_void_p]),
    "uyd_letterbox_geometry": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                         C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_double)]),
    "uyd_letterbox_boxes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p]),
    "uyd_host_alloc": (C.c_int, [C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
    "uyd_host_free": (C.c_int, [C.c_void_p]),
    "uyd_memcpy_d2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise UydError(
                f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                "(nvcc, sm_100a).  There is no CPU or PyTorch fallback for this path.")
        L = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(code: int, what: str = "") -> None:
    if code != 0:
        msg = lib().uyd_last_error().decode(errors="replace")
        raise UydError(f"{what or 'libuyd'} failed with code {code}: {msg}")


_ctx = {}


def context(device: int) -> C.c_void_p:
    """One handle per device (replaces the reference's global singleton, gpu_postprocess.cu:56)."""
    if device not in _ctx:
        h = C.c_void_p()
        check(lib().uyd_create(device, C.byref(h)), "uyd_create")
        _ctx[device] = h
    return _ctx[device]
