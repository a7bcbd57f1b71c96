"""ctypes binding of libnerf_b200.so (the C ABI declared in include/nerf_b200.h).

There is no fallback: if the shared library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libnerf_b200.so")
MAX_D = 16
PREC_TC_FP16, PREC_FP32 = 0, 1

c_fp = C.c_void_p     # device pointers travel as integers


class NerfNetParams(C.Structure):
    _fields_ = [("D", C.c_int32), ("W", C.c_int32), ("input_ch", C.c_int32), ("input_ch_views", C.c_int32),
                ("skip", C.c_int32), ("use_viewdirs", C.c_int32), ("output_ch", C.c_int32), ("reserved", C.c_int32),
                ("pts_w", c_fp * MAX_D), ("pts_b", c_fp * MAX_D),
                ("feature_w", c_fp), ("feature_b", c_fp), ("alpha_w", c_fp), ("alpha_b", c_fp),
                ("views_w", c_fp), ("views_b", c_fp), ("rgb_w", c_fp), ("rgb_b", c_fp),
                ("output_w", c_fp), ("output_b", c_fp)]


class NerfNetGrads(C.Structure):
    _fields_ = [("pts_w", c_fp * MAX_D), ("pts_b", c_fp * MAX_D),
                ("feature_w", c_fp), ("feature_b", c_fp), ("alpha_w", c_fp), ("alpha_b", c_fp),
                ("views_w", c_fp), ("views_b", c_fp), ("rgb_w", c_fp), ("rgb_b", c_fp),
                ("output_w", c_fp), ("output_b", c_fp)]


class NerfCamera(C.Structure):
    _fields_ = [("H", C.c_int32), ("W", C.c_int32), ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float),
                ("cy", C.c_float), ("c2w", C.c_float * 12)]


class NerfRenderCfg(C.Structure):
    _fields_ = [("N_samples", C.c_int32), ("N_importance", C.c_int32), ("multires", C.c_int32),
                ("multires_views", C.c_int32), ("lindisp", C.c_int32), ("perturb", C.c_int32),
                ("white_bkgd", C.c_int32), ("ray_stride", C.c_int32), ("precision", C.c_int32),
                ("reserved", C.c_int32 * 3)]


class NerfPassOut(C.Structure):
    _fields_ = [("rgb_map", c_fp), ("disp_map", c_fp), ("acc_map", c_fp), ("depth_map", c_fp),
                ("weights", c_fp), ("raw", c_fp)]


class NerfTrainSave(C.Structure):
    _fields_ = [("act", c_fp), ("act_bytes", C.c_size_t), ("mask", c_fp), ("mask_bytes", C.c_size_t)]


class NerfRayGen(C.Structure):
    _fields_ = [("rays_o", c_fp), ("rays_d", c_fp), ("view_src", c_fp), ("cam", C.POINTER(NerfCamera)), ("pixel0", C.c_int64),
                ("ndc", C.c_int32), ("use_viewdirs", C.c_int32), ("near", C.c_float), ("far", C.c_float)]


class NerfBwdPass(C.Structure):
    _fields_ = [("z_vals", c_fp), ("noise", c_fp), ("S", C.c_int), ("net", C.POINTER(NerfNetParams)), ("packed", c_fp), ("raw", c_fp),
                ("save", C.POINTER(NerfTrainSave)), ("g_rgb", c_fp), ("grads", C.POINTER(NerfNetGrads))]


# name -> (restype, argtypes); mirrors include/nerf_b200.h one to one
SIGNATURES = {
    "nerf_b200_abi_version": (C.c_int, []),
    "nerf_b200_last_error": (C.c_char_p, []),
    "nerf_b200_launch_count": (C.c_int64, []),
    "nerf_b200_embed": (C.c_int, [c_fp, C.c_int64, C.c_int, c_fp, c_fp]),
    "nerf_b200_packed_bytes": (C.c_size_t, [C.POINTER(NerfNetParams)]),
    "nerf_b200_pack_weights": (C.c_int, [C.POINTER(NerfNetParams), c_fp, C.c_size_t, c_fp]),
    "nerf_b200_run_network": (C.c_int, [c_fp, c_fp, C.c_int64, C.c_int, C.POINTER(NerfNetParams), c_fp, C.c_int,
                                        C.c_int, C.c_int, c_fp, c_fp, C.c_size_t, c_fp]),
    "nerf_b200_raw2outputs": (C.c_int, [c_fp, c_fp, c_fp, C.c_int, c_fp, C.c_int64, C.c_int, C.c_int,
                                        C.POINTER(NerfPassOut), c_fp]),
    "nerf_b200_raw2outputs_bwd": (C.c_int, [c_fp, c_fp, c_fp, C.c_int, c_fp, C.c_int64, C.c_int, C.c_int, c_fp, c_fp, c_fp]),
    "nerf_b200_pack_rays": (C.c_int, [c_fp, c_fp, c_fp, C.POINTER(NerfCamera), C.c_int64, C.c_int64, C.c_int, C.c_float,
                                      C.c_float, C.c_int, c_fp, c_fp]),
    "nerf_b200_pack_rays_pixels": (C.c_int, [C.POINTER(NerfCamera), c_fp, C.c_int64, C.c_int, C.c_float, C.c_float, C.c_int, c_fp, c_fp]),
    "nerf_b200_to8b": (C.c_int, [c_fp, C.c_int64, c_fp, c_fp]),
    "nerf_b200_sample_pdf": (C.c_int, [c_fp, c_fp, c_fp, C.c_int64, C.c_int64, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_coarse_z": (C.c_int, [c_fp, C.c_int, c_fp, c_fp, C.c_int64, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_fine_z": (C.c_int, [c_fp, c_fp, c_fp, C.c_int64, C.c_int64, C.c_int, C.c_int, c_fp, c_fp, c_fp, c_fp]),
    "nerf_b200_march": (C.c_int, [c_fp, c_fp, c_fp, C.c_int64, C.c_int, C.POINTER(NerfNetParams), c_fp,
                                  C.POINTER(NerfRenderCfg), C.POINTER(NerfPassOut), c_fp, C.c_size_t, c_fp]),
    "nerf_b200_march_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int]),
    "nerf_b200_render_rays_fwd": (C.c_int, [c_fp, C.c_int64, C.POINTER(NerfRenderCfg),
                                            C.POINTER(NerfNetParams), c_fp, C.POINTER(NerfNetParams), c_fp,
                                            c_fp, c_fp, c_fp, c_fp, c_fp, c_fp,
                                            c_fp, C.POINTER(NerfPassOut), c_fp, c_fp, C.POINTER(NerfPassOut),
                                            c_fp, C.c_size_t, c_fp]),
    "nerf_b200_render_fwd": (C.c_int, [C.POINTER(NerfRayGen), c_fp, C.c_int64, C.POINTER(NerfRenderCfg),
                                       C.POINTER(NerfNetParams), c_fp, C.POINTER(NerfNetParams), c_fp,
                                       c_fp, c_fp, c_fp, c_fp, c_fp, c_fp,
                                       c_fp, C.POINTER(NerfPassOut), c_fp, c_fp, C.POINTER(NerfPassOut),
                                       c_fp, C.c_size_t, c_fp]),
    "nerf_b200_march_train": (C.c_int, [c_fp, c_fp, c_fp, C.c_int64, C.c_int, C.POINTER(NerfNetParams), c_fp,
                                        C.POINTER(NerfRenderCfg), C.POINTER(NerfPassOut), c_fp, C.c_size_t,
                                        C.POINTER(NerfTrainSave), c_fp]),
    "nerf_b200_train_record_bytes": (C.c_int, [C.c_int64, C.c_int, C.POINTER(NerfNetParams), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "nerf_b200_render_rays_fwd_train": (C.c_int, [c_fp, C.c_int64, C.POINTER(NerfRenderCfg),
                                                  C.POINTER(NerfNetParams), c_fp, C.POINTER(NerfNetParams), c_fp,
                                                  c_fp, c_fp, c_fp, c_fp, c_fp, c_fp,
                                                  c_fp, C.POINTER(NerfPassOut), c_fp, c_fp, C.POINTER(NerfPassOut),
                                                  c_fp, C.c_size_t, C.POINTER(NerfTrainSave), C.POINTER(NerfTrainSave), c_fp]),
    "nerf_b200_march_bwd_tc": (C.c_int, [c_fp, c_fp, c_fp, C.c_int64, C.c_int, C.POINTER(NerfNetParams), c_fp,
                                         C.POINTER(NerfRenderCfg), c_fp, C.POINTER(NerfTrainSave), c_fp,
                                         C.POINTER(NerfNetGrads), c_fp, C.c_size_t, c_fp]),
    "nerf_b200_march_bwd_tc_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.POINTER(NerfNetParams)]),
    "nerf_b200_march_bwd_tc_layout": (C.c_int, [C.c_int64, C.c_int, C.POINTER(NerfNetParams), C.POINTER(C.c_int64)]),
    "nerf_b200_render_rays_bwd_tc": (C.c_int, [c_fp, C.c_int64, C.POINTER(NerfRenderCfg), C.POINTER(NerfBwdPass), C.POINTER(NerfBwdPass),
                                               c_fp, C.c_size_t, c_fp]),
    "nerf_b200_render_rays_bwd_tc_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.POINTER(NerfNetParams), C.c_int, C.POINTER(NerfNetParams)]),
    "nerf_b200_march_bwd": (C.c_int, [c_fp, c_fp, c_fp, C.c_int64, C.c_int, C.POINTER(NerfNetParams), c_fp,
                                      C.POINTER(NerfRenderCfg), c_fp, C.POINTER(NerfNetGrads), c_fp, C.c_size_t, c_fp]),
    "nerf_b200_march_bwd_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int, C.POINTER(NerfNetParams)]),
    "nerf_b200_mse_seed": (C.c_int, [c_fp, c_fp, C.c_int64, C.c_float, c_fp, c_fp, c_fp]),
    "nerf_b200_adam_step": (C.c_int, [c_fp, c_fp, c_fp, c_fp, C.c_int64, c_fp, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                      C.c_float, C.c_float, c_fp]),
    "nerf_b200_timing_enable": (C.c_int, [C.c_int]),
    "nerf_b200_timing_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "nerf_b200_timing_read_kinds": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

# bring-up self-tests and micro-benchmarks: libnerf_b200_dev.so (include/nerf_b200_dev.h), never used by the product path
DEV_SIGNATURES = {
    "nerf_b200_dev_last_error": (C.c_char_p, []),
    "nerf_b200_debug_mma_rate": (C.c_int, [C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_debug_epi_rate": (C.c_int, [C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_debug_ldtm_rate": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_debug_issue_probe": (C.c_int, [C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_debug_l2_stream": (C.c_int, [c_fp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_debug_dram_stream": (C.c_int, [c_fp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, c_fp, c_fp]),
    "nerf_b200_debug_hbm_stream": (C.c_int, [c_fp, c_fp, C.c_size_t, C.c_int, C.c_int, c_fp]),
    "nerf_b200_selftest_gemm": (C.c_int, [c_fp, c_fp, C.c_int, C.c_int, c_fp, c_fp, C.c_size_t, c_fp]),
    "nerf_b200_selftest_gemm_tn": (C.c_int, [c_fp, c_fp, c_fp, C.c_int, C.c_int, c_fp]),
}

_lib = None
_dev = None
DEV_LIB_PATH = os.path.join(_HERE, "libnerf_b200_dev.so")


def load():
    """Load libnerf_b200.so; raises RuntimeError (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"nerf_b200: CUDA library not built ({LIB_PATH} missing). Run `python -c 'import __graft_entry__ as g; "
            "g.build()'` at the repo root. There is no CPU/PyTorch fallback for the hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)         # AttributeError -> the library does not match the header
        fn.restype, fn.argtypes = res, args
    if lib.nerf_b200_abi_version() != 1:
        raise RuntimeError("nerf_b200: ABI version mismatch between the Python host and libnerf_b200.so")
    _lib = lib
    return lib


def load_dev():
    """Load libnerf_b200_dev.so (self-tests / probes used by tests/ and tools/ only)."""
    global _dev
    if _dev is not None:
        return _dev
    if not os.path.isfile(DEV_LIB_PATH):
        raise RuntimeError(f"nerf_b200: dev library not built ({DEV_LIB_PATH} missing); run __graft_entry__.build()")
    lib = C.CDLL(DEV_LIB_PATH)
    for name, (res, args) in DEV_SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _dev = lib
    return lib


def check_dev(rc, what):
    if rc != 0:
        msg = load_dev().nerf_b200_dev_last_error()
        raise RuntimeError(f"nerf_b200_dev.{what} failed ({rc}): {msg.decode() if msg else '?'}")


def check(rc, what):
    if rc != 0:
        msg = load().nerf_b200_last_error()
        raise RuntimeError(f"nerf_b200.{what} failed ({rc}): {msg.decode() if msg else '?'}")


def launch_count():
    return int(load().nerf_b200_launch_count())
