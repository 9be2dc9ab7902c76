"""ctypes binding of libpn12_b200.so (the C ABI declared in include/pn12_b200.h).

There is no CPU fallback and no alternative backend: if the library is missing or a call fails,
a RuntimeError is raised.  Pointers come from `tensor.data_ptr()`, the stream from
`torch.cuda.current_stream()`, so every call is asynchronous and CUDA-graph capturable.
"""
from __future__ import annotations

import ctypes as C
import os
import re

PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG, "libpn12_b200.so")
HEADER = os.path.join(os.path.dirname(PKG), "include", "pn12_b200.h")

_lib = None

vp, i64, i32, f32 = C.c_void_p, C.c_int64, C.c_int, C.c_float

MLP_MAX_LAYERS = 6


class MlpDesc(C.Structure):
    """pn_mlp_desc of include/pn12_b200.h."""
    _fields_ = [("nlayers", C.c_int), ("cin", C.c_int * MLP_MAX_LAYERS), ("cout", C.c_int * MLP_MAX_LAYERS),
                ("relu", C.c_int * MLP_MAX_LAYERS)]


_descp = C.POINTER(MlpDesc)


class LaunchOpts(C.Structure):
    """pn_launch_opts of include/pn12_b200.h: per-call launch options (all zeros = defaults)."""
    _fields_ = [("mlp_passes", C.c_int), ("mlp_engine", C.c_int), ("reserved_sms", C.c_int), ("fps_cluster", C.c_int),
                ("fps_threads", C.c_int), ("fps_exchange", C.c_int), ("tile_counter", C.c_void_p), ("mlp_debug", C.c_void_p)]


_optsp = C.POINTER(LaunchOpts)

# name -> argtypes, mirroring include/pn12_b200.h
_SIGNATURES = {
    "pn_version": [],
    "pn_device_check": [C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)],
    "pn_fps_f32": [vp, i64, i64, i64, i32, i32, i32, vp, vp, _optsp, vp],
    "pn_square_distance_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, vp, vp],
    "pn_square_distance_bwd_f32": [vp, i64, i64, vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, vp, vp, vp, vp],
    "pn_ball_query_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, f32, i32, vp, vp],
    "pn_ball_grid_build_f32": [vp, i64, i64, i64, i32, i32, f32, vp, C.c_size_t, vp],
    "pn_ball_query_grid_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, f32, i32, vp, C.c_size_t, i32, vp, vp,
                               vp],
    "pn_fps_progress_f32": [vp, i64, i64, i64, i32, i32, i32, vp, vp, vp, _optsp, vp],
    "pn_fps_sorted_f32": [vp, i64, i64, i64, vp, C.c_size_t, i32, i32, i32, vp, vp, vp, _optsp, vp],
    "pn_fps_launch_info": [i32, i32, i32, _optsp, C.POINTER(i32), C.POINTER(C.c_size_t)],
    "pn_ball_query_stream_f32": [vp, i64, i64, i64, vp, i32, i32, i32, i32, f32, i32, vp, C.c_size_t, i32, C.c_size_t, vp, vp,
                                 vp],
    "pn_index_points_f32": [vp, i64, i64, i64, i32, i32, i32, vp, i64, vp, vp],
    "pn_group_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, vp, i64, i64, i64, vp, i32, i32, i32, i32, i32, vp,
                     i64, vp],
    "pn_linear_f32": [vp, i64, i64, vp, i64, vp, i64, i32, i32, i64, i32, i32, vp, i64, i64, vp],
    "pn_group_max_f32": [vp, i64, i64, i32, i32, vp, i64, vp],
    "pn_three_nn_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, vp, vp, vp],
    "pn_three_nn_blocks_build_f32": [vp, i64, i64, i64, i32, i32, vp, C.c_size_t, vp],
    "pn_three_nn_blocks_f32": [vp, i64, i64, i64, vp, i64, i64, vp, C.c_size_t, i32, i32, i32, i32, vp, vp, vp],
    "pn_three_interpolate_f32": [vp, i64, i64, i64, i32, vp, i64, i64, i64, i32, i32, vp, vp, i32, i32, vp, i64, i64,
                                 vp],
    "pn_log_softmax_f32": [vp, i64, i64, i32, vp, i64, vp],
    "pn_argmax_labels_u8": [vp, i64, i64, i32, vp, vp],
    "pn_mlp_pack_bf16x3": [_descp, C.POINTER(vp), C.POINTER(vp), vp, vp],
    "pn_mlp_pack_t_bf16x3": [_descp, C.POINTER(vp), C.POINTER(vp), C.POINTER(i32), vp, vp],
    "pn_mlp_rows_bf16x3": [_descp, vp, vp, i64, i64, i32, vp, i64, _optsp, vp],
    "pn_sa_mlp_max_bf16x3": [_descp, vp, vp, i64, i64, i64, vp, i64, i64, i64, i32, vp, i64, i64, i64, vp, i32, i32, i32,
                             i32, i32, vp, i64, _optsp, vp],
    "pn_sa_mlp_bf16x3": [_descp, vp, vp, i64, i64, i64, vp, i64, i64, i64, i32, vp, i64, i64, i64, vp, i32, i32, i32,
                         i32, i32, i32, vp, i64, _optsp, vp],
    "pn_fp_mlp_bf16x3": [_descp, vp, vp, i64, i64, i64, i32, vp, i64, i64, i64, i32, i32, vp, vp, i32, vp, i64, i64, vp,
                         i64, i32, i32, i32, vp, i64, _optsp, vp],
    "pn_ball_grid_order": [vp, i32, C.POINTER(vp), C.POINTER(i64), C.POINTER(i64)],
    "pn_bn_stats_f32": [vp, i64, i64, i32, vp, vp, vp],
    "pn_bn_finalize_f32": [vp, vp, i64, i32, vp, vp, f32, f32, vp, vp, vp, vp, vp, vp, vp, vp],
    "pn_bn_act_f32": [vp, i64, i64, i32, vp, vp, i32, vp, i64, vp],
    "pn_bn_act_max_f32": [vp, i64, i64, i32, i32, vp, vp, i32, vp, i64, vp, vp],
    "pn_bn_bwd_stats_f32": [vp, i64, i64, i32, vp, i64, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp],
    "pn_bn_bwd_apply_f32": [vp, i64, i64, i32, vp, i64, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, i64, vp, vp, vp],
    "pn_bn_eval_bwd_f32": [vp, i64, i64, i32, vp, i64, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, i64, vp, vp, vp],
    "pn_grad_weight_f32": [vp, i64, vp, i64, i64, i32, i32, vp, i64, vp, vp],
    "pn_grad_weight_bf16x3": [vp, i64, vp, i64, i64, i32, i32, vp, i64, vp, vp],
    "pn_grad_weight_bn_bf16x3": [vp, i64, vp, i64, vp, vp, i32, i64, i32, i32, vp, i64, vp, vp],
    "pn_train_gemm_supported": [i32, i32],
    "pn_train_pack_many": [vp, i32, i32, i32, vp],
    "pn_train_gemm_bf16x3": [vp, i64, i64, i32, vp, vp, i32, vp, i32, vp, i32, vp, i64, vp, vp, vp, vp],
    "pn_train_gemm_bnbwd_bf16x3": [vp, i64, i64, i32, vp, i32, i32, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp],
    "pn_train_gemm_bneval_bf16x3": [vp, i64, i64, i32, vp, i32, i32, vp, i64, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp],
    "pn_transpose_f32": [vp, i32, i32, vp, vp],
    "pn_group_bwd_f32": [vp, i64, i32, i32, vp, i32, i32, i32, i32, vp, vp],
    "pn_three_interpolate_bwd_f32": [vp, i64, i32, i32, vp, vp, i32, i32, i32, vp, vp, vp],
    "pn_group_bwd_xyz_f32": [vp, i64, i32, vp, i32, i32, i32, i32, vp, vp, vp],
    "pn_three_interpolate_bwd_xyz_f32": [vp, i64, i32, i32, vp, vp, vp, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64, i64,
                                         i32, i32, i32, vp, vp, vp, vp, vp],
    "pn_dropout_f32": [vp, i64, i64, i32, f32, vp, vp, vp, vp, i64, vp],
    "pn_cross_entropy_f32": [vp, i64, vp, i64, i32, vp, vp, vp, i64, f32, vp],
    "pn_log_softmax_bwd_f32": [vp, i64, vp, i64, i64, i32, vp, i64, vp],
    "pn_adam_f32": [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i64, f32, vp],
    "pn_adam_dev_f32": [vp, vp, vp, vp, i64, vp, vp, f32, f32, f32, f32, f32, vp],
    "pn_seg_metrics_f32": [vp, i64, vp, i64, i32, vp, vp, vp],
    "pn_scan_filter_f32": [vp, vp, vp, i32, i64, vp, i32, i32, f32, f32, f32, f32, vp, vp, vp, C.c_size_t, vp],
    "pn_scan_sample_f32": [vp, vp, vp, i32, vp, i32, vp, vp, i32, vp, vp, f32, f32, vp, vp, vp, vp],
    "pn_chamfer_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, vp],
    "pn_chamfer_argmin_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, vp, vp],
    "pn_chamfer_bwd_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, f32, vp, vp, vp],
    "pn_class_merge_f32": [vp, i64, i64, i32, i32, vp, vp, vp, vp],
    "pn_seg_metrics_accumulate": [vp, i32, i64, vp, vp, vp, vp, vp],
    # deterministic variants (*_det_*): the default signature plus a workspace (pointer, bytes) or a prebuilt CSR
    "pn_bn_stats_det_f32": [vp, i64, i64, i32, vp, vp, vp, C.c_size_t, vp],
    "pn_bn_bwd_stats_det_f32": [vp, i64, i64, i32, vp, i64, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, C.c_size_t, vp],
    "pn_bn_eval_bwd_det_f32": [vp, i64, i64, i32, vp, i64, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp, i64, vp, vp, vp, C.c_size_t,
                               vp],
    "pn_grad_weight_det_f32": [vp, i64, vp, i64, i64, i32, i32, vp, i64, vp, vp, C.c_size_t, vp],
    "pn_grad_weight_det_bf16x3": [vp, i64, vp, i64, i64, i32, i32, vp, i64, vp, vp, C.c_size_t, vp],
    "pn_grad_weight_bn_det_bf16x3": [vp, i64, vp, i64, vp, vp, i32, i64, i32, i32, vp, i64, vp, vp, C.c_size_t, vp],
    "pn_csr_build": [vp, i32, i64, i64, i32, i32, vp, C.c_size_t, vp, vp, vp],
    "pn_csr_pull_f32": [vp, i64, i32, i32, i32, vp, vp, vp, i64, vp, vp],
    "pn_group_bwd_det_f32": [vp, i64, i32, i32, vp, vp, i32, i32, vp, vp],
    "pn_group_bwd_xyz_det_f32": [vp, i64, i32, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp],
    "pn_three_interpolate_bwd_det_f32": [vp, i64, i32, i32, vp, vp, vp, i32, i32, i32, vp, vp, vp],
    "pn_three_interpolate_bwd_xyz_det_f32": [vp, i64, i32, i32, vp, vp, vp, i64, i64, i64, vp, i64, i64, i64, vp, i64, i64, i64,
                                             i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp],
    "pn_cross_entropy_det_f32": [vp, i64, vp, i64, i32, vp, C.c_size_t, vp, vp, i64, f32, vp],
    "pn_chamfer_det_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, vp, vp, C.c_size_t, vp],
    "pn_chamfer_bwd_det_f32": [vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, i32, vp, vp, f32, vp, vp, vp, vp, vp, vp],
    "pn_square_distance_bwd_det_f32": [vp, i64, i64, vp, i64, i64, i64, vp, i64, i64, i64, i32, i32, i32, vp, C.c_size_t, vp, vp,
                                       vp],
}

# size_t helpers of the deterministic variants: name -> argtypes
_SIZE_HELPERS = {
    "pn_bn_stats_workspace_bytes": [i64, i32],
    "pn_grad_weight_f32_workspace_bytes": [i64, i32, i32],
    "pn_grad_weight_bf16x3_workspace_bytes": [i64, i32, i32],
    "pn_csr_workspace_bytes": [i64, i64],
    "pn_cross_entropy_workspace_bytes": [i64],
    "pn_chamfer_workspace_bytes": [i32, i32],
    "pn_square_distance_bwd_det_workspace_bytes": [i32, i32, i32],
}


def declared_symbols() -> list:
    """Every function name include/pn12_b200.h declares (used by the export test)."""
    with open(HEADER) as f:
        text = f.read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pn_[a-z0-9_]+)\s*\(", text)))


def lib():
    """Load the library once; fail loudly when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m pointnet12_b200.build` "
                "(nvcc, sm_100a). pointnet12_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        handle.pn_last_error_string.restype = C.c_char_p
        handle.pn_last_error_string.argtypes = []
        for name, argtypes in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = i32
        handle.pn_mlp_blob_bytes.argtypes = [_descp]
        handle.pn_mlp_blob_bytes.restype = C.c_size_t
        handle.pn_mlp_resident_groups.argtypes = [_descp]
        handle.pn_mlp_resident_groups.restype = C.c_int
        handle.pn_ball_grid_bytes.argtypes = [i32, i32]
        handle.pn_ball_grid_bytes.restype = C.c_size_t
        handle.pn_three_nn_blocks_bytes.argtypes = [i32, i32]
        handle.pn_three_nn_blocks_bytes.restype = C.c_size_t
        handle.pn_train_gemm_scratch_bytes.argtypes = [i32, i32]
        handle.pn_train_gemm_scratch_bytes.restype = C.c_size_t
        handle.pn_scan_workspace_bytes.argtypes = [i32, i64]
        handle.pn_scan_workspace_bytes.restype = C.c_size_t
        for name, argtypes in _SIZE_HELPERS.items():
            fn = getattr(handle, name)
            fn.argtypes = argtypes
            fn.restype = C.c_size_t
        _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().pn_last_error_string().decode("utf-8", "replace")
        kind = "CUDA error" if status > 0 else "argument error"
        raise RuntimeError(f"{what} failed ({kind} {status}): {msg}")


# ---- launch accounting (used by bench.py): how many of our kernels were launched, and optional CUDA-event
# timing of selected entry points on the launching stream.
launch_count = 0
_timed = {}          # name -> list of (start_event, stop_event, tag)


def time_entry_points(names=None):
    """Enable (names = iterable of entry points) or disable (None) CUDA-event timing; returns the old records."""
    global _timed
    old, _timed = _timed, ({n: [] for n in names} if names else {})
    return old


def call(name: str, *args, tag=None) -> None:
    global launch_count
    launch_count += 1
    rec = _timed.get(name)
    if rec is None:
        check(getattr(lib(), name)(*args), name)
        return
    import torch

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    check(getattr(lib(), name)(*args), name)
    b.record()
    rec.append((a, b, tag))
