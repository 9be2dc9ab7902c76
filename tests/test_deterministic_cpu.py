"""CPU checks of the deterministic variants: the new entry points refuse bad arguments and short workspaces before any launch,
the workspace helpers reject bad sizes, and ops.deterministic() follows torch's flag."""
import ctypes as C

import torch

from pointnet12_b200 import _native as nv
from pointnet12_b200 import ops


def _buf(n=4096):
    raw = (C.c_ubyte * (n + 16))()
    base = C.cast(raw, C.c_void_p).value
    return raw, C.c_void_p((base + 15) // 16 * 16)


def test_version_and_workspace_helpers():
    lib = nv.lib()
    assert lib.pn_version() >= 403
    assert lib.pn_bn_stats_workspace_bytes(0, 8) == 0 and lib.pn_bn_stats_workspace_bytes(64, 0) == 0
    assert lib.pn_grad_weight_f32_workspace_bytes(0, 8, 8) == 0 and lib.pn_grad_weight_bf16x3_workspace_bytes(64, 0, 8) == 0
    assert lib.pn_csr_workspace_bytes(0, 8) == 0 and lib.pn_csr_workspace_bytes(8, 1 << 31) == 0
    assert lib.pn_csr_workspace_bytes(1000, 100) >= 4 * 4 * 1000
    assert lib.pn_cross_entropy_workspace_bytes(0) == 0 and lib.pn_chamfer_workspace_bytes(1, 0) == 0
    assert lib.pn_square_distance_bwd_det_workspace_bytes(1, 8, 0) == 0


def test_deterministic_abi_refuses_bad_arguments():
    lib = nv.lib()
    raw, p = _buf()
    # y, ldy, rows, C, sum, sumsq, workspace, bytes, stream
    assert lib.pn_bn_stats_det_f32(p, 8, 64, 8, p, p, None, 4096, None) == -1
    assert b"null workspace" in lib.pn_last_error_string()
    assert lib.pn_bn_stats_det_f32(p, 8, 64, 8, p, p, p, 8, None) == -1
    assert b"need" in lib.pn_last_error_string()
    q = C.c_void_p(p.value + 4)
    assert lib.pn_bn_stats_det_f32(p, 8, 64, 8, p, p, q, 4096, None) == -1
    assert b"aligned" in lib.pn_last_error_string()
    assert lib.pn_bn_stats_det_f32(p, 4, 64, 8, p, p, p, 4096, None) == -1         # ldy < C
    assert b"bad shape" in lib.pn_last_error_string()
    # bwd stats: rows not a multiple of K with argmax
    assert lib.pn_bn_bwd_stats_det_f32(p, 8, 10, 8, p, 8, p, 3, p, p, p, p, 1, p, p, p, 4096, None) == -1
    assert b"multiple of K" in lib.pn_last_error_string()
    assert lib.pn_bn_eval_bwd_det_f32(p, 8, 64, 8, p, 8, None, 1, p, p, p, p, 1, p, p, None, 8, None, None, p, 4096, None) == -1
    assert b"null pointer" in lib.pn_last_error_string()
    # weight gradients
    assert lib.pn_grad_weight_det_f32(p, 8, p, 8, 64, 8, 8, p, 8, None, p, 4, None) == -1
    assert b"need" in lib.pn_last_error_string()
    assert lib.pn_grad_weight_det_bf16x3(p, 8, p, 8, 64, 8, 8, None, 8, None, p, 1 << 20, None) == -1
    assert b"null pointer" in lib.pn_last_error_string()
    assert lib.pn_grad_weight_bn_det_bf16x3(p, 8, p, 8, None, p, 1, 64, 8, 8, p, 8, None, p, 1 << 20, None) == -1
    assert b"scale" in lib.pn_last_error_string()
    # inverse index
    assert lib.pn_csr_build(p, 16, 8, 8, 4, 1, p, 4096, p, p, None) == -1
    assert b"idx_bits" in lib.pn_last_error_string()
    assert lib.pn_csr_build(p, 64, 9, 8, 4, 1, p, 4096, p, p, None) == -1            # n_slots != B * slots_per_batch
    assert b"bad shape" in lib.pn_last_error_string()
    assert lib.pn_csr_build(p, 64, 8, 8, 4, 1, p, 16, p, p, None) == -1
    assert b"need" in lib.pn_last_error_string()
    assert lib.pn_csr_pull_f32(p, 4, 2, 4, 1, None, p, p, 8, p, None) == -1           # ld < col0 + D
    assert lib.pn_csr_pull_f32(p, 8, 0, 4, 0, None, p, p, 8, p, None) == -1           # div = 0
    assert lib.pn_group_bwd_det_f32(p, 8, 0, 4, None, p, 1, 8, p, None) == -1
    assert lib.pn_group_bwd_xyz_det_f32(p, 2, 0, p, p, p, 1, 8, 2, 4, p, None, None) == -1
    assert lib.pn_three_interpolate_bwd_det_f32(p, 8, 4, 4, p, p, p, 1, 8, 4, None, p, None) == -1
    assert lib.pn_three_interpolate_bwd_xyz_det_f32(p, 8, 0, 8, p, p, p, 24, 8, 1, p, 24, 3, 1, p, 6, 3, 1, 1, 8, 2, p, p, p,
                                                    None, p, p, p, None) == -1         # S < 3
    assert b"S >= 3" in lib.pn_last_error_string()
    # losses and function-level gradients
    assert lib.pn_cross_entropy_det_f32(p, 4, p, 64, 4, p, 8, p, None, 4, 1.0, None) == -1
    assert b"need" in lib.pn_last_error_string()
    assert lib.pn_chamfer_det_f32(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 9, None, p, None, p, 4096, None) == -1
    assert b"D <= 8" in lib.pn_last_error_string()
    assert lib.pn_chamfer_bwd_det_f32(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 3, p, p, 1.0, None, p, p, None, p, None) == -1
    assert b"null pointer" in lib.pn_last_error_string()
    assert lib.pn_square_distance_bwd_det_f32(p, 64, 8, p, 12, 3, 1, p, 24, 3, 1, 1, 8, 8, p, 8, p, p, None) == -1
    assert b"need" in lib.pn_last_error_string()
    assert lib.pn_square_distance_bwd_det_f32(p, 64, 8, p, 12, 3, 1, p, 24, 3, 1, 1, 8, 8, p, 4096, None, None, None) == -1
    del raw


def test_deterministic_follows_torch_flag():
    old, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    try:
        torch.use_deterministic_algorithms(False)
        assert not ops.deterministic()
        torch.use_deterministic_algorithms(True)
        assert ops.deterministic()
        torch.use_deterministic_algorithms(True, warn_only=True)
        assert ops.deterministic()
    finally:
        torch.use_deterministic_algorithms(old, warn_only=warn)
