"""CPU checks of the function-level gradients: the new entry points refuse bad arguments before any launch, and the rule
that decides when the functions of model/pointnet_util.py and model/chamfer.py return a result with a grad_fn."""
import ctypes as C

import pytest
import torch

from pointnet12_b200 import _native as nv


def _ptr():
    buf = (C.c_float * 64)()
    return buf, C.cast(buf, C.c_void_p)


def test_square_distance_bwd_abi_refuses_bad_arguments():
    lib = nv.lib()
    buf, p = _ptr()
    f = lib.pn_square_distance_bwd_f32
    # g, gB, gN, src, aB, aN, aC, dst, bB, bN, bC, B, N, M, workspace, dsrc, ddst, stream
    assert f(None, 64, 8, p, 12, 3, 1, p, 24, 3, 1, 1, 8, 8, p, p, p, None) == -1
    assert b"null pointer" in lib.pn_last_error_string()
    assert f(p, 64, 8, p, 12, 3, 1, p, 24, 3, 1, 1, 8, 8, None, p, p, None) == -1            # no workspace
    assert f(p, 64, 8, p, 12, 3, 1, p, 24, 3, 1, 1, 8, 8, p, None, None, None) == -1         # neither side wanted
    assert b"null pointer" in lib.pn_last_error_string()
    for B, N, M in ((0, 8, 8), (1, 0, 8), (1, 8, 0)):
        assert f(p, 64, 8, p, 12, 3, 1, p, 24, 3, 1, B, N, M, p, p, p, None) == -1
        assert b"positive" in lib.pn_last_error_string()
    assert f(p, 64, 8, p, 12, 3, 1, p, 24, 3, 1, 65536, 8, 8, p, p, p, None) == -2           # B > 65535
    assert f(p, 64, -8, p, 12, 3, 1, p, 24, 3, 1, 1, 8, 8, p, p, p, None) == -1              # negative row stride
    assert b"negative stride" in lib.pn_last_error_string()
    q = C.c_void_p(C.cast(buf, C.c_void_p).value + 4 if C.cast(buf, C.c_void_p).value % 16 == 0 else
                   C.cast(buf, C.c_void_p).value + (16 - C.cast(buf, C.c_void_p).value % 16) + 4)
    assert f(p, 64, 8, p, 12, 3, 1, p, 24, 3, 1, 1, 8, 8, q, p, p, None) == -1               # workspace not 16-byte aligned
    assert b"aligned" in lib.pn_last_error_string()


def test_chamfer_argmin_and_bwd_abi_refuse_bad_arguments():
    lib = nv.lib()
    _buf, p = _ptr()
    fa = lib.pn_chamfer_argmin_f32
    # p1, aB, aN, aC, p2, bB, bN, bC, B, N, M, D, per_point, total, argmin, stream
    assert fa(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 3, None, p, None, None) == -1                # no argmin
    assert b"null pointer" in lib.pn_last_error_string()
    assert fa(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 9, None, p, p, None) == -1                   # D <= 8
    assert b"D <= 8" in lib.pn_last_error_string()
    assert fa(p, 9, 3, 1, p, 9, 3, 1, 1, 0, 3, 3, None, p, p, None) == -1
    fb = lib.pn_chamfer_bwd_f32
    # p1, aB, aN, aC, p2, bB, bN, bC, B, N, M, D, argmin, g_total, scale, dp1, dp2, stream
    assert fb(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 3, None, p, 1.0, p, p, None) == -1           # no argmin
    assert b"null pointer" in lib.pn_last_error_string()
    assert fb(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 3, p, None, 1.0, p, p, None) == -1           # no upstream gradient
    assert fb(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 3, p, p, 1.0, None, None, None) == -1        # no output
    assert fb(p, 9, 3, 1, p, 9, 3, 1, 1, 3, 3, 9, p, p, 1.0, p, p, None) == -1              # D <= 8
    assert b"D <= 8" in lib.pn_last_error_string()
    for B, N, M in ((0, 3, 3), (1, 0, 3), (1, 3, 0)):
        assert fb(p, 9, 3, 1, p, 9, 3, 1, B, N, M, 3, p, p, 1.0, p, p, None) == -1


def test_grad_path_rule():
    from pointnet12_b200.model.pointnet_util import grad_path

    x, g = torch.zeros(1, 4, 3), torch.zeros(1, 4, 3, requires_grad=True)
    assert grad_path(g) and grad_path(x, None, g) and not grad_path(x, None)
    assert not grad_path(torch.zeros(1, 4, dtype=torch.long))
    with torch.no_grad():
        assert not grad_path(g)


@pytest.mark.parametrize("call", ["square_distance", "index_points", "sample_and_group", "sample_and_group_all", "chamfer"])
def test_gradient_path_has_no_cpu_fallback(call):
    from pointnet12_b200.model import pointnet_util as U
    from pointnet12_b200.model.chamfer import chamfer_batch

    x = torch.zeros(1, 16, 3, requires_grad=True)
    fns = {"square_distance": lambda: U.square_distance(x, x),
           "index_points": lambda: U.index_points(x, torch.zeros(1, 4, dtype=torch.long)),
           "sample_and_group": lambda: U.sample_and_group(4, 0.2, 8, x, None, start_idx=torch.zeros(1, dtype=torch.long)),
           "sample_and_group_all": lambda: U.sample_and_group_all(x, None),
           "chamfer": lambda: chamfer_batch(x, x)}
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        fns[call]()
