"""CPU checks of gradients in eval() mode and with frozen BatchNorm: the fixed-statistics backward refuses bad arguments
before any launch, and the module-mode rules (which path a module takes, BatchNorm statistics, dropout) follow torch."""
import ctypes as C

import pytest
import torch

from pointnet12_b200 import _native as nv


def test_bn_eval_backward_abi_refuses_bad_arguments():
    lib = nv.lib()
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    f = lib.pn_bn_eval_bwd_f32
    # y, ldy, rows, C, dz, lddz, argmax, K, scale, shift, mean, invstd, relu, s1, s2, dy, lddy, dgamma, dbeta, stream
    assert f(None, 4, 10, 4, p, 4, None, 1, p, p, p, p, 1, p, p, p, 4, None, None, None) == -1
    assert b"null pointer" in lib.pn_last_error_string()
    assert f(p, 4, 10, 4, p, 4, None, 1, p, p, p, p, 1, None, p, p, 4, None, None, None) == -1       # no accumulator
    assert b"null pointer" in lib.pn_last_error_string()
    assert f(p, 4, 10, 4, p, 4, None, 1, p, p, p, p, 1, p, p, None, 4, None, None, None) == -1       # no dy
    for ldy, lddz, lddy in ((3, 4, 4), (4, 3, 4), (4, 4, 3)):                                          # a ld below C
        assert f(p, ldy, 10, 4, p, lddz, None, 1, p, p, p, p, 1, p, p, p, lddy, None, None, None) == -1
        assert b"bad shape" in lib.pn_last_error_string()
    assert f(p, 4, 0, 4, p, 4, None, 1, p, p, p, p, 1, p, p, p, 4, None, None, None) == -1            # no rows
    assert f(p, 4, 10, 0, p, 4, None, 1, p, p, p, p, 1, p, p, p, 4, None, None, None) == -1            # no channels
    assert f(p, 4, 10, 4, p, 4, p, 3, p, p, p, p, 1, p, p, p, 4, p, p, None) == -1                    # pooled: 10 % 3
    assert b"multiple of K" in lib.pn_last_error_string()
    assert f(p, 4, 10, 4, p, 4, p, 0, p, p, p, p, 1, p, p, p, 4, p, p, None) == -1


def test_bneval_gemm_abi_refuses_bad_arguments():
    lib = nv.lib()
    buf = (C.c_float * 64)()
    p = C.cast(buf, C.c_void_p)
    q = C.c_void_p(1 << 20)          # a 128-byte aligned address; validation fails before anything is dereferenced
    f = lib.pn_train_gemm_bneval_bf16x3
    # dy, lddy, rows, cin, w, w_transposed, cout, dy_prev, ld_dy_prev, prev_y, ld_prev, scale, shift, mean, invstd, s1, s2,
    # dgamma, dbeta, w_scratch, stream
    assert f(p, 4, 10, 4, p, 1, 4, p, 4, None, 4, p, p, p, p, p, p, None, None, q, None) == -1          # no prev_y
    assert b"null pointer" in lib.pn_last_error_string()
    assert f(p, 4, 10, 4, p, 1, 4, p, 4, p, 4, p, p, p, p, None, p, None, None, q, None) == -1          # no accumulator
    assert f(p, 4, 10, 4, p, 1, 4, None, 4, p, 4, p, p, p, p, p, p, None, None, q, None) == -1          # no output
    assert f(p, 4, 10, 4, p, 1, 4, p, 4, p, 3, p, p, p, p, p, p, None, None, q, None) == -1             # ld_prev < cout
    assert b"ld_prev" in lib.pn_last_error_string()
    assert f(p, 4, 10, 4, p, 1, 4, p, 3, p, 4, p, p, p, p, p, p, None, None, q, None) == -1             # ld_dy_prev < cout
    assert f(p, 259, 10, 259, p, 1, 256, p, 256, p, 256, p, p, p, p, p, p, None, None, q, None) == -2   # does not fit
    assert f(p, 4, 10, 4, p, 1, 4, p, 4, p, 4, p, p, p, p, p, p, None, None, C.c_void_p((1 << 20) + 4), None) == -3


def test_running_stats_are_the_folding_expressions_and_write_nothing():
    from pointnet12_b200 import ops
    from pointnet12_b200.model.pointnet_util import fold_conv_bn

    torch.manual_seed(0)
    conv, bn = torch.nn.Conv1d(8, 6, 1), torch.nn.BatchNorm1d(6).eval()
    with torch.no_grad():
        bn.weight.uniform_(0.5, 1.5)
        bn.bias.normal_()
        bn.running_mean.normal_()
        bn.running_var.uniform_(0.5, 2.0)
        bn.running_var[0] = 0.0
    before = [t.clone() for t in (bn.running_mean, bn.running_var, bn.num_batches_tracked)]
    versions = [t._version for t in (bn.running_mean, bn.running_var, bn.num_batches_tracked)]
    st = ops.running_stats(bn)
    assert st.running
    w, b = fold_conv_bn(conv, bn)
    w_plain = conv.weight.detach().reshape(6, -1)
    assert torch.equal(w, w_plain * st.scale[:, None])
    assert torch.equal(b, (conv.bias.detach() - bn.running_mean) * st.scale + bn.bias.detach())
    assert torch.equal(st.shift, bn.bias.detach() - bn.running_mean * st.scale)
    assert torch.equal(st.invstd, 1.0 / torch.sqrt(bn.running_var + bn.eps)) and torch.equal(st.mean, bn.running_mean)
    assert all(torch.equal(a, c) for a, c in zip(before, (bn.running_mean, bn.running_var, bn.num_batches_tracked)))
    assert versions == [t._version for t in (bn.running_mean, bn.running_var, bn.num_batches_tracked)]
    assert ops.running_stats(bn) is st                      # cached ...
    with torch.no_grad():
        bn.weight.mul_(2.0)
    assert ops.running_stats(bn) is not st                  # ... until a parameter changes


def test_module_mode_rules():
    from pointnet12_b200 import ops
    from pointnet12_b200.model.pointnet_util import PointNetFeaturePropagation, autograd_path
    from pointnet12_b200.train import _dropout_on

    bn = torch.nn.BatchNorm1d(4)
    assert not ops.uses_running_stats(bn.train()) and ops.uses_running_stats(bn.eval())
    assert not ops.uses_running_stats(torch.nn.BatchNorm1d(4, track_running_stats=False).eval())
    drop = torch.nn.Dropout(0.5)
    assert _dropout_on(drop.train()) and not _dropout_on(drop.eval())
    assert not _dropout_on(drop.eval(), mask=torch.ones(1)) and not _dropout_on(torch.nn.Dropout(0.0).train())
    m = PointNetFeaturePropagation(8, [8])
    x, g = torch.zeros(1, 3, 4), torch.zeros(1, 3, 4, requires_grad=True)
    assert autograd_path(m.train(), x, None)
    assert not autograd_path(m.eval(), x, None, x)
    assert autograd_path(m.eval(), x, None, g)
    with torch.no_grad():
        assert not autograd_path(m.eval(), x, g)
    assert not autograd_path(m.eval(), torch.zeros(1, 3, 4, dtype=torch.long))


def test_semseg_host_out_refuses_an_input_that_requires_a_gradient():
    from pointnet12_b200.model.pointnet2 import PointNet2SemSeg

    net = PointNet2SemSeg(19, 1).eval()
    points = torch.zeros(1, 4, 2048, requires_grad=True)
    with pytest.raises(ValueError, match="host_out"):
        net(points, host_out=torch.empty(1, 2048, 19))
