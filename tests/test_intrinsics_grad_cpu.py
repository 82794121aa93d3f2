"""-m "not gpu": gradient of the fused loss w.r.t. the camera intrinsics (d total / d intrinsics).

The oracle's gintrinsics (O.sfm_loss(want_intrinsics_grad=True)) is checked against torch fp64 autograd through an
independent restatement of the whole K-dependent path (tests/torch_restatement.py: K a leaf through torch.linalg.inv and
K @ [R|t], the grid with the x2 rule, grid_sample, the L1 / explainability / SSIM terms), against central differences
of the numpy oracle, and on the poses where the formula has a closed form.  The C ABI additions are checked for their argument errors without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests.torch_restatement import torch_total

FLAGS = {
    'l1': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.0),
    'exp': dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
}


def _data(B, S, H, W, ns, harsh, seed=0):
    return make_snippets(B, S, H, W, seed=seed, n_scales=ns, harsh=harsh, dtype=np.float64)


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 2, 4])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_oracle_intrinsics_grad_matches_torch_autograd(flags, S, ns, harsh):
    d = _data(2, S, 32, 64, ns, harsh, seed=S + 10 * ns + 100 * harsh)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L, G, _ = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg,
                         want_intrinsics_grad=True)
    K = torch.from_numpy(d['intrinsics']).requires_grad_(True)
    tot = torch_total(d, cfg, torch.from_numpy(d['tgt']), torch.from_numpy(d['src']), K)
    tot.backward()
    # the restatement leaves out only K-independent terms
    np.testing.assert_allclose(tot.item(), L['total_loss'] - L['smooth_loss'] - L['exp_loss'], rtol=1e-9, atol=1e-12)
    ref = K.grad.numpy()
    got = G['gintrinsics']
    assert got.dtype == np.float64 and got.shape == (2, ns, 3, 3)
    np.testing.assert_allclose(got, ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())
    assert np.abs(ref).max() > 0


@pytest.mark.parametrize('flags', sorted(FLAGS))
def test_oracle_intrinsics_grad_central_differences(flags):
    """fp64 central differences of the reported total on every entry of K, the step scaled per entry.  Floor flips
    of the sampling coordinates and the x2 rule's boundary move with K: a kink or jump inside [-eps, eps] shows as a
    one-sided difference that disagrees with the other side, and that entry is skipped."""
    d = _data(2, 2, 32, 64, 4, True, seed=7)
    cfg = O.LossConfig(n_scales=4, **FLAGS[flags])

    def total(K):
        return O.sfm_loss(d['tgt'], d['src'], K, d['disps'], d['poses'], d['logits'], cfg, want_grads=False)[0]['total_loss']

    _, G, _ = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg,
                         want_intrinsics_grad=True)
    ref = G['gintrinsics']
    mid = total(d['intrinsics'])
    checked = 0
    for ix in np.ndindex(*ref.shape):
        eps = 1e-7 * max(1.0, abs(d['intrinsics'][ix]))
        vals = []
        for sgn in (1, -1):
            K = d['intrinsics'].copy()
            K[ix] += sgn * eps
            vals.append(total(K))
        if abs((vals[0] - mid) - (mid - vals[1])) > 1e-3 * abs(vals[0] - vals[1]) + 1e-15:
            continue
        fd = (vals[0] - vals[1]) / (2 * eps)
        # the difference of two totals of order 1 carries ~1e-16 / eps of rounding
        assert abs(fd - ref[ix]) <= 1e-5 * abs(ref[ix]) + 2e-16 / eps, (ix, fd, ref[ix])
        checked += 1
    assert checked >= 60


def test_zero_rotation_closed_forms():
    """R = I, t = 0: the loss does not depend on K and the formula is A - A; R = I, t != 0: exactly sum_i g_i t_i^T."""
    d = _data(2, 3, 32, 64, 4, False, seed=21)
    cfg = O.LossConfig(n_scales=4, **FLAGS['ssim'])
    for t in (np.zeros(3), np.array([0.02, -0.01, 0.03])):
        poses = np.zeros_like(d['poses'])
        poses[..., 3:] = t
        _, G, _ = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], poses, d['logits'], cfg, want_intrinsics_grad=True)
        A = G['dP'][..., :3]
        closed = np.einsum('bisk,j->bskj', G['dP'][..., 3], t)
        np.testing.assert_allclose(G['gintrinsics'], closed, rtol=0, atol=1e-12 * np.abs(A).max())
        if t.any():
            assert np.abs(closed).max() > 1e3 * 1e-12 * np.abs(A).max()


def test_raw_counterpart_uses_the_reduced_poses():
    from sfm_learner_chainer_b200.synthetic import make_raw_seam
    d = _data(2, 2, 32, 64, 4, True, seed=31)
    raw_disps, raw_poses = make_raw_seam(d, (1, 4), seed=32)
    cfg = O.LossConfig(n_scales=4, **FLAGS['l1'])
    L, G, dbg = O.sfm_loss_raw(d['tgt'], d['src'], d['intrinsics'], raw_disps, raw_poses, d['logits'], cfg,
                               raw_disp_scales=0xF, raw_pose=True, want_intrinsics_grad=True)
    L2, G2, _ = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], dbg['disps'], dbg['poses'], d['logits'], cfg,
                           want_intrinsics_grad=True)
    assert L == L2
    np.testing.assert_array_equal(G['gintrinsics'], G2['gintrinsics'])


# ---- C ABI, without a device ---------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sfm_learner_chainer_b200 import lib as L
    return L


def test_intrinsics_grad_symbols(lib):
    so = lib.load()
    for name in ('sfm_intrinsics_grad', 'sfm_scale_intrinsics_grad'):
        assert name in lib.SYMBOLS and getattr(so, name) is not None


def test_intrinsics_grad_argument_errors(lib):
    so = lib.load()
    d = lib.SfmDesc(4, 2, 128, 416, 4, 0, 0.1, 0.0, 0.15, 0)
    buf = (C.c_float * 16)()
    inp = lib.SfmInputs()
    inp.intrinsics, inp.poses = C.cast(buf, C.c_void_p), C.cast(buf, C.c_void_p)
    ws, gk = C.c_void_p(256), C.cast(buf, C.c_void_p)
    call = lambda desc, i, w, g: so.sfm_intrinsics_grad(C.byref(desc), i, w, g, None)
    assert call(d, None, ws, gk) == lib.SFM_E_NULL_POINTER
    assert call(d, C.byref(lib.SfmInputs()), ws, gk) == lib.SFM_E_NULL_POINTER     # no intrinsics / poses
    assert call(d, C.byref(inp), None, gk) == lib.SFM_E_NULL_POINTER
    assert call(d, C.byref(inp), ws, None) == lib.SFM_E_NULL_POINTER
    assert call(d, C.byref(inp), C.c_void_p(16), gk) == lib.SFM_E_INVALID_DESC    # misaligned workspace
    assert so.sfm_intrinsics_grad(None, C.byref(inp), ws, gk, None) == lib.SFM_E_NULL_POINTER
    bad = lib.SfmDesc(0, 2, 128, 416, 4, 0, 0.1, 0.0, 0.15, 0)
    assert call(bad, C.byref(inp), ws, gk) == lib.SFM_E_INVALID_DESC
    d.flags = lib.SFM_FLAG_TABLES_PROVIDED
    assert call(d, C.byref(inp), ws, gk) == lib.SFM_E_UNSUPPORTED
    assert b'SFM_FLAG_TABLES_PROVIDED' in so.sfm_last_error()
    d.flags = 0
    assert so.sfm_scale_intrinsics_grad(C.byref(d), None, gk, None) == lib.SFM_E_NULL_POINTER
    assert so.sfm_scale_intrinsics_grad(C.byref(d), C.c_void_p(256), None, None) == lib.SFM_E_NULL_POINTER
    assert so.sfm_scale_intrinsics_grad(C.byref(bad), C.c_void_p(256), gk, None) == lib.SFM_E_INVALID_DESC


def test_operator_refuses_caller_tables(lib):
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    op = ViewSynthesisLoss(0.1, 0.0, 0.15, intrinsics_grad=True)
    d = _data(1, 2, 32, 64, 4, False)
    args = (d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'])
    with pytest.raises(ValueError):
        op.forward_backward(*args, proj=np.zeros(1), kinv=np.zeros(1))
    with pytest.raises(ValueError):
        op.backward(*args, proj=np.zeros(1), kinv=np.zeros(1))
