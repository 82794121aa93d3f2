"""Monodepth2's axis-angle pose (SFM_FLAG_AXISANGLE_POSE): the numpy reference (tests/axisangle_oracle.py) against torch
fp64 autograd of Monodepth2's own functions (tests/torch_axisangle_restatement.py), the whole-loss gradients against
central differences, and the ABI / operator checks that need no GPU."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import axisangle_oracle as AA
from tests.torch_axisangle_restatement import transform_rows

THETAS = [0.0, 1e-8, 1e-7, 1e-3, 0.1, 1.0, 4.0]     # 4 > pi: no clipping, the angle wraps


def _poses(theta, n=8, seed=0):
    rs = np.random.RandomState(seed)
    ax = rs.standard_normal((n, 3))
    ax /= np.linalg.norm(ax, axis=1, keepdims=True)
    t = rs.standard_normal((n, 3)) * 0.3
    return np.concatenate([ax * theta, t], 1)


@pytest.mark.parametrize('inv', [False, True])
@pytest.mark.parametrize('theta', THETAS)
def test_transform_and_chain_match_torch_autograd(theta, inv):
    p = _poses(theta, seed=int(theta * 1e3) + 7).astype(np.float32).astype(np.float64)    # fp32 values, as the device's
    pt = torch.from_numpy(p).requires_grad_(True)
    M = transform_rows(pt, inv)
    q = AA.rot(p[:, :3])
    R, t = q['R'], p[:, 3:]
    T = np.concatenate([np.swapaxes(R, 1, 2), -np.einsum('nji,nj->ni', R, t)[:, :, None]], 2) if inv else \
        np.concatenate([R, t[:, :, None]], 2)
    np.testing.assert_allclose(T, M.detach().numpy(), rtol=1e-9, atol=1e-15)
    # the fp32 tables round exactly this transform
    Rf, tf = AA.transform(p.astype(np.float32), inv)
    np.testing.assert_array_equal(np.concatenate([Rf, tf[:, :, None]], 2), T.astype(np.float32))
    dT = np.random.RandomState(3).standard_normal((p.shape[0], 3, 4))
    (M * torch.from_numpy(dT)).sum().backward()
    ref = pt.grad.numpy()
    got = AA.chain(p, dT, inv)
    np.testing.assert_allclose(got, ref, rtol=1e-7, atol=1e-7 * np.abs(ref).max())


def test_zero_angle_follows_torch_convention():
    """At theta = 0 torch's norm backward gives d theta / d v = 0: dL/dv = dL/da / 1e-7 alone."""
    p = np.zeros((1, 6))
    dT = np.random.RandomState(5).standard_normal((1, 3, 4))
    pt = torch.from_numpy(p).requires_grad_(True)
    (transform_rows(pt) * torch.from_numpy(dT)).sum().backward()
    assert np.all(np.isfinite(pt.grad.numpy()))
    np.testing.assert_allclose(AA.chain(p, dT, False), pt.grad.numpy(), rtol=1e-9)


@pytest.mark.parametrize('inv', [(), (0,), (0, 1)])
def test_tables_are_k_times_the_transform(inv):
    d = make_snippets(2, 2, 32, 64, seed=11, n_scales=2)
    proj, kinv = AA.tables(d['poses'], d['intrinsics'], inv)
    for i in range(2):
        Rf, tf = AA.transform(d['poses'][:, i], i in inv)
        T = np.concatenate([Rf, tf[:, :, None]], 2).astype(np.float64)
        for s in range(2):
            np.testing.assert_allclose(proj[:, i, s], d['intrinsics'][:, s].astype(np.float64) @ T, rtol=1e-6, atol=1e-4)
    np.testing.assert_array_equal(kinv[:, 1], O.batch_inv3(d['intrinsics'][:, 1]))


@pytest.mark.parametrize('inv', [(), (1,)])
def test_whole_loss_gradients_central_differences(inv):
    """gposes and gintrinsics of the reference against fp64 central differences of its loss (the total is a smooth
    function of the pose and K away from floor flips and |P - T| kinks: entries with a kink in range are skipped)."""
    cfg = O.LossConfig(n_scales=2, smooth_reg=0.1, ssim_rate=0.15)
    d = make_snippets(1, 2, 24, 48, seed=31, n_scales=2, dtype=np.float64)
    args = lambda a: (a['tgt'], a['src'], a['intrinsics'], a['disps'], a['poses'], cfg)
    _, G = AA.loss(*args(d), invert_sources=inv, want_intrinsics_grad=True)

    def total(**over):
        return AA.loss(*args(dict(d, **over)), invert_sources=inv, want_grads=False)[0]['total_loss']
    mid = total()
    eps = 1e-7
    checked = 0
    cases = [('poses', ix) for ix in np.ndindex(*d['poses'].shape)]
    cases += [('intrinsics', (0, s, r, c)) for s in range(2) for r, c in ((0, 0), (0, 2), (1, 1), (1, 2))]
    for key, ix in cases:
        vals = []
        for sgn in (1, -1):
            a = d[key].copy()
            a[ix] += sgn * eps
            vals.append(total(**{key: a}))
        if abs((vals[0] - mid) - (mid - vals[1])) > 1e-3 * abs(vals[0] - vals[1]) + 1e-15:
            continue
        fd = (vals[0] - vals[1]) / (2 * eps)
        ref = G['gpose'][ix] if key == 'poses' else G['gintrinsics'][ix]
        assert abs(fd - ref) <= 1e-4 * abs(ref) + 1e-8, (key, ix, fd, ref)
        checked += 1
    assert checked >= 16


@pytest.mark.parametrize('inv', [(), (0,)])
def test_intrinsics_grad_matches_torch_autograd(inv):
    """gintrinsics of the reference (R and t of the axis-angle transform) against torch fp64 autograd of the restatement
    with K a leaf and Monodepth2's transform; the photometric part only (smooth_reg = 0)."""
    from tests.torch_axisangle_restatement import torch_total_axisangle
    cfg = O.LossConfig(n_scales=2, smooth_reg=0.0, ssim_rate=0.15)
    d = make_snippets(2, 2, 24, 48, seed=41, n_scales=2, dtype=np.float64)
    _, G = AA.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], cfg, invert_sources=inv,
                   want_intrinsics_grad=True)
    K = torch.from_numpy(d['intrinsics']).requires_grad_(True)
    tot = torch_total_axisangle(d, cfg, torch.from_numpy(d['tgt']), torch.from_numpy(d['src']), K, invert_sources=inv)
    tot.backward()
    ref = K.grad.numpy()
    np.testing.assert_allclose(G['gintrinsics'], ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())


@pytest.fixture
def lib():
    from sfm_learner_chainer_b200 import lib as L
    try:
        L.load()
    except ImportError:
        pytest.skip('libsfmloss.so not built')
    return L


def test_flag_values_and_abi(lib):
    import os
    hdr = open(os.path.join(os.path.dirname(__file__), '..', 'include', 'sfmloss.h')).read()
    assert '#define SFM_FLAG_AXISANGLE_POSE 0x800u' in hdr and lib.SFM_FLAG_AXISANGLE_POSE == 0x800
    assert '#define SFM_FLAG_POSE_INVERT_SHIFT 16' in hdr and lib.SFM_FLAG_POSE_INVERT_SHIFT == 16
    so = lib.load()
    assert so.sfm_version() == 102
    assert C.sizeof(lib.SfmDesc) == 48
    F, sh = lib.SFM_FLAG_AXISANGLE_POSE, lib.SFM_FLAG_POSE_INVERT_SHIFT
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, 0)
    n0 = so.sfm_workspace_bytes(C.byref(d))
    for flags, ok in ((F, True), (F | 1 << sh, True), (F | 3 << sh, True), (1 << sh, False), (F | 4 << sh, False),
                      (F | 0x80 << sh, False)):
        d.flags = flags
        assert (so.sfm_workspace_bytes(C.byref(d)) == n0) == ok, hex(flags)     # the flag does not size the workspace
    buf = (C.c_float * 64)()
    ptr = C.cast(buf, C.c_void_p)
    inp = lib.SfmInputs()
    for flags in (1 << sh, F | 4 << sh):
        d.flags = flags
        assert so.sfm_loss_forward(C.byref(d), C.byref(inp), ptr, None, ptr, None) == lib.SFM_E_INVALID_DESC
        assert so.sfm_build_tables(C.byref(d), ptr, ptr, ptr, ptr, None) == lib.SFM_E_INVALID_DESC
        assert so.sfm_intrinsics_grad(C.byref(d), C.byref(inp), ptr, ptr, None) == lib.SFM_E_INVALID_DESC
    d.flags = F | 1 << sh
    ctx = C.c_void_p()
    assert so.sfm_host_ctx_create(C.byref(d), C.byref(ctx)) == lib.SFM_E_UNSUPPORTED
    # a valid descriptor gets as far as the inputs check
    assert so.sfm_loss_forward(C.byref(d), C.byref(inp), ptr, None, ptr, None) == lib.SFM_E_NULL_POINTER


def test_operator_options(lib):
    from sfm_learner_chainer_b200.functions import ViewSynthesisLoss
    with pytest.raises(ValueError):
        ViewSynthesisLoss(invert_sources=(0,))
    with pytest.raises(ValueError):
        ViewSynthesisLoss(axisangle_pose=True, invert_sources=(-1,))
    op = ViewSynthesisLoss(ssim_rate=0.15, axisangle_pose=True, invert_sources=(0,))
    f = op._desc(2, 2, 64, 208).flags
    assert f & lib.SFM_FLAG_AXISANGLE_POSE and f >> lib.SFM_FLAG_POSE_INVERT_SHIFT == 1
    assert ViewSynthesisLoss(axisangle_pose=True, invert_sources=(0, 3))._desc(2, 4, 64, 208).flags >> 16 == 0b1001
    with pytest.raises(ValueError):
        ViewSynthesisLoss(axisangle_pose=True, invert_sources=(2,))._desc(2, 2, 64, 208)
    assert not ViewSynthesisLoss(ssim_rate=0.15)._desc(2, 2, 64, 208).flags & lib.SFM_FLAG_AXISANGLE_POSE
