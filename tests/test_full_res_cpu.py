"""-m "not gpu": the full-resolution multi-scale loss (SFM_FLAG_FULL_RES_MULTISCALE).

The numpy upsampling pair U / U^T of tests/full_res_oracle.py is checked against F.interpolate and its autograd and for
adjointness; the composed reference against torch fp64 autograd of an independent restatement
(tests/torch_full_res_restatement.py) and against central differences; the C ABI additions for their workspace size
and argument errors without a device, and the Python option for its argument checks."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import full_res_oracle as FR
from tests.torch_full_res_restatement import torch_full_res


def _args(d):
    return d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses']


@pytest.mark.parametrize('hw,HW', [((4, 6), (36, 52)), ((9, 13), (36, 52)), ((16, 52), (128, 416)), ((7, 5), (7, 11))])
def test_upsample_pair_matches_interpolate_and_is_adjoint(hw, HW):
    rs = np.random.RandomState(5)
    x = rs.uniform(0.01, 10, (2, 1) + hw)
    y = rs.standard_normal((2, 1) + HW)
    ref = F.interpolate(torch.from_numpy(x), size=HW, mode='bilinear', align_corners=False).numpy()
    np.testing.assert_allclose(FR.upsample(x, *HW), ref, rtol=1e-14, atol=0)
    # fp32 (torch's CPU kernel associates differently; the 2-ulp comparison with torch is made on the GPU)
    x32 = x.astype(np.float32)
    np.testing.assert_allclose(FR.upsample(x32, *HW), FR.upsample(x32.astype(np.float64), *HW), rtol=1e-5)
    # U^T against autograd of F.interpolate, and <U x, y> == <x, U^T y>
    xt = torch.from_numpy(x).requires_grad_(True)
    F.interpolate(xt, size=HW, mode='bilinear', align_corners=False).backward(torch.from_numpy(y))
    ut = FR.upsample_adjoint(y, *hw, dtype=np.float64)
    np.testing.assert_allclose(ut, xt.grad.numpy(), rtol=1e-12, atol=1e-12)
    assert np.isclose(np.sum(FR.upsample(x, *HW) * y), np.sum(x * ut), rtol=1e-12)
    # the matrix form of U is the elementwise one
    U = np.einsum('Yy,ncyx,Xx->ncYX', FR.up_matrix(hw[0], HW[0], np.float64), x, FR.up_matrix(hw[1], HW[1], np.float64))
    np.testing.assert_allclose(U, FR.upsample(x, *HW), rtol=1e-14)


CASES = {
    'l1': dict(smooth_reg=0.0, ssim_rate=0.0),
    'ssim_smooth': dict(smooth_reg=0.1, ssim_rate=0.15),
    'edge': dict(smooth_reg=0.1, ssim_rate=0.15, edge_aware_smooth=True),
}


@pytest.mark.parametrize('case', sorted(CASES))
@pytest.mark.parametrize('mode', ['plain', 'weighted', 'minrep', 'minrep_automask'])
def test_oracle_matches_torch_autograd(case, mode):
    """36 x 52 is not a multiple of 2^3: U's scale h_s / H differs from 2^-s."""
    d = make_snippets(2, 2, 36, 52, seed=610, n_scales=4, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=4, **CASES[case])
    rs = np.random.RandomState(611)
    pw = [rs.uniform(-0.5, 2.0, (2, 2, 36, 52)) for _ in range(4)] if mode == 'weighted' else None
    pw = None if pw is None else [pw[0], None, pw[2], pw[3]]
    minrep, automask = mode.startswith('minrep'), mode == 'minrep_automask'
    L, G = FR.sfm_loss_full_res(*_args(d), cfg, pixel_weights=pw, min_reprojection=minrep, automask=automask,
                                want_intrinsics_grad=True)
    disps = [torch.from_numpy(x).requires_grad_(True) for x in d['disps']]
    poses = torch.from_numpy(d['poses']).requires_grad_(True)
    K = torch.from_numpy(d['intrinsics']).requires_grad_(True)
    tw = None if pw is None else [None if w is None else torch.from_numpy(w) for w in pw]
    total, pixel, ssim, smooth, sels = torch_full_res(d, cfg, disps, poses, K, pixel_weights=tw, min_reprojection=minrep,
                                                      automask=automask)
    if minrep:
        for s in range(4):
            np.testing.assert_array_equal(L['selection'][s], sels[s].numpy())
        if automask:
            assert any((x == -1).any() for x in L['selection'])
    for k, v in (('total_loss', total), ('pixel_loss', pixel), ('ssim_loss', ssim), ('smooth_loss', smooth)):
        np.testing.assert_allclose(L[k], float(torch.as_tensor(v).detach()), rtol=1e-10, atol=1e-15)
    total.backward()
    for s in range(4):
        ref = disps[s].grad.numpy()
        np.testing.assert_allclose(G['gdisp'][s], ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    for got, ref in ((G['gpose'], poses.grad.numpy()), (G['gintrinsics'], K.grad.numpy())):
        np.testing.assert_allclose(got, ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max())
    assert not G['gintrinsics'][:, 1:].any()


@pytest.mark.parametrize('minrep', [False, True])
def test_gradients_central_differences(minrep):
    """gdisp of every scale and gpose against fp64 central differences of the reference's total on sampled entries,
    skipping entries with a kink in range."""
    cfg = O.LossConfig(n_scales=3, smooth_reg=0.1, ssim_rate=0.15)
    d = make_snippets(1, 2, 20, 28, seed=620, n_scales=3, harsh=True, dtype=np.float64)
    _, G = FR.sfm_loss_full_res(*_args(d), cfg, min_reprojection=minrep)

    def total(**over):
        a = dict(d, **over)
        return FR.sfm_loss_full_res(*_args(a), cfg, min_reprojection=minrep, want_grads=False)[0]['total_loss']
    mid = total()
    rs = np.random.RandomState(9)
    eps = 1e-7
    checked = 0
    for _ in range(30):
        s = rs.randint(-1, 3)
        arr, ref = (d['poses'], G['gpose']) if s < 0 else (d['disps'][s], G['gdisp'][s])
        ix = tuple(rs.randint(0, n) for n in arr.shape)
        vals = []
        for sgn in (1, -1):
            a = arr.copy()
            a[ix] += sgn * eps
            if s < 0:
                vals.append(total(poses=a))
            else:
                lst = list(d['disps'])
                lst[s] = a
                vals.append(total(disps=lst))
        if abs((vals[0] - mid) - (mid - vals[1])) > 1e-3 * abs(vals[0] - vals[1]) + 1e-15:
            continue
        fd = (vals[0] - vals[1]) / (2 * eps)
        assert abs(fd - ref[ix]) <= 1e-4 * abs(ref[ix]) + 1e-8, (s, ix, fd, ref[ix])
        checked += 1
    assert checked >= 20


def test_raw_inputs_are_activated_before_the_upsampling():
    """Raw bits: the reference of the raw inputs equals the plain reference of the activated maps, with gdisp times the
    activation's derivative at the native pixel."""
    cfg = O.LossConfig(n_scales=3, smooth_reg=0.1, ssim_rate=0.15)
    d = make_snippets(2, 2, 20, 28, seed=630, n_scales=3, harsh=True, dtype=np.float64)
    raw = [np.log(np.clip((x - 0.01) / 10, 1e-6, 1 - 1e-6) / (1 - np.clip((x - 0.01) / 10, 1e-6, 1 - 1e-6))) for x in d['disps']]
    L, G = FR.sfm_loss_full_res(d['tgt'], d['src'], d['intrinsics'], raw, d['poses'], cfg, raw_disp_scales=0x7)
    act = [O.disp_activation(x) for x in raw]
    Lp, Gp = FR.sfm_loss_full_res(d['tgt'], d['src'], d['intrinsics'], [a for a, _ in act], d['poses'], cfg)
    assert L['total_loss'] == Lp['total_loss']
    for s in range(3):
        np.testing.assert_allclose(G['gdisp'][s], Gp['gdisp'][s] * act[s][1], rtol=1e-12)


# ---- C ABI and Python option, without a device
@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sfm_learner_chainer_b200 import lib as L
    return L


def test_flag_sizes_the_workspace_only_when_set(lib):
    so = lib.load()
    assert lib.SFM_FLAG_FULL_RES_MULTISCALE == 0x80
    for B, S, H, W, ns in ((4, 2, 128, 416, 4), (2, 3, 36, 52, 4), (1, 2, 64, 208, 1)):
        plain = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, 0)
        fr = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_FULL_RES_MULTISCALE)
        n0, n1 = so.sfm_workspace_bytes(C.byref(plain)), so.sfm_workspace_bytes(C.byref(fr))
        assert n0 > 0 and n1 > 0
        if ns == 1:
            assert n1 == n0                      # one scale: the flag changes nothing
            continue
        extra = (ns - 1) * 2 * B * H * W * 4 + B * ns * 9 * 4      # U_s(d_s) and its gradient per scale >= 1, K_0 copy
        assert extra <= n1 - n0 <= extra + 256 * (2 * ns + 1)
        # the min-reprojection planes grow to B*S*H*W per scale
        mr0 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_MIN_REPROJECTION)
        mr1 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_MIN_REPROJECTION | lib.SFM_FLAG_FULL_RES_MULTISCALE)
        planes0 = sum(B * S * (H >> s) * (W >> s) * 4 for s in range(ns))
        grow = so.sfm_workspace_bytes(C.byref(mr1)) - so.sfm_workspace_bytes(C.byref(mr0))
        assert abs(grow - (n1 - n0) - (ns * B * S * H * W * 4 - planes0)) <= 256 * (3 * ns + 1)


def test_unsupported_combinations_and_stage_errors(lib):
    so = lib.load()
    fr = lib.SFM_FLAG_FULL_RES_MULTISCALE
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, fr | lib.SFM_FLAG_IMAGE_GRADS)
    inp, g = lib.SfmInputs(), lib.SfmGrads()
    ig = lib.SfmImageGrads(C.c_void_p(256), None)
    rc = so.sfm_loss_forward_backward_images(C.byref(d), C.byref(inp), C.c_void_p(256), C.byref(g), C.byref(ig),
                                             C.c_void_p(256), None)
    assert rc == lib.SFM_E_UNSUPPORTED and b'FULL_RES' in so.sfm_last_error()
    rc = so.sfm_loss_snippets(C.byref(d), C.byref(inp), None, C.c_void_p(256), C.byref(g), C.byref(ig), C.c_void_p(256),
                              None, None)
    assert rc == lib.SFM_E_UNSUPPORTED and b'FULL_RES' in so.sfm_last_error()
    ctx = C.c_void_p()
    assert so.sfm_host_ctx_create(C.byref(d), C.byref(ctx)) == lib.SFM_E_UNSUPPORTED
    assert b'FULL_RES' in so.sfm_last_error()
    assert so.sfm_upsample_disparity(1, 8, 8, 4, 16, C.c_void_p(256), C.c_void_p(256), None) == lib.SFM_E_INVALID_SHAPE
    assert so.sfm_upsample_disparity(1, 8, 8, 16, 16, None, C.c_void_p(256), None) == lib.SFM_E_NULL_POINTER


def test_python_option_checks(lib):
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    with pytest.raises(ValueError, match='exp_reg'):
        ViewSynthesisLoss(0.1, 0.2, 0.0, full_res_multiscale=True)
    with pytest.raises(ValueError, match='image_grads'):
        ViewSynthesisLoss(0.1, 0.0, 0.15, full_res_multiscale=True, image_grads=True)
    op = ViewSynthesisLoss(0.1, 0.0, 0.15, full_res_multiscale=True, min_reprojection=True, pixel_terms=False)
    desc = op._desc(2, 2, 64, 208)
    assert desc.flags & lib.SFM_FLAG_FULL_RES_MULTISCALE and desc.flags & lib.SFM_FLAG_MIN_REPROJECTION
    assert op._step_hw(desc, 3) == (64, 208)
    assert ViewSynthesisLoss(0.1, 0.0, 0.15)._step_hw(desc, 3) == (8, 26)
