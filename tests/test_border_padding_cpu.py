"""Monodepth2's image borders (SFM_FLAG_BORDER_PADDING) without a GPU: the numpy reference (tests/border_oracle.py, the
weighted, min-reprojection and full-resolution references under the flag) against autograd of an independent
torch fp64 restatement of Monodepth2's code and against central differences, and the flag's argument checks."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import border_oracle as BO
from tests.border_oracle import avg_pool3_reflect, avg_pool3_reflect_adjoint
from tests.pixel_oracle import sfm_loss_pixel
from tests.torch_border_restatement import torch_border

FLAGS = {
    'l1': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.15),
}
MODES = ['plain', 'min_reprojection', 'full_res', 'full_res_min_reprojection']
SHAPES = {'32x64': (32, 64, 2), '16x16': (16, 16, 3)}          # the second has a 4x4 coarsest scale


def _args(d):
    return d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses']


def _reference(d, cfg, mode, **kw):
    if mode.startswith('full_res'):
        return BO.loss_full_res(*_args(d), cfg, min_reprojection=mode.endswith('min_reprojection'), **kw)
    if mode == 'min_reprojection':
        return BO.loss_min_reprojection(*_args(d), cfg, **kw)
    return BO.loss_pixel(*_args(d), cfg, **kw)


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [2, 4])
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('shape', sorted(SHAPES))
def test_oracle_matches_torch_autograd(flags, S, mode, shape):
    H, W, ns = SHAPES[shape]
    d = make_snippets(2, S, H, W, seed=310 + S, n_scales=ns, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L, G = _reference(d, cfg, mode)
    disps = [torch.from_numpy(x).requires_grad_(True) for x in d['disps']]
    poses = torch.from_numpy(d['poses']).requires_grad_(True)
    minrep = mode.endswith('min_reprojection')
    phot, pixel, ssim, sels = torch_border(d, cfg, disps, poses, min_reprojection=minrep, full_res=mode.startswith('full_res'))
    if minrep:
        for s in range(ns):
            np.testing.assert_array_equal(L['selection'][s], sels[s].numpy())
    np.testing.assert_allclose(L['pixel_loss'], pixel.item(), rtol=1e-9)
    np.testing.assert_allclose(L['ssim_loss'], float(torch.as_tensor(ssim).detach()), rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose(L['total_loss'], phot.item(), rtol=1e-9)
    phot.backward()
    for s in range(ns):
        ref = disps[s].grad.numpy()
        np.testing.assert_allclose(G['gdisp'][s], ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())
    ref = poses.grad.numpy()
    np.testing.assert_allclose(G['gpose'], ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())


def test_border_pixels_are_scored():
    """With a pose that moves much of the image out of view, the reference masks those pixels and the border rule
    scores them: the border loss differs, and no pixel is masked (every map entry is finite and non-negative)."""
    d = make_snippets(1, 2, 32, 64, seed=5, n_scales=1, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=1, ssim_rate=0.15)
    Lb, _ = BO.loss_pixel(*_args(d), cfg, want_grads=False)
    Lz, _ = sfm_loss_pixel(*_args(d), None, cfg, want_grads=False)
    assert Lb['pixel_loss'] > Lz['pixel_loss']
    assert (Lz['pixel_losses'][0] == 0).any() and (Lb['pixel_losses'][0] > 0).all()


def test_reflected_pool_adjoint():
    """<pool(x), g> == <x, pool^T(g)> at shapes down to 3x3 (the folds of both ends meet)."""
    rs = np.random.RandomState(3)
    for h, w in ((3, 3), (4, 5), (7, 4), (9, 13)):
        x, g = rs.randn(2, 3, h, w), rs.randn(2, 3, h, w)
        np.testing.assert_allclose(np.sum(avg_pool3_reflect(x) * g), np.sum(x * avg_pool3_reflect_adjoint(g)), rtol=1e-12)


@pytest.mark.parametrize('flags', sorted(FLAGS))
def test_gradients_central_differences(flags):
    """gdisp and gpose against fp64 central differences of the reference's total on sampled entries, skipping entries
    with a kink in range (a clamp boundary, |P - T|, a floor flip, the SSIM clip, a selection flip)."""
    cfg = O.LossConfig(n_scales=3, **dict(FLAGS[flags], smooth_reg=0.1))
    d = make_snippets(1, 2, 32, 64, seed=177, n_scales=3, harsh=True, dtype=np.float64)
    _, G = BO.loss_min_reprojection(*_args(d), cfg)

    def total(**over):
        a = dict(d, **over)
        return BO.loss_min_reprojection(*_args(a), cfg, want_grads=False)[0]['total_loss']
    mid = total()
    rs = np.random.RandomState(9)
    eps = 1e-7
    checked = 0
    for key in ('disps', 'poses'):
        for _ in range(24):
            if key == 'poses':
                arr, ref, s = d['poses'], G['gpose'], None
            else:
                s = rs.randint(0, 3)
                arr, ref = d['disps'][s], G['gdisp'][s]
            ix = tuple(rs.randint(0, n) for n in arr.shape)
            vals = []
            for sgn in (1, -1):
                a = arr.copy()
                a[ix] += sgn * eps
                if s is None:
                    vals.append(total(poses=a))
                else:
                    lst = list(d['disps'])
                    lst[s] = a
                    vals.append(total(disps=lst))
            if abs((vals[0] - mid) - (mid - vals[1])) > 1e-3 * abs(vals[0] - vals[1]) + 1e-15:
                continue
            fd = (vals[0] - vals[1]) / (2 * eps)
            assert abs(fd - ref[ix]) <= 1e-4 * abs(ref[ix]) + 1e-8, (key, s, ix, fd, ref[ix])
            checked += 1
    assert checked >= 20


@pytest.fixture
def lib():
    from sfm_learner_chainer_b200 import lib as L
    try:
        L.load()
    except ImportError:
        pytest.skip('libsfmloss.so not built')
    return L


def test_flag_value_and_workspace(lib):
    import os
    hdr = open(os.path.join(os.path.dirname(__file__), '..', 'include', 'sfmloss.h')).read()
    assert '#define SFM_FLAG_BORDER_PADDING 0x400u' in hdr and lib.SFM_FLAG_BORDER_PADDING == 0x400
    so = lib.load()
    d = lib.SfmDesc(2, 3, 64, 208, 4, 0, 0.1, 0.0, 0.15, 0)
    n0 = so.sfm_workspace_bytes(C.byref(d))
    d.flags = lib.SFM_FLAG_BORDER_PADDING
    assert so.sfm_workspace_bytes(C.byref(d)) == n0                  # the flag does not size the workspace


def test_abi_unsupported_combinations(lib):
    so = lib.load()
    buf = (C.c_float * 64)()
    ptr = C.cast(buf, C.c_void_p)
    inp = lib.SfmInputs()
    F = lib.SFM_FLAG_BORDER_PADDING
    # the explainability branch
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.2, 0.0, F)
    assert so.sfm_loss_forward(C.byref(d), C.byref(inp), ptr, None, ptr, None) == lib.SFM_E_UNSUPPORTED
    # debug dumps
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, F)
    dbg = lib.SfmDebug()
    assert so.sfm_loss_forward(C.byref(d), C.byref(inp), ptr, C.byref(dbg), ptr, None) == lib.SFM_E_UNSUPPORTED
    # image gradients
    d.flags = F | lib.SFM_FLAG_IMAGE_GRADS
    ig = lib.SfmImageGrads(ptr, ptr)
    grads = lib.SfmGrads()
    assert so.sfm_loss_forward_backward_images(C.byref(d), C.byref(inp), ptr, C.byref(grads), C.byref(ig), ptr,
                                               None) == lib.SFM_E_UNSUPPORTED
    # the host-buffer path
    d.flags = F
    ctx = C.c_void_p()
    assert so.sfm_host_ctx_create(C.byref(d), C.byref(ctx)) == lib.SFM_E_UNSUPPORTED
    # a supported combination gets as far as the inputs check
    assert so.sfm_loss_forward(C.byref(d), C.byref(inp), ptr, None, ptr, None) == lib.SFM_E_NULL_POINTER


def test_operator_options(lib):
    from sfm_learner_chainer_b200.functions import ViewSynthesisLoss
    for kw in (dict(image_grads=True), dict(exp_reg=0.2)):
        with pytest.raises(ValueError):
            ViewSynthesisLoss(border_padding=True, **kw)
    op = ViewSynthesisLoss(ssim_rate=0.15, border_padding=True, min_reprojection=True, full_res_multiscale=True)
    assert op._desc(2, 2, 64, 208).flags & lib.SFM_FLAG_BORDER_PADDING
    assert not ViewSynthesisLoss(ssim_rate=0.15)._desc(2, 2, 64, 208).flags & lib.SFM_FLAG_BORDER_PADDING
    with pytest.raises(ValueError):
        op.forward(None, None, None, None, None, debug=True)
