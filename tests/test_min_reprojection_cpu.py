"""-m "not gpu": per-pixel minimum reprojection with auto-masking (sfm_loss_min_reprojection).

The reference (tests/min_reprojection_oracle.py) is checked against torch fp64 autograd of an independent restatement
(torch.min over the stacked errors), its gradients against central differences of its own total away from ties, and its
selection rules on hand-made cases.  The C ABI additions are checked for their symbol, struct layout, workspace size and
argument errors without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import min_reprojection_oracle as MR
from tests.torch_min_reprojection_restatement import torch_min_reprojection

FLAGS = {
    'l1': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.15),
    'ssim_only': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=1.0),
}


def _args(d):
    return d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses']


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 2, 4])
@pytest.mark.parametrize('automask', [True, False])
def test_oracle_matches_torch_autograd(flags, S, automask):
    d = make_snippets(2, S, 32, 64, seed=140 + S, n_scales=2, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=2, **FLAGS[flags])
    L, G = MR.sfm_loss_min_reprojection(*_args(d), cfg, automask=automask)
    disps = [torch.from_numpy(x).requires_grad_(True) for x in d['disps']]
    poses = torch.from_numpy(d['poses']).requires_grad_(True)
    phot, pixel, ssim, sels = torch_min_reprojection(d, cfg, disps, poses, automask=automask)
    for s in range(2):
        np.testing.assert_array_equal(L['selection'][s], sels[s].numpy())
    counts = np.bincount(np.concatenate([x.ravel() for x in L['selection']]) + 2, minlength=2 + S)
    assert counts[2:].min() > 0 and (counts[1] > 0) == automask and counts[0] > 0      # every kind of outcome occurs
    r = cfg.ssim_rate
    np.testing.assert_allclose(L['pixel_loss'], pixel.item(), rtol=1e-9)
    np.testing.assert_allclose(L['ssim_loss'], ssim.item(), rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose(L['total_loss'], phot.item(), rtol=1e-9)
    assert np.isclose(phot.item(), (1 - r) * pixel.item() + r * ssim.item(), rtol=1e-12)
    phot.backward()
    for s in range(2):
        ref = disps[s].grad.numpy()
        np.testing.assert_allclose(G['gdisp'][s], ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())
    ref = poses.grad.numpy()
    np.testing.assert_allclose(G['gpose'], ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())


@pytest.mark.parametrize('flags', ['l1', 'ssim'])
def test_gradients_central_differences(flags):
    """gdisp and gpose against fp64 central differences of the oracle's total (selection recomputed at every point) on
    sampled entries, skipping entries with a kink (a selection flip, |P - T|, the mask, a floor flip, the clip) in range."""
    cfg = O.LossConfig(n_scales=4, **dict(FLAGS[flags], smooth_reg=0.1))
    d = make_snippets(1, 2, 32, 64, seed=171, n_scales=4, harsh=True, dtype=np.float64)
    _, G = MR.sfm_loss_min_reprojection(*_args(d), cfg)

    def total(**over):
        a = dict(d, **over)
        return MR.sfm_loss_min_reprojection(*_args(a), cfg, want_grads=False)[0]['total_loss']
    mid = total()
    rs = np.random.RandomState(8)
    eps = 1e-7
    checked = 0
    for key, gkey in (('disps', 'gdisp'), ('poses', 'gpose')):
        for _ in range(24):
            if key == 'poses':
                arr, ref, s = d['poses'], G['gpose'], None
            else:
                s = rs.randint(0, 4)
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


def test_selection_rules_by_hand():
    e = np.array([[[[0.5]], [[0.2]], [[0.2]], [[0.0]]]])                 # (B=1, S=4, 1, 1)
    masked = np.array([[[[False]], [[False]], [[False]], [[True]]]])
    e_id = np.full((1, 4, 1, 1), 1.0)
    # a masked source never wins, not even with error 0; equal errors go to the lowest index
    assert MR.select(e, masked, e_id, automask=False)[0, 0, 0] == 1
    assert MR.select(e, masked, e_id, automask=True)[0, 0, 0] == 1
    # auto-masking: e_i* >= min e_id drops the pixel (the identity minimum may come from any source, masked ones too),
    # a strict < keeps it
    e_id[0, 3] = 0.2
    assert MR.select(e, masked, e_id, automask=True)[0, 0, 0] == -1
    e_id[0, 3] = np.nextafter(0.2, 1.0)
    assert MR.select(e, masked, e_id, automask=True)[0, 0, 0] == 1
    # no candidate: -2, with or without auto-masking
    allm = np.ones_like(masked)
    assert MR.select(e, allm, e_id, automask=False)[0, 0, 0] == -2
    assert MR.select(e, allm, np.zeros_like(e_id), automask=True)[0, 0, 0] == -2


def test_identical_source_is_auto_masked_everywhere():
    """A source equal to the target, warped with a non-zero pose: its identity error is 0 at every pixel, so every pixel
    with a candidate is auto-masked and the photometric loss and its gradients vanish."""
    d = make_snippets(2, 2, 32, 64, seed=181, n_scales=4, dtype=np.float64)
    d['src'][:, 1] = d['tgt']
    cfg = O.LossConfig(n_scales=4, smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.15)
    L, G = MR.sfm_loss_min_reprojection(*_args(d), cfg)
    assert all(np.all(s < 0) for s in L['selection'])
    assert L['total_loss'] == 0 and L['pixel_loss'] == 0 and L['ssim_loss'] == 0
    assert not np.any(G['gpose']) and not any(np.any(g) for g in G['gdisp'])


def test_single_source_without_automask_is_the_unit_weighted_loss():
    from tests.pixel_oracle import sfm_loss_pixel
    d = make_snippets(2, 1, 32, 64, seed=191, n_scales=4, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=4, smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15)
    L, G = MR.sfm_loss_min_reprojection(*_args(d), cfg, automask=False)
    L0, G0 = sfm_loss_pixel(*_args(d), None, cfg)
    for k in O.LOSS_KEYS:
        assert L[k] == pytest.approx(L0[k], rel=1e-12, abs=1e-15), k
    np.testing.assert_allclose(G['gpose'], G0['gpose'], rtol=1e-10, atol=1e-15)


@pytest.fixture
def lib():
    from sfm_learner_chainer_b200 import lib as L
    try:
        L.load()
    except ImportError:
        pytest.skip('libsfmloss.so not built')
    return L


def test_abi_symbol_struct_and_workspace(lib):
    so = lib.load()
    assert 'sfm_loss_min_reprojection' in lib.SYMBOLS and so.sfm_loss_min_reprojection is not None
    assert C.sizeof(lib.SfmMinReprojection) == 8 + 4 * C.sizeof(C.c_void_p)
    assert lib.SfmMinReprojection.selection.offset == 8
    d = lib.SfmDesc(2, 3, 64, 208, 4, 0, 0.1, 0.0, 0.15, 0)
    n0 = so.sfm_workspace_bytes(C.byref(d))
    d.flags = lib.SFM_FLAG_MIN_REPROJECTION
    n1 = so.sfm_workspace_bytes(C.byref(d))
    assert n1 - n0 >= 4 * 2 * 3 * sum((64 >> s) * (208 >> s) for s in range(4))


def test_abi_argument_errors(lib):
    so = lib.load()
    buf = (C.c_float * 64)()
    ptr = C.cast(buf, C.c_void_p)
    inp = lib.SfmInputs()
    mr = lib.SfmMinReprojection(1, 0)

    def call(d, mr_=C.byref(mr), losses=ptr, terms=None, grads=None):
        return so.sfm_loss_min_reprojection(C.byref(d), C.byref(inp), terms, mr_, losses, grads, ptr, None, None)
    F = lib.SFM_FLAG_MIN_REPROJECTION
    # the workspace flag is required
    assert call(lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, 0)) == lib.SFM_E_INVALID_DESC
    # ssim_rate outside [0, 1]
    for rate in (-0.1, 1.5, float('inf')):
        assert call(lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, rate, F)) == lib.SFM_E_INVALID_DESC
    # the explainability branch
    assert call(lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.2, 0.0, F)) == lib.SFM_E_UNSUPPORTED
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, F)
    # NULL pointers
    assert call(d, mr_=None) == lib.SFM_E_NULL_POINTER
    assert call(d, losses=None) == lib.SFM_E_NULL_POINTER
    assert call(d) == lib.SFM_E_NULL_POINTER                         # the inputs hold NULL images
    # reserved_ must be 0
    bad = lib.SfmMinReprojection(1, 7)
    assert call(d, mr_=C.byref(bad)) == lib.SFM_E_INVALID_DESC
    # snippet members without their flag
    terms = lib.SfmSnippetTerms(ptr, None)
    assert call(d, terms=C.byref(terms)) == lib.SFM_E_INVALID_DESC
    # the edge values of ssim_rate are accepted (the call gets as far as the inputs check)
    for rate in (0.0, 1.0):
        assert call(lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, rate, F)) == lib.SFM_E_NULL_POINTER


def test_operator_argument_errors(lib):
    from sfm_learner_chainer_b200.functions import ViewSynthesisLoss
    for kw in (dict(image_grads=True), dict(pixel_terms=True), dict(exp_reg=0.2), dict(ssim_rate=1.5)):
        with pytest.raises(ValueError):
            ViewSynthesisLoss(min_reprojection=True, **kw)
    op = ViewSynthesisLoss(ssim_rate=0.15, min_reprojection=True)
    assert op.automask
    assert not ViewSynthesisLoss(min_reprojection=True, automask=False).automask
