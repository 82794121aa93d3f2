"""-m "not gpu": per-pixel weights and per-pixel loss maps (sfm_loss_weighted).

The weighted reference (tests/pixel_oracle.py) is checked against the plain oracle bit for bit without weights and with
M = 1, its maps against torch fp64 autograd of an independent restatement with the weights as leaves (the map is
d total / d M), its weighted gdisp / gpose / glogits against central differences of its own weighted total, and M = 0
against the regularisers alone.  The C ABI
additions are checked for their symbol, struct size and argument errors without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests.pixel_oracle import sfm_loss_pixel, sfm_loss_pixel_raw
from tests.torch_pixel_restatement import torch_total_weighted

FLAGS = {
    'l1': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.0),
    'exp': dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
}


def _args(d):
    return d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits']


def pixel_weights(d, seed, null_scale=None, lo=-0.25, hi=1.0):
    """Per-pixel weights in [lo, hi] (some negative) shaped like the logits; scale `null_scale` is None (= 1)."""
    rs = np.random.RandomState(seed)
    return [None if s == null_scale else rs.uniform(lo, hi, l.shape).astype(l.dtype) for s, l in enumerate(d['logits'])]


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 2, 4])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_oracle_maps_match_torch_autograd(flags, S, ns, harsh):
    d = make_snippets(2, S, 32, 64, seed=90 + S + 10 * ns, n_scales=ns, harsh=harsh, dtype=np.float64)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    W = pixel_weights(d, 5 + S, null_scale=1 if ns > 1 else None)
    L, _ = sfm_loss_pixel(*_args(d), cfg, pixel_weights=W, want_grads=False)
    leaves = [torch.from_numpy(w if w is not None else np.ones_like(d['logits'][s])).requires_grad_(True)
              for s, w in enumerate(W)]
    tot = torch_total_weighted(d, cfg, leaves)
    tot.backward()
    r = cfg.ssim_rate
    np.testing.assert_allclose(tot.item(), (1 - r) * L['pixel_loss'] + r * L['ssim_loss'], rtol=1e-9, atol=1e-12)
    for s in range(ns):
        ref = leaves[s].grad.numpy()
        np.testing.assert_allclose(L['pixel_losses'][s], ref, rtol=1e-7, atol=1e-9 * np.abs(ref).max())


@pytest.mark.parametrize('flags', sorted(FLAGS))
def test_weighted_gradients_central_differences(flags):
    """gdisp, gpose and glogits of the weighted loss against fp64 central differences of the oracle's weighted total on
    sampled entries, skipping entries with a kink (|P - T|, the all-zero mask, a floor flip, the SSIM clip) in range."""
    d = make_snippets(1, 2, 32, 64, seed=17, n_scales=4, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=4, **FLAGS[flags])
    W = pixel_weights(d, 3, null_scale=2)
    _, G = sfm_loss_pixel(*_args(d), cfg, pixel_weights=W)

    def total(**over):
        a = dict(d, **over)
        return sfm_loss_pixel(a['tgt'], a['src'], a['intrinsics'], a['disps'], a['poses'], a['logits'], cfg, want_grads=False,
                              pixel_weights=W)[0]['total_loss']
    mid = total()
    rs = np.random.RandomState(4)
    eps = 1e-7
    checked = 0
    kinds = [('disps', 'gdisp'), ('poses', 'gpose')] + ([('logits', 'glogits')] if flags == 'exp' else [])
    for key, gkey in kinds:
        for _ in range(24):
            if key == 'poses':
                arr, ref, ix = d['poses'], G['gpose'], tuple(rs.randint(0, n) for n in d['poses'].shape)
                s = None
            else:
                s = rs.randint(0, 4)
                arr, ref = d[key][s], G[gkey][s]
                ix = tuple(rs.randint(0, n) for n in arr.shape)
            vals = []
            for sgn in (1, -1):
                a = arr.copy()
                a[ix] += sgn * eps
                if s is None:
                    vals.append(total(poses=a))
                else:
                    lst = list(d[key])
                    lst[s] = a
                    vals.append(total(**{key: lst}))
            if abs((vals[0] - mid) - (mid - vals[1])) > 1e-3 * abs(vals[0] - vals[1]) + 1e-15:
                continue
            fd = (vals[0] - vals[1]) / (2 * eps)
            assert abs(fd - ref[ix]) <= 1e-4 * abs(ref[ix]) + 1e-8, (key, s, ix, fd, ref[ix])
            checked += 1
    assert checked >= 20


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('ns', [1, 4])
def test_unit_weights_equal_the_plain_oracle_and_maps_sum_to_the_loss(flags, ns):
    d = make_snippets(2, 2, 32, 64, seed=30 + ns, n_scales=ns, harsh=True)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L0, G0, _ = O.sfm_loss(*_args(d), cfg, want_intrinsics_grad=True)
    ones = [np.ones_like(l) for l in d['logits']]
    L1, G1 = sfm_loss_pixel(*_args(d), cfg, want_intrinsics_grad=True, pixel_weights=ones)
    for k in O.LOSS_KEYS:
        assert L1[k] == L0[k], k
    for k in ('gdisp', 'glogits'):
        if G0[k] is not None:
            for a, b in zip(G1[k], G0[k]):
                np.testing.assert_array_equal(a, b)
    for k in ('gpose', 'dP', 'gintrinsics'):
        np.testing.assert_array_equal(G1[k], G0[k])
    # sum M * map = (1 - r) pixel + r ssim, for unit and for random weights
    r = cfg.ssim_rate
    assert np.isclose(sum(m.sum() for m in L1['pixel_losses']), (1 - r) * L0['pixel_loss'] + r * L0['ssim_loss'], rtol=1e-6)
    W = pixel_weights(d, 9)
    Lw, _ = sfm_loss_pixel(*_args(d), cfg, want_grads=False, pixel_weights=W)
    for a, b in zip(Lw['pixel_losses'], L1['pixel_losses']):
        np.testing.assert_array_equal(a, b)                  # the map does not depend on M
    got = sum((w.astype(np.float64) * m).sum() for w, m in zip(W, Lw['pixel_losses']))
    assert np.isclose(got, (1 - r) * Lw['pixel_loss'] + r * Lw['ssim_loss'], rtol=1e-5)


@pytest.mark.parametrize('flags', sorted(FLAGS))
def test_zero_weights_leave_the_regularisers(flags):
    d = make_snippets(2, 2, 32, 64, seed=51, n_scales=4, harsh=True)
    cfg = O.LossConfig(n_scales=4, **FLAGS[flags])
    zeros = [np.zeros_like(l) for l in d['logits']]
    L, G = sfm_loss_pixel(*_args(d), cfg, pixel_weights=zeros)
    # other images: only the photometric terms could see them
    L0, G0 = sfm_loss_pixel(d['tgt'], d['src'][:, ::-1].copy(), *_args(d)[2:], cfg, pixel_weights=zeros)
    assert L['pixel_loss'] == 0 and L['ssim_loss'] == 0
    assert L['smooth_loss'] == L0['smooth_loss'] and L['exp_loss'] == L0['exp_loss']
    assert L['total_loss'] == pytest.approx(L['smooth_loss'] + L['exp_loss'], rel=1e-12)
    assert not np.any(G['gpose'])
    for a, b in zip(G['gdisp'], G0['gdisp']):                 # the smoothness gradient alone
        np.testing.assert_array_equal(a, b)
    if flags == 'exp':
        for s, g in enumerate(G['glogits']):                  # the regulariser alone: -exp_reg (1 - sigma) / (B h w)
            sg = 1 / (1 + np.exp(-d['logits'][s].astype(np.float64)))
            h, w = g.shape[2:]
            np.testing.assert_allclose(g, -cfg.exp_reg * (1 - sg) / (2 * h * w), rtol=1e-5)


@pytest.mark.parametrize('flags', sorted(FLAGS) + ['edge'])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('dtype', [np.float32, np.float64])
def test_reference_without_weights_is_the_oracle_bit_for_bit(flags, ns, dtype):
    """The weighted reference restates the oracle's loss loop; without weights it must do the oracle's arithmetic."""
    edge = flags == 'edge'
    d = make_snippets(2, 2, 32, 64, seed=60 + ns, n_scales=ns, harsh=True, dtype=dtype)
    cfg = O.LossConfig(n_scales=ns, edge_aware_smooth=edge, **FLAGS['ssim' if edge else flags])
    L0, G0, _ = O.sfm_loss(*_args(d), cfg, want_intrinsics_grad=True)
    L, G = sfm_loss_pixel(*_args(d), cfg, want_intrinsics_grad=True)
    for k in O.LOSS_KEYS:
        assert L[k] == L0[k], k
    assert [m.shape for m in L['pixel_losses']] == [(2, 2, 32 >> s, 64 >> s) for s in range(ns)]
    for k in ('gpose', 'dT', 'dP', 'gintrinsics'):
        np.testing.assert_array_equal(G[k], G0[k], err_msg=k)
    for k in ('gdisp', 'glogits'):
        if G0[k] is not None:
            for a, b in zip(G[k], G0[k]):
                np.testing.assert_array_equal(a, b, err_msg=k)


def test_raw_reference_without_weights_is_the_oracle_bit_for_bit():
    from sfm_learner_chainer_b200.synthetic import make_raw_seam
    d = make_snippets(2, 2, 32, 64, seed=66, n_scales=4, harsh=True)
    raw_disps, raw_poses = make_raw_seam(d, (1, 4), seed=67)
    cfg = O.LossConfig(n_scales=4, **FLAGS['ssim'])
    args = (d['tgt'], d['src'], d['intrinsics'], raw_disps, raw_poses, d['logits'])
    L0, G0, _ = O.sfm_loss_raw(*args, cfg, raw_disp_scales=0xF, raw_pose=True)
    L, G = sfm_loss_pixel_raw(*args, cfg, raw_disp_scales=0xF, raw_pose=True)
    for k in O.LOSS_KEYS:
        assert L[k] == L0[k], k
    np.testing.assert_array_equal(G['gpose'], G0['gpose'])
    for a, b in zip(G['gdisp'], G0['gdisp']):
        np.testing.assert_array_equal(a, b)


@pytest.fixture
def lib():
    from sfm_learner_chainer_b200 import lib as L
    try:
        L.load()
    except ImportError:
        pytest.skip('libsfmloss.so not built')
    return L


def test_abi_symbol_and_struct(lib):
    so = lib.load()
    assert 'sfm_loss_weighted' in lib.SYMBOLS and so.sfm_loss_weighted is not None
    assert C.sizeof(lib.SfmPixelTerms) == 2 * 4 * C.sizeof(C.c_void_p)


def test_abi_argument_errors(lib):
    so = lib.load()
    buf = (C.c_float * 64)()
    ptr = C.cast(buf, C.c_void_p)
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_IMAGE_GRADS)
    pix = lib.SfmPixelTerms()
    pix.weights[0] = ptr
    ig = lib.SfmImageGrads(ptr, None)
    # per-pixel terms with image gradients
    rc = so.sfm_loss_weighted(C.byref(d), C.byref(lib.SfmInputs()), None, C.byref(pix), ptr, C.byref(lib.SfmGrads()),
                              C.byref(ig), ptr, None, None)
    assert rc == lib.SFM_E_UNSUPPORTED
    pix = lib.SfmPixelTerms()
    pix.losses[3] = ptr
    rc = so.sfm_loss_weighted(C.byref(d), C.byref(lib.SfmInputs()), None, C.byref(pix), ptr, C.byref(lib.SfmGrads()),
                              C.byref(ig), ptr, None, None)
    assert rc == lib.SFM_E_UNSUPPORTED
    # snippet members without their flag: the error sfm_loss_snippets gives
    d.flags = 0
    terms = lib.SfmSnippetTerms(ptr, None)
    rc = so.sfm_loss_weighted(C.byref(d), C.byref(lib.SfmInputs()), C.byref(terms), C.byref(pix), ptr, None, None, ptr,
                              None, None)
    assert rc == lib.SFM_E_INVALID_DESC
    # losses_out is required
    rc = so.sfm_loss_weighted(C.byref(d), C.byref(lib.SfmInputs()), None, C.byref(pix), None, None, None, ptr, None, None)
    assert rc == lib.SFM_E_NULL_POINTER
    # a member of a scale >= n_scales is ignored: with image gradients this is the plain combination, which gets as far
    # as the inputs check here
    d = lib.SfmDesc(2, 2, 64, 208, 2, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_IMAGE_GRADS)
    rc = so.sfm_loss_weighted(C.byref(d), C.byref(lib.SfmInputs()), None, C.byref(pix), ptr, C.byref(lib.SfmGrads()),
                              C.byref(ig), ptr, None, None)
    assert rc == lib.SFM_E_NULL_POINTER
