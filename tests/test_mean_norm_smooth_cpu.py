"""-m "not gpu": the mean-normalised smoothness (SFM_FLAG_MEAN_NORM_SMOOTH) and Monodepth2's edge weight
(SFM_FLAG_EDGE_MEAN_ABS).

The reference of tests/mean_norm_smooth_oracle.py (gradients from the homogeneity identity) against torch fp64 autograd of
the literal restatement (tests/torch_mean_norm_smooth_restatement.py) and against central differences, its properties,
its agreement with the oracle with both flags off, the C ABI additions without a device, and the Python options."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import mean_norm_smooth_oracle as MN
from tests.pixel_oracle import sfm_loss_pixel
from tests.torch_mean_norm_smooth_restatement import torch_smoothness

KINDS = {'second': {}, 'edge': dict(edge_aware_smooth=True), 'edge_mean_abs': dict(edge_aware_smooth=True)}


def _cfg(kind, n_scales=4, B_global=None):
    return O.LossConfig(smooth_reg=0.1, n_scales=n_scales, B_global=B_global, **KINDS[kind])


@pytest.mark.parametrize('kind', sorted(KINDS))
@pytest.mark.parametrize('mean_norm', [True, False])
@pytest.mark.parametrize('variant', ['plain', 'raw', 'B_global', 'weights'])
def test_reference_matches_torch_autograd(kind, mean_norm, variant):
    """36 x 52 is not a multiple of 8."""
    d = make_snippets(3, 2, 36, 52, seed=710, n_scales=4, dtype=np.float64)
    raw = 0b1011 if variant == 'raw' else 0
    rs = np.random.RandomState(711)
    disps = [rs.standard_normal(x.shape) for x in d['disps']] if raw else d['disps']
    disps = [x if (raw >> s) & 1 else d['disps'][s] for s, x in enumerate(disps)]
    Bg = 7 if variant == 'B_global' else None
    wb = np.array([1.5, 0.0, -0.75]) if variant == 'weights' else None
    cfg = _cfg(kind, B_global=Bg)
    ema = kind == 'edge_mean_abs'
    loss, rows, g = MN.smoothness(d['tgt'], disps, cfg, raw, mean_norm, ema, snippet_weights=wb)
    xt = [torch.from_numpy(x).requires_grad_(True) for x in disps]
    tl, trows = torch_smoothness(torch.from_numpy(d['tgt']), xt, 0.1, Bg, edge=cfg.edge_aware_smooth, edge_mean_abs=ema,
                                 mean_norm=mean_norm, raw_disp_scales=raw, snippet_weights=wb)
    tl.backward()
    assert np.isclose(loss, tl.item(), rtol=1e-10, atol=0)
    np.testing.assert_allclose(rows, trows.detach().numpy(), rtol=1e-10, atol=0)
    for s in range(4):
        ref = xt[s].grad.numpy()
        np.testing.assert_allclose(g[s], ref, rtol=1e-10, atol=1e-10 * np.abs(ref).max(), err_msg='gdisp[%d]' % s)


@pytest.mark.parametrize('kind', sorted(KINDS))
def test_gradients_central_differences(kind):
    d = make_snippets(2, 2, 24, 40, seed=720, n_scales=3, dtype=np.float64)
    cfg = _cfg(kind, n_scales=3)
    ema = kind == 'edge_mean_abs'
    f = lambda dd: MN.smoothness(d['tgt'], dd, cfg, 0, True, ema, want_grads=False)[0]
    _, _, g = MN.smoothness(d['tgt'], d['disps'], cfg, 0, True, ema)
    rs = np.random.RandomState(721)
    eps = 1e-6
    for s in range(3):
        for _ in range(12):
            idx = tuple(rs.randint(n) for n in d['disps'][s].shape)
            dp = [x.copy() for x in d['disps']]
            dm = [x.copy() for x in d['disps']]
            dp[s][idx] += eps
            dm[s][idx] -= eps
            fd = (f(dp) - f(dm)) / (2 * eps)
            assert abs(fd - g[s][idx]) <= 1e-6 * max(1.0, abs(g[s][idx])) + 1e-7, (s, idx, fd, g[s][idx])


@pytest.mark.parametrize('kind', sorted(KINDS))
def test_scale_invariance_and_euler(kind):
    """d_b -> alpha_b d_b leaves the normalised term unchanged up to the epsilon, and sum_j g_j d_j ~ 0 (Euler)."""
    d = make_snippets(3, 2, 36, 52, seed=730, n_scales=4, dtype=np.float64)
    cfg = _cfg(kind)
    ema = kind == 'edge_mean_abs'
    loss, rows, g = MN.smoothness(d['tgt'], d['disps'], cfg, 0, True, ema)
    alpha = np.array([0.25, 3.0, 40.0])
    scaled = [x * alpha[:, None, None, None] for x in d['disps']]
    loss2, rows2, _ = MN.smoothness(d['tgt'], scaled, cfg, 0, True, ema)
    np.testing.assert_allclose(rows2, rows, rtol=1e-5)
    for s in range(4):
        dot = np.sum(g[s] * d['disps'][s], axis=(1, 2, 3))
        scale = np.sum(np.abs(g[s] * d['disps'][s]), axis=(1, 2, 3))
        assert np.all(np.abs(dot) <= 1e-5 * scale), (s, dot, scale)


@pytest.mark.parametrize('kind', ['second', 'edge'])
def test_flags_off_reproduce_the_oracle(kind):
    """Without either flag the term is the oracle's: added to the photometric reference run with smooth_reg = 0 it gives
    the oracle's losses and gradients (to the association of the fp64 sums)."""
    d = make_snippets(2, 2, 64, 208, seed=740, n_scales=4)
    cfg = _cfg(kind)
    cfg.ssim_rate = 0.15
    args = (d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'])
    L, G, _ = O.sfm_loss(*args, None, cfg)
    cfg0 = O.LossConfig(ssim_rate=0.15, n_scales=4)
    L0, G0 = sfm_loss_pixel(*args, None, cfg0)
    L1, G1 = MN.add_smoothness(L0, G0, d['tgt'], d['disps'], cfg, mean_norm=False)
    np.testing.assert_allclose(O.losses_vec(L1), O.losses_vec(L), rtol=1e-12, atol=1e-15)
    for s in range(4):
        np.testing.assert_allclose(G1['gdisp'][s], G['gdisp'][s].astype(np.float64), rtol=1e-6,
                                   atol=1e-6 * np.abs(G['gdisp'][s]).max())


def _smooth_tasks(B, ns, H, W):
    """sfm_smooth_plan: the number of second-order smoothness tasks the workspace holds one loss for."""
    hseg = 64
    while True:
        n = sum(B * (((W >> s) + 27) // 28) * (((H >> s) + hseg - 1) // hseg) for s in range(ns))
        if n >= 148 * 4 * 8 or hseg <= 8:
            return n
        hseg >>= 1


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sfm_learner_chainer_b200 import lib as L
    return L


def test_flag_values_and_workspace(lib):
    so = lib.load()
    assert lib.SFM_FLAG_MEAN_NORM_SMOOTH == 0x100 and lib.SFM_FLAG_EDGE_MEAN_ABS == 0x200
    mn, snip = lib.SFM_FLAG_MEAN_NORM_SMOOTH, lib.SFM_FLAG_SNIPPET_TERMS
    al = lambda n: (n + 255) // 256 * 256
    ws = lambda *a: so.sfm_workspace_bytes(C.byref(lib.SfmDesc(*a)))
    for B, S, H, W, ns in ((4, 2, 128, 416, 4), (3, 2, 36, 52, 4), (64, 2, 256, 832, 4), (1, 2, 64, 208, 1)):
        base = (B, S, H, W, ns, 0, 0.1, 0.0, 0.15)
        n0 = ws(*base, 0)
        assert n0 > 0
        assert ws(*base, lib.SFM_FLAG_EDGE_AWARE_SMOOTH | lib.SFM_FLAG_EDGE_MEAN_ABS) == n0     # the edge weight sizes nothing
        slots = 2 * al(B * ns * 32 * 4) + al(B * 4)
        assert ws(*base, mn | snip) - ws(*base, snip) == slots
        assert ws(*base, mn) - n0 == slots + al(_smooth_tasks(B, ns, H, W) * 4)


def test_argument_errors(lib):
    so = lib.load()
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_EDGE_MEAN_ABS)
    assert so.sfm_workspace_bytes(C.byref(d)) == 0
    inp = lib.SfmInputs()
    assert so.sfm_loss_forward(C.byref(d), C.byref(inp), C.c_void_p(256), None, C.c_void_p(256), None) == lib.SFM_E_INVALID_DESC
    assert b'EDGE_MEAN_ABS' in so.sfm_last_error()
    ctx = C.c_void_p()
    for flags in (lib.SFM_FLAG_MEAN_NORM_SMOOTH, lib.SFM_FLAG_EDGE_AWARE_SMOOTH | lib.SFM_FLAG_EDGE_MEAN_ABS):
        d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, flags)
        assert so.sfm_host_ctx_create(C.byref(d), C.byref(ctx)) == lib.SFM_E_UNSUPPORTED
        assert b'MEAN' in so.sfm_last_error()


def test_python_options(lib):
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    with pytest.raises(ValueError, match='edge_mean_abs needs edge_aware_smooth'):
        ViewSynthesisLoss(0.1, 0.0, 0.15, edge_mean_abs=True)
    with pytest.raises(ValueError, match='image_grads'):
        ViewSynthesisLoss(0.1, 0.0, 0.15, edge_aware_smooth=True, edge_mean_abs=True, image_grads=True)
    op = ViewSynthesisLoss(0.1, 0.0, 0.15, edge_aware_smooth=True, edge_mean_abs=True, mean_norm_smooth=True)
    desc = op._desc(2, 2, 64, 208)
    assert desc.flags & lib.SFM_FLAG_MEAN_NORM_SMOOTH and desc.flags & lib.SFM_FLAG_EDGE_MEAN_ABS
    assert not ViewSynthesisLoss(0.1, 0.0, 0.15)._desc(2, 2, 64, 208).flags & (lib.SFM_FLAG_MEAN_NORM_SMOOTH | lib.SFM_FLAG_EDGE_MEAN_ABS)
