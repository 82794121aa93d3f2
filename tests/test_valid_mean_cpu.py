"""CPU checks of the valid-pixel-mean reference (tests/valid_mean_oracle.py) against SC-SfMLearner's compute_pairwise_loss
and mean_on_mask restated in torch fp64 (tests/torch_valid_mean_restatement.py) and against central differences, and of
the C ABI of sfm_loss_geometry_valid_mean (flag, struct layout, workspace size, argument errors that precede the device
check)."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from tests import geometry_oracle as GO
from tests import valid_mean_oracle as VM
from tests.test_geometry_cpu import make_case, _close
from tests.torch_valid_mean_restatement import torch_total_valid_mean

FLAGS = {'l1': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0), 'ssim': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.85)}


def bright_case(B, S, H, W, ns, seed, harsh, dtype=np.float32):
    """make_case with a target 2.5 times brighter, so that many L1 differences exceed 1 and are clamped."""
    d, sd = make_case(B, S, H, W, ns, seed, harsh, dtype)
    d['tgt'] = (d['tgt'] * dtype(2.5)).astype(dtype)
    return d, sd


def _torch(d, sd, cfg, self_mask, automask, groups, min_count):
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64)).requires_grad_(True)
    disps = [t(x) for x in d['disps']]
    srcd = [t(x) for x in sd]
    poses = t(d['poses'])
    K = t(d['intrinsics'])
    tot, geo = torch_total_valid_mean(torch.from_numpy(d['tgt'].astype(np.float64)),
                                      torch.from_numpy(d['src'].astype(np.float64)), K, disps, poses, srcd, cfg, 0.5,
                                      self_mask, automask, groups, min_count)
    tot.backward()
    return float(tot.detach()), float(geo.detach()), [x.grad.numpy() for x in disps], poses.grad.numpy(), [x.grad.numpy() for x in srcd]


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('harsh', [False, True])
@pytest.mark.parametrize('self_mask', [False, True])
@pytest.mark.parametrize('automask', [False, True])
def test_reference_matches_torch_autograd(flags, S, harsh, self_mask, automask):
    ns, B = 2, 2
    d, sd = bright_case(B, S, 24, 40, ns, 5100 + S + 10 * harsh, harsh, dtype=np.float64)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    groups = 2 if S == 3 else 1
    L, G = VM.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, geometry_reg=0.5,
                   self_mask=self_mask, automask=automask, groups=groups, min_count=0.0)
    tot, geo, gd, gp, gs = _torch(d, sd, cfg, self_mask, automask, groups, 0.0)
    np.testing.assert_allclose(L['total_loss'], tot, rtol=1e-6)
    np.testing.assert_allclose(L['exp_loss'], geo, rtol=1e-6)
    for s in range(ns):
        _close(G['gdisp'][s], gd[s], 'gdisp[%d]' % s, rtol=1e-5, atol_rel=1e-6)
        _close(G['gsrc_disp'][s], gs[s], 'gsrc_disp[%d]' % s, rtol=1e-5, atol_rel=1e-6)
    _close(G['gpose'], gp, 'gpose', rtol=1e-5, atol_rel=1e-6)
    # the case reaches clamped L1 differences, and the auto-mask drops some in-view pairs
    T = GO.geometry_terms(d['intrinsics'], d['disps'], d['poses'], sd, cfg)
    inb = T[0]['per'][0]['inb'].reshape(B, 24, 40)
    assert (np.abs(d['tgt'] - d['src'][:, 0]) > 1).any()
    if automask:
        assert (inb & ~L['valid_masks'][0][:, 0]).any()
    else:
        np.testing.assert_array_equal(L['valid_masks'][0][:, 0], inb)


def test_counts_and_groups():
    d, sd = bright_case(4, 2, 24, 40, 2, 5201, True)
    cfg = O.LossConfig(n_scales=2, **FLAGS['ssim'])
    L1, _ = VM.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, groups=1, min_count=0.0,
                    want_grads=False)
    L2, _ = VM.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, groups=2, min_count=0.0,
                    want_grads=False)
    for s in range(2):
        per_b = L1['valid_masks'][s].reshape(4, 2, -1).sum(-1)
        np.testing.assert_array_equal(L1['valid_counts'][s, :, 0], per_b.sum(0))
        np.testing.assert_array_equal(L2['valid_counts'][s, :, 0], per_b[0::2].sum(0))
        np.testing.assert_array_equal(L2['valid_counts'][s, :, 1], per_b[1::2].sum(0))
    # zero-weight snippets count nowhere
    L3, _ = VM.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, groups=1, min_count=0.0,
                    snippet_weights=np.array([1, 0, 1, 1], np.float32), want_grads=False)
    assert not L3['valid_masks'][0][1].any()
    np.testing.assert_array_equal(L3['valid_counts'][0, :, 0],
                                  L1['valid_counts'][0, :, 0] - L1['valid_masks'][0][1].reshape(2, -1).sum(-1))


def test_min_count_thresholds():
    """min_count just below / at 3 n and n switches the photometric and the geometry parts separately."""
    d, sd = make_case(2, 1, 24, 40, 1, 5301, False)
    cfg = O.LossConfig(n_scales=1, **FLAGS['l1'])
    run = lambda mc: VM.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, min_count=mc,
                             want_grads=False)[0]
    L0 = run(0.0)
    n = int(L0['valid_counts'][0, 0, 0])
    assert n > 0
    for mc, photo, geo in ((3 * n - 0.5, True, False), (3 * n, False, False), (n - 0.5, True, True), (n, True, False)):
        L = run(mc)
        assert (L['pixel_loss'] == L0['pixel_loss']) if photo else (L['pixel_loss'] == 0.0), mc
        assert (L['exp_loss'] == L0['exp_loss']) if geo else (L['exp_loss'] == 0.0), mc


@pytest.mark.parametrize('self_mask', [False, True])
def test_reference_central_differences(self_mask):
    """The whole-loss gradient of the fp64 reference against central differences, on a bright case (clamped pixels)
    with two groups, one of them below min_count for the photometric part.  (The harsh poses are covered against
    autograd above: there a step of 1e-6 can move a pixel across the view's edge and change a count.)"""
    ns, B, S = 1, 2, 2
    d, sd = bright_case(B, S, 16, 24, ns, 5401, False, dtype=np.float64)
    cfg = O.LossConfig(n_scales=ns, smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.85)
    L0, _ = VM.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, groups=2, min_count=0.0,
                    want_grads=False)
    cnt = L0['valid_counts'][0]                                   # (S, G)
    mc = float(3 * cnt[0, 0]) - 0.5 if 3 * cnt[0, 0] < 3 * cnt[0, 1] else float(3 * cnt[0, 1]) - 0.5
    mc = min(mc, float(3 * cnt.min()) + 0.5)                      # at least one (source, group) drops its photometric part
    masks = L0['valid_masks']

    def total(dd, ss):
        L, _ = VM.loss(dd['tgt'], dd['src'], dd['intrinsics'], dd['disps'], dd['poses'], ss, cfg, groups=2, min_count=mc,
                       self_mask=self_mask, masks=masks, want_grads=False)
        return L['total_loss']

    _, G = VM.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, groups=2, min_count=mc,
                   self_mask=self_mask, masks=masks)
    rs = np.random.RandomState(7)
    checks = []
    for _ in range(4):
        checks.append(('disps', (0, rs.randint(B), 0, rs.randint(16), rs.randint(24)), G['gdisp'][0]))
        checks.append(('src', (0, rs.randint(B), rs.randint(S), rs.randint(16), rs.randint(24)), G['gsrc_disp'][0]))
    for k in range(6):
        checks.append(('poses', (k % 2, k % 2, k), G['gpose']))
    for name, idx, g in checks:
        eps = 1e-6
        vals = []
        for sgn in (1, -1):
            dd = copy.deepcopy(d)
            ss = [x.copy() for x in sd]
            if name == 'disps':
                dd['disps'][idx[0]][idx[1:]] += sgn * eps
            elif name == 'src':
                ss[idx[0]][idx[1:]] += sgn * eps
            else:
                dd['poses'][idx] += sgn * eps
            vals.append(total(dd, ss))
        num = (vals[0] - vals[1]) / (2 * eps)
        ana = g[idx[1:]] if name in ('disps', 'src') else g[idx]
        assert abs(num - ana) <= 1e-5 * max(1.0, abs(num)) + 1e-4 * abs(num), (name, idx, num, ana)


@pytest.fixture
def lib():
    from sfm_learner_chainer_b200 import lib as L
    try:
        L.load()
    except ImportError:
        pytest.skip('libsfmloss.so not built')
    return L


def test_abi_flag_struct_and_workspace(lib):
    assert lib.SFM_FLAG_VALID_MEAN == 0x2000
    vp = C.sizeof(C.c_void_p)
    assert lib.SfmValidMean.automask.offset == 0
    assert lib.SfmValidMean.groups.offset == 4
    assert lib.SfmValidMean.min_count.offset == 8
    assert lib.SfmValidMean.masks.offset == 16
    assert lib.SfmValidMean.counts.offset == 16 + 4 * vp
    assert C.sizeof(lib.SfmValidMean) == 16 + 5 * vp
    so = lib.load()
    assert 'sfm_loss_geometry_valid_mean' in lib.SYMBOLS and so.sfm_loss_geometry_valid_mean is not None
    B, S, H, W, ns = 3, 2, 128, 416, 4
    G = lib.SFM_FLAG_GEOMETRY_CONSISTENCY
    d0 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, G)
    d1 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, G | lib.SFM_FLAG_VALID_MEAN)
    extra = sum(-(-B * S * (H >> s) * (W >> s) // 256) * 256 for s in range(ns)) + -(-ns * S * B * 4 // 256) * 256
    assert so.sfm_workspace_bytes(C.byref(d1)) - so.sfm_workspace_bytes(C.byref(d0)) == extra


def test_abi_argument_errors(lib):
    so = lib.load()
    buf = (C.c_float * 64)()
    ptr = C.cast(buf, C.c_void_p)
    GC, VF = lib.SFM_FLAG_GEOMETRY_CONSISTENCY, lib.SFM_FLAG_VALID_MEAN
    ge = lib.SfmGeometry()
    for s in range(4):
        ge.src_disps[s] = ptr
    ge.geometry_reg = 0.5

    def call(flags, groups=1, min_count=10000.0, exp_reg=0.0, B_global=0, peer=None, vm=True):
        d = lib.SfmDesc(2, 2, 64, 208, 4, B_global, 0.1, exp_reg, 0.0 if exp_reg else 0.15, flags)
        v = lib.SfmValidMean()
        v.automask, v.groups, v.min_count = 1, groups, min_count
        return so.sfm_loss_geometry_valid_mean(C.byref(d), C.byref(lib.SfmInputs()), None, C.byref(ge),
                                               C.byref(v) if vm else None, ptr, None, ptr, peer, None)

    assert call(GC) == lib.SFM_E_INVALID_DESC                                  # the flag sizes the workspace
    for g in (0, 3, -1):
        assert call(GC | VF, groups=g) == lib.SFM_E_INVALID_DESC
    for mc in (-1.0, float('nan'), float('inf')):
        assert call(GC | VF, min_count=mc) == lib.SFM_E_INVALID_DESC
    assert call(GC | VF, peer=ptr) == lib.SFM_E_UNSUPPORTED
    assert call(GC | VF, B_global=4) == lib.SFM_E_UNSUPPORTED
    assert call(VF) == lib.SFM_E_INVALID_DESC                                  # geometry consistency's flag
    assert call(GC | VF, exp_reg=0.2) == lib.SFM_E_UNSUPPORTED
    for f in (lib.SFM_FLAG_FULL_RES_MULTISCALE, lib.SFM_FLAG_BORDER_PADDING, lib.SFM_FLAG_MIN_REPROJECTION):
        assert call(GC | VF | f) == lib.SFM_E_UNSUPPORTED
    # vm == NULL is sfm_loss_geometry, which refuses what it refuses
    assert call(0, vm=False) == lib.SFM_E_INVALID_DESC
    assert call(GC, exp_reg=0.2, vm=False) == lib.SFM_E_UNSUPPORTED
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, VF)
    ctx = C.c_void_p()
    assert so.sfm_host_ctx_create(C.byref(d), C.byref(ctx)) == lib.SFM_E_UNSUPPORTED


def test_operator_argument_errors(lib):
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    with pytest.raises(ValueError):
        ViewSynthesisLoss(0.1, 0.0, 0.85, valid_mean=True)                  # needs geometry_consistency
    for kw in (dict(valid_min_count=-1.0), dict(valid_min_count=float('nan')), dict(count_groups=0), dict(B_global=8)):
        with pytest.raises(ValueError):
            ViewSynthesisLoss(0.1, 0.0, 0.85, geometry_consistency=True, valid_mean=True, **kw)
    op = ViewSynthesisLoss(0.1, 0.0, 0.85, geometry_consistency=True, valid_mean=True, count_groups=3)
    with pytest.raises(ValueError):
        op._valid_mean(lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.85, 0), None)   # G > B
