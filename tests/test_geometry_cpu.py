"""CPU checks of the geometry-consistency reference (tests/geometry_oracle.py) against an independent torch fp64
restatement (tests/torch_geometry_restatement.py) and against central differences, and of the C ABI of
sfm_loss_geometry (flag, struct layout, workspace size, argument errors that precede the device check)."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import geometry_oracle as GO
from tests.torch_geometry_restatement import torch_total_geometry


def make_case(B, S, H, W, ns, seed, harsh, dtype=np.float32):
    """Snippets and source disparities.  harsh: wide poses, and source 0 moves half a unit forward, so that near points
    lie behind its camera and some of them still project into view (z' < 0, z' + D' <= 0) while others leave it."""
    d = make_snippets(B, S, H, W, seed=seed, n_scales=ns, harsh=harsh, dtype=dtype)
    if harsh:
        d['poses'][:, 0, 5] -= dtype(0.5)
    sd = [x.astype(dtype) for x in GO.make_src_disps(B, S, H, W, ns, seed + 7)]
    return d, sd


FLAGS = {'l1': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0), 'ssim': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.15)}


def _torch_grads(d, sd, cfg, reg, self_mask):
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64)).requires_grad_(True)
    disps = [t(x) for x in d['disps']]
    srcd = [t(x) for x in sd]
    poses = t(d['poses'])
    K = t(d['intrinsics'])
    tot, geo = torch_total_geometry(torch.from_numpy(d['tgt'].astype(np.float64)), torch.from_numpy(d['src'].astype(np.float64)),
                                    K, disps, poses, srcd, cfg, reg, self_mask)
    tot.backward()
    return float(tot.detach()), float(geo.detach()), [x.grad.numpy() for x in disps], poses.grad.numpy(), [x.grad.numpy() for x in srcd], K.grad.numpy()


def _close(got, ref, what, rtol=2e-3, atol_rel=2e-4):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    atol = atol_rel * float(np.max(np.abs(ref))) + 1e-30
    bad = np.abs(got - ref) > atol + rtol * np.abs(ref)
    # fp32 reference vs fp64 restatement: a pixel whose in-view flag or clip side flips between the two is allowed
    assert bad.mean() < 2e-3, '%s: %d / %d off, max err %.3e (max |ref| %.3e)' % (
        what, int(bad.sum()), bad.size, float(np.max(np.abs(got - ref))), float(np.max(np.abs(ref))))


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('harsh', [False, True])
@pytest.mark.parametrize('self_mask', [False, True])
def test_reference_matches_torch_autograd(flags, S, harsh, self_mask):
    ns = 2
    d, sd = make_case(2, S, 24, 40, ns, 3100 + S + 10 * harsh, harsh)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L, G = GO.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, geometry_reg=0.5,
                   self_mask=self_mask, want_intrinsics_grad=True)
    tot, geo, gd, gp, gs, gk = _torch_grads(d, sd, cfg, 0.5, self_mask)
    np.testing.assert_allclose(L['total_loss'], tot, rtol=1e-4)
    np.testing.assert_allclose(L['exp_loss'], geo, rtol=1e-4)
    for s in range(ns):
        _close(G['gdisp'][s], gd[s], 'gdisp[%d]' % s)
        _close(G['gsrc_disp'][s], gs[s], 'gsrc_disp[%d]' % s)
    _close(G['gpose'], gp, 'gpose', rtol=1e-3, atol_rel=1e-3)
    _close(G['gintrinsics'], gk, 'gintrinsics', rtol=1e-3, atol_rel=1e-3)
    if harsh:
        # the harsh case reaches the branches the definition singles out
        T = GO.geometry_terms(d['intrinsics'], d['disps'], d['poses'], sd, cfg)
        r = T[0]['per'][0]
        assert (r['inb'] & (r['c'] <= 0)).any(), 'no in-view pair with z\' + D\' <= 0'
        assert (~r['inb']).any(), 'no pixel leaves the view'


@pytest.mark.parametrize('self_mask', [False, True])
def test_reference_central_differences(self_mask):
    """The whole-loss gradient of the fp64 reference against central differences at a few entries of every input."""
    ns = 1
    d, sd = make_case(1, 2, 16, 24, ns, 3301, False, dtype=np.float64)
    cfg = O.LossConfig(n_scales=ns, smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.15)

    def total(dd, ss):
        L, _ = GO.loss(dd['tgt'], dd['src'], dd['intrinsics'], dd['disps'], dd['poses'], ss, cfg, geometry_reg=0.5,
                       self_mask=self_mask, want_grads=False)
        return L['total_loss']

    _, G = GO.loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], sd, cfg, geometry_reg=0.5,
                   self_mask=self_mask, want_intrinsics_grad=True)
    rs = np.random.RandomState(5)
    checks = []
    for _ in range(4):
        checks.append(('disps', (0, 0, 0, rs.randint(16), rs.randint(24)), G['gdisp'][0]))
        checks.append(('src', (0, 0, rs.randint(2), rs.randint(16), rs.randint(24)), G['gsrc_disp'][0]))
    for k in range(6):
        checks.append(('poses', (0, k % 2, k), G['gpose']))
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
    assert lib.SFM_FLAG_GEOMETRY_CONSISTENCY == 0x1000
    vp = C.sizeof(C.c_void_p)
    assert C.sizeof(lib.SfmGeometry) == 3 * 4 * vp + 8
    assert lib.SfmGeometry.geometry_reg.offset == 3 * 4 * vp
    assert lib.SfmGeometry.self_mask.offset == 3 * 4 * vp + 4
    so = lib.load()
    assert 'sfm_loss_geometry' in lib.SYMBOLS and so.sfm_loss_geometry is not None
    B, S, H, W, ns = 3, 2, 128, 416, 4
    d0 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, 0)
    d1 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_GEOMETRY_CONSISTENCY)
    n0, n1 = so.sfm_workspace_bytes(C.byref(d0)), so.sfm_workspace_bytes(C.byref(d1))
    planes = 0
    for s in range(ns):
        planes += -(-B * S * (H >> s) * (W >> s) * 4 // 256) * 256
    assert n1 - n0 == 2 * planes
    # the other sizing flags are unchanged by it
    d2 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_SNIPPET_TERMS)
    d3 = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, lib.SFM_FLAG_SNIPPET_TERMS | lib.SFM_FLAG_GEOMETRY_CONSISTENCY)
    assert so.sfm_workspace_bytes(C.byref(d3)) - so.sfm_workspace_bytes(C.byref(d2)) == 2 * planes


def test_abi_argument_errors(lib):
    so = lib.load()
    buf = (C.c_float * 64)()
    ptr = C.cast(buf, C.c_void_p)
    G = lib.SFM_FLAG_GEOMETRY_CONSISTENCY
    ge = lib.SfmGeometry()
    for s in range(4):
        ge.src_disps[s] = ptr
    ge.geometry_reg = 0.5

    def call(flags, geo=ge, exp_reg=0.0, ns=4, terms=None, losses=ptr):
        d = lib.SfmDesc(2, 2, 64, 208, ns, 0, 0.1, exp_reg, 0.0 if exp_reg else 0.15, flags)
        return so.sfm_loss_geometry(C.byref(d), C.byref(lib.SfmInputs()), terms, C.byref(geo) if geo is not None else None,
                                    losses, None, ptr, None, None)

    assert call(0) == lib.SFM_E_INVALID_DESC                                   # the flag sizes the workspace
    assert call(G, exp_reg=0.2) == lib.SFM_E_UNSUPPORTED
    for f in (lib.SFM_FLAG_FULL_RES_MULTISCALE, lib.SFM_FLAG_BORDER_PADDING, lib.SFM_FLAG_MIN_REPROJECTION):
        assert call(G | f) == lib.SFM_E_UNSUPPORTED
    assert call(G, geo=None) == lib.SFM_E_NULL_POINTER
    g2 = lib.SfmGeometry()
    for s in range(3):
        g2.src_disps[s] = ptr
    assert call(G, geo=g2) == lib.SFM_E_NULL_POINTER                         # src_disps[3] missing
    # ... which is not needed with 3 scales: the call gets as far as the inputs check
    assert call(G, geo=g2, ns=3) == lib.SFM_E_NULL_POINTER
    terms = lib.SfmSnippetTerms(ptr, None)
    assert call(G, terms=C.byref(terms)) == lib.SFM_E_INVALID_DESC           # snippet terms without their flag
    assert call(G, losses=None) == lib.SFM_E_NULL_POINTER
    d = lib.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, G)
    ctx = C.c_void_p()
    assert so.sfm_host_ctx_create(C.byref(d), C.byref(ctx)) == lib.SFM_E_UNSUPPORTED


def test_operator_argument_errors():
    pytest.importorskip('sfm_learner_chainer_b200.lib')
    from sfm_learner_chainer_b200 import lib as L
    try:
        L.load()
    except ImportError:
        pytest.skip('libsfmloss.so not built')
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    with pytest.raises(ValueError):
        ViewSynthesisLoss(0.1, 0.0, 0.15, self_mask=True)
    for kw in (dict(image_grads=True), dict(pixel_terms=True), dict(min_reprojection=True),
               dict(full_res_multiscale=True), dict(border_padding=True)):
        with pytest.raises(ValueError):
            ViewSynthesisLoss(0.1, 0.0, 0.15, geometry_consistency=True, **kw)
    with pytest.raises(ValueError):
        ViewSynthesisLoss(0.1, 0.2, 0.0, geometry_consistency=True)
