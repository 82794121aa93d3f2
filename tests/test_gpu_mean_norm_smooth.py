"""-m gpu: the mean-normalised smoothness (SFM_FLAG_MEAN_NORM_SMOOTH, ViewSynthesisLoss(mean_norm_smooth=True)) and
Monodepth2's edge weight (SFM_FLAG_EDGE_MEAN_ABS) against the reference of tests/mean_norm_smooth_oracle.py added to the
existing photometric references: losses and every gradient at the configuration shapes, both kinds and both edge
weights, raw disparity, the three step kinds, the compositions with the other options, Monodepth2's whole configuration,
the untouched photometric side, reproducibility, graph replay, the edge cases and the torch adapter."""
import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests import full_res_oracle as FR
from tests import mean_norm_smooth_oracle as MN
from tests import min_reprojection_oracle as MR
from tests.gpu_util import FLAGSETS, make_op, to_dev, dev_inputs, host, assert_grad_close
from tests.pixel_oracle import sfm_loss_pixel, sfm_loss_pixel_raw

pytestmark = pytest.mark.gpu

KINDS = {'second': {}, 'edge': dict(edge_aware_smooth=True), 'edge_mean_abs': dict(edge_aware_smooth=True, edge_mean_abs=True)}


def _args(g):
    return g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses']


def _cfgs(flags, kind, ns=4, B_global=None):
    """(the photometric reference's cfg with smooth_reg = 0, the smoothness cfg)"""
    edge = bool(KINDS[kind].get('edge_aware_smooth'))
    c0 = O.LossConfig(exp_reg=flags['exp_reg'], ssim_rate=flags['ssim_rate'], n_scales=ns, B_global=B_global)
    cs = O.LossConfig(smooth_reg=flags['smooth_reg'], n_scales=ns, B_global=B_global, edge_aware_smooth=edge)
    return c0, cs


def _reference(d, flags, kind, ns=4, raw=0, disps=None):
    disps = d['disps'][:ns] if disps is None else disps
    c0, cs = _cfgs(flags, kind, ns)
    args = (d['tgt'], d['src'], d['intrinsics'][:, :ns], disps, d['poses'], d['logits'][:ns] if flags['exp_reg'] else None, c0)
    L, G = sfm_loss_pixel_raw(*args, raw_disp_scales=raw) if raw else sfm_loss_pixel(*args)
    return MN.add_smoothness(L, G, d['tgt'], disps, cs, raw, True, kind == 'edge_mean_abs')


def _check(l, g, L, G, ns, exp=False):
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    if G is None:
        return
    for s in range(ns):
        assert_grad_close(host(g['gdisps'][s]), G['gdisp'][s], what='gdisp[%d]' % s)
        if exp:
            assert_grad_close(host(g['glogits'][s]), G['glogits'][s], what='glogits[%d]' % s)
    assert_grad_close(host(g['gposes']), G['gpose'], what='gposes')


CASES = [
    ('cfg1', dict(FLAGSETS['cfg1'], smooth_reg=0.1), (4, 2, 128, 416), 4, 0),
    ('cfg2', FLAGSETS['cfg2'], (4, 2, 128, 416), 4, 0),
    ('cfg4', FLAGSETS['cfg4'], (8, 4, 128, 416), 4, 0),
    ('cfg5_shape', FLAGSETS['cfg2'], (2, 2, 256, 832), 4, 0),
    ('ns1', FLAGSETS['cfg2'], (3, 2, 128, 416), 1, 0),
    ('ns2', FLAGSETS['cfg2'], (3, 2, 128, 416), 2, 0),
    ('ns3_raw1', FLAGSETS['cfg2'], (3, 2, 128, 416), 3, 0b1),
    ('raw_all', FLAGSETS['cfg2'], (3, 2, 128, 416), 4, 0b1111),
]


@pytest.mark.parametrize('kind', sorted(KINDS))
@pytest.mark.parametrize('name,flags,shape,ns,raw', CASES, ids=[c[0] for c in CASES])
def test_losses_and_gradients_match_reference(name, flags, shape, ns, raw, kind):
    d = make_snippets(*shape, seed=8100 + shape[0], n_scales=4, harsh=True)
    disps = d['disps'][:ns]
    if raw:
        rd = make_raw_seam(d, seed=8101)[0]
        disps = [rd[s] if (raw >> s) & 1 else x for s, x in enumerate(disps)]
    g = dev_inputs(d)
    gd = [to_dev(x) for x in disps]
    op = make_op(flags, n_scales=ns, raw_disp_scales=raw, mean_norm_smooth=True, **KINDS[kind])
    a = (g['tgt'], g['src'], g['intrinsics'][:, :ns].contiguous(), gd, g['poses'])
    lg = [g['logits'][s] for s in range(ns)] if flags['exp_reg'] else None
    L, G = _reference(d, flags, kind, ns, raw, disps)
    l, gg = op.forward_backward(*a, logits=lg)
    _check(l, gg, L, G, ns, bool(flags['exp_reg']))
    lf = op.forward(*a, logits=lg)
    np.testing.assert_allclose(host(lf), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    gb = op.backward(*a, logits=lg)
    for s in range(ns):
        np.testing.assert_array_equal(host(gb['gdisps'][s]), host(gg['gdisps'][s]))


@pytest.mark.parametrize('kind', sorted(KINDS))
def test_snippet_and_pixel_terms(kind):
    flags = FLAGSETS['cfg2']
    B, S, H, W = 3, 2, 64, 208
    d = make_snippets(B, S, H, W, seed=8200, harsh=True)
    g = dev_inputs(d)
    rs = np.random.RandomState(8201)
    pw = [rs.uniform(-0.5, 2.0, (B, S, H >> s, W >> s)).astype(np.float32) for s in range(4)]
    wb = np.array([0.7, 0.0, -1.3], np.float32)
    op = make_op(flags, snippet_terms=True, pixel_terms=True, mean_norm_smooth=True, **KINDS[kind])
    l, gg = op.forward_backward(*_args(g), snippet_weights=to_dev(wb), pixel_weights=[to_dev(w) for w in pw])
    _, cs = _cfgs(flags, kind)
    # the photometric terms are linear in the snippet weights: per-snippet rows from one-snippet references
    rows = np.zeros((B, 5))
    gdisp = [np.zeros(x.shape) for x in d['disps']]
    gpose = np.zeros(d['poses'].shape)
    for b in range(B):
        sl = slice(b, b + 1)
        Lb, Gb = sfm_loss_pixel(d['tgt'][sl], d['src'][sl], d['intrinsics'][sl], [x[sl] for x in d['disps']], d['poses'][sl],
                                None, O.LossConfig(exp_reg=0.0, ssim_rate=flags['ssim_rate'], n_scales=4, B_global=B),
                                pixel_weights=[w[sl] for w in pw])
        rows[b] = O.losses_vec(Lb)
        for s in range(4):
            gdisp[s][sl] += wb[b] * Gb['gdisp'][s]
        gpose[sl] += wb[b] * Gb['gpose']
    sm, srows, sg = MN.smoothness(d['tgt'], d['disps'], cs, 0, True, kind == 'edge_mean_abs', snippet_weights=wb)
    rows[:, 2] = srows
    rows[:, 0] += srows
    np.testing.assert_allclose(host(gg['snippet_losses']), rows, rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(host(l), (wb[:, None].astype(np.float64) * rows).sum(0), rtol=1e-5, atol=1e-8)
    for s in range(4):
        assert_grad_close(host(gg['gdisps'][s]), gdisp[s] + sg[s], what='gdisp[%d]' % s)
    assert_grad_close(host(gg['gposes']), gpose, what='gposes')
    # the maps are the photometric side's: those of the step without the flag
    ext = {k: v for k, v in KINDS[kind].items() if k != 'edge_mean_abs'}
    lp, gp = make_op(flags, snippet_terms=True, pixel_terms=True, **ext).forward_backward(
        *_args(g), snippet_weights=to_dev(wb), pixel_weights=[to_dev(w) for w in pw])
    for s in range(4):
        np.testing.assert_array_equal(host(gg['pixel_losses'][s]), host(gp['pixel_losses'][s]))
    np.testing.assert_array_equal(host(l)[[1, 4]], host(lp)[[1, 4]])


@pytest.mark.parametrize('full_res', [False, True])
def test_min_reprojection_full_res_and_intrinsics(full_res):
    """Minimum reprojection with auto-masking (and full-res multi-scale: Monodepth2's whole configuration with the
    mean-absolute edge weight, SSIM 0.85); the selection, pixel terms and intrinsics gradient are the photometric side's."""
    flags = dict(FLAGSETS['cfg2'], ssim_rate=0.85, smooth_reg=1e-3)
    d = make_snippets(3, 2, 128, 416, seed=8300, harsh=True)
    g = dev_inputs(d)
    kw = dict(min_reprojection=True, automask=True, intrinsics_grad=True, full_res_multiscale=full_res,
              edge_aware_smooth=True)
    l, gg = make_op(flags, mean_norm_smooth=True, edge_mean_abs=True, **kw).forward_backward(*_args(g))
    lp, gp = make_op(flags, **kw).forward_backward(*_args(g))
    sel = [host(x) for x in gg['selection']]
    for s in range(4):
        np.testing.assert_array_equal(sel[s], host(gp['selection'][s]))
    np.testing.assert_array_equal(host(l)[[1, 4]], host(lp)[[1, 4]])
    np.testing.assert_allclose(host(gg['gintrinsics']), host(gp['gintrinsics']), rtol=1e-5,
                               atol=1e-6 * np.abs(host(gp['gintrinsics'])).max())
    c0, cs = _cfgs(flags, 'edge_mean_abs')
    if full_res:
        L, G = FR.sfm_loss_full_res(*_args(d), c0, min_reprojection=True, selection=sel)
    else:
        L, G = MR.sfm_loss_min_reprojection(*_args(d), c0, selection=sel)
    L, G = MN.add_smoothness(L, G, d['tgt'], d['disps'], cs, 0, True, True)
    _check(l, gg, L, G, 4)


def _off(got, ref, rtol=1e-4, atol_rel=5e-5):
    """The entries assert_grad_close rejects (its bar: rtol, plus a floor relative to the largest reference entry)."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    return np.abs(got - ref) > atol_rel * float(np.max(np.abs(ref))) + rtol * np.abs(ref)


def test_monodepth2_configuration_against_the_torch_restatement():
    """full-res + min-reprojection + automask + edge-aware + EDGE_MEAN_ABS + MEAN_NORM_SMOOTH, SSIM 0.85, against the
    torch fp64 restatements (tests/torch_full_res_restatement.py for the photometric terms, the literal Monodepth2
    smoothness of tests/torch_mean_norm_smooth_restatement.py).

    A full-resolution pixel whose photometric term sits on a kink (the x2 out-of-view rule, the SSIM clip) can be resolved
    differently by fp32 and fp64 arithmetic; its gradient then reaches the bilinear taps of the native maps.  At this seed
    the two references themselves disagree, on the CPU, at 1 of 6656 entries of gdisp[1], 4 of 1664 of gdisp[2] and 4 of
    416 of gdisp[3] (and so in gposes, a sum over every pixel), in the photometric part only: the smoothness parts agree to
    1e-7.  So every entry is checked at the default bar against the composed fp32-arithmetic reference (full_res_oracle +
    mean_norm_smooth_oracle, with the device's selection), and against the torch restatement wherever the two references
    agree, which must be everywhere but the taps of at most four full-resolution pixels per scale."""
    import torch
    from tests.torch_full_res_restatement import torch_full_res
    from tests.torch_mean_norm_smooth_restatement import torch_smoothness
    flags = dict(FLAGSETS['cfg2'], ssim_rate=0.85, smooth_reg=1e-3)
    d = make_snippets(2, 2, 64, 208, seed=8350, harsh=True)
    g = dev_inputs(d)
    op = make_op(flags, full_res_multiscale=True, min_reprojection=True, automask=True, edge_aware_smooth=True,
                 edge_mean_abs=True, mean_norm_smooth=True)
    l, gg = op.forward_backward(*_args(g))
    d64 = {k: (v.astype(np.float64) if isinstance(v, np.ndarray) else [x.astype(np.float64) for x in v]) for k, v in d.items()}
    rd = [torch.from_numpy(x).requires_grad_(True) for x in d64['disps']]
    rp = torch.from_numpy(d64['poses']).requires_grad_(True)
    ph, _, _, _, rsel = torch_full_res(d64, O.LossConfig(ssim_rate=0.85), rd, rp, torch.from_numpy(d64['intrinsics']),
                                       min_reprojection=True)
    sm, _ = torch_smoothness(torch.from_numpy(d64['tgt']), rd, 1e-3, edge=True, edge_mean_abs=True)
    (ph + sm).backward()
    np.testing.assert_allclose(host(l)[2], sm.item(), rtol=1e-5)
    sel = [host(x) for x in gg['selection']]
    same = all(np.array_equal(a, b.numpy()) for a, b in zip(sel, rsel))
    np.testing.assert_allclose(host(l)[0], (ph + sm).item(), rtol=1e-4 if same else 1e-3)
    c0, cs = _cfgs(flags, 'edge_mean_abs')
    L, G = FR.sfm_loss_full_res(*_args(d), c0, min_reprojection=True, selection=sel)
    L, G = MN.add_smoothness(L, G, d['tgt'], d['disps'], cs, 0, True, True)
    _check(l, gg, L, G, 4)
    if not same:
        return
    for s in range(4):
        ref_t = rd[s].grad.numpy()
        agree = ~_off(G['gdisp'][s], ref_t)
        assert (~agree).sum() <= 16, 'gdisp[%d]: the references disagree at %d of %d entries' % (s, (~agree).sum(), agree.size)
        bad = _off(host(gg['gdisps'][s]), ref_t) & agree
        assert not bad.any(), 'gdisp[%d]: %d entries off the torch restatement' % (s, int(bad.sum()))
    if not _off(G['gpose'], rp.grad.numpy()).any():
        assert_grad_close(host(gg['gposes']), rp.grad.numpy(), what='gposes')


def test_image_grads_with_second_order_smoothness():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=8400, harsh=True)
    g = dev_inputs(d)
    l, gg = make_op(flags, image_grads=True, mean_norm_smooth=True).forward_backward(*_args(g))
    lp, gp = make_op(flags, image_grads=True).forward_backward(*_args(g))
    np.testing.assert_array_equal(host(gg['gtgt']), host(gp['gtgt']))
    np.testing.assert_allclose(host(gg['gsrc']), host(gp['gsrc']), rtol=1e-5, atol=1e-6 * np.abs(host(gp['gsrc'])).max())
    L, G = _reference(d, flags, 'second')
    _check(l, gg, L, G, 4)


def test_peer_step_on_one_rank_reproducibility_and_graph_replay():
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=8500, harsh=True)
    g = dev_inputs(d)
    for kind in sorted(KINDS):
        op = make_op(flags, mean_norm_smooth=True, **KINDS[kind])
        l0, g0 = op.forward_backward(*_args(g))
        l1, g1 = op.forward_backward(*_args(g))
        np.testing.assert_array_equal(host(l1), host(l0))
        for s in range(4):
            np.testing.assert_array_equal(host(g1['gdisps'][s]), host(g0['gdisps'][s]))
        peer = PeerLossSum(0, 1)
        try:
            lp, gp = op.forward_backward(*_args(g), peer=peer)
            np.testing.assert_allclose(host(lp), host(l0), rtol=1e-6, atol=1e-12)
            for s in range(4):
                np.testing.assert_array_equal(host(gp['gdisps'][s]), host(g0['gdisps'][s]))
        finally:
            torch.cuda.synchronize()
            peer.close()
    # a captured graph replayed with new disparities recomputes the means
    d2 = make_snippets(3, 2, 64, 208, seed=8501, harsh=True)
    op = make_op(flags, mean_norm_smooth=True, edge_aware_smooth=True, edge_mean_abs=True)
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        op.forward_backward(*_args(g))
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l, gg = op.forward_backward(*_args(g))
    for dd in (d2, d):
        for s in range(4):
            g['disps'][s].copy_(torch.from_numpy(dd['disps'][s]))
        graph.replay()
        torch.cuda.synchronize()
        L, G = _reference(dict(d, disps=dd['disps']), flags, 'edge_mean_abs')     # the captured images, new disparities
        _check(l, gg, L, G, 4)


def test_edge_cases():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=8600, harsh=True)
    g = dev_inputs(d)
    for kind in sorted(KINDS):
        ext = {k: v for k, v in KINDS[kind].items() if k != 'edge_mean_abs'}
        # smooth_reg = 0 with the flag is the plain step, bitwise
        z = dict(flags, smooth_reg=0.0)
        l, gg = make_op(z, mean_norm_smooth=True, **KINDS[kind]).forward_backward(*_args(g))
        lp, gp = make_op(z, **ext).forward_backward(*_args(g))
        np.testing.assert_array_equal(host(l), host(lp))
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gp['gdisps'][s]))
        # a constant disparity: zero smoothness loss and gradient
        gc = dict(g, disps=[torch_full(x, 2.5) for x in g['disps']])
        l, gg = make_op(flags, mean_norm_smooth=True, **KINDS[kind]).forward_backward(*_args(gc))
        lp, gp = make_op(z, **ext).forward_backward(*_args(gc))
        assert host(l)[2] == 0.0
        np.testing.assert_array_equal(host(l)[[1, 4]], host(lp)[[1, 4]])
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gp['gdisps'][s]))


def torch_full(x, v):
    import torch
    return torch.full_like(x, v)


def test_torch_adapter_autograd():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 64, 208, seed=8700, harsh=True)
    g = dev_inputs(d)
    gy = 0.37
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    poses = g['poses'].clone().requires_grad_(True)
    out = view_synthesis_loss(make_op(flags, mean_norm_smooth=True, edge_aware_smooth=True, edge_mean_abs=True),
                              g['tgt'], g['src'], g['intrinsics'], disps, poses)
    total = out[0] if isinstance(out, tuple) else out
    (gy * total).backward()
    L, G = _reference(d, flags, 'edge_mean_abs')
    np.testing.assert_allclose(float(total.detach()), L['total_loss'], rtol=1e-5)
    for s in range(4):
        assert_grad_close(host(disps[s].grad), gy * G['gdisp'][s], what='disps[%d].grad' % s)
    assert_grad_close(host(poses.grad), gy * G['gpose'], what='poses.grad')
