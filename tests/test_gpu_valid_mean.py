"""-m gpu: SC-SfMLearner's valid-pixel means, auto-mask and clamped L1 (sfm_loss_geometry_valid_mean,
ViewSynthesisLoss(geometry_consistency=True, valid_mean=True)) against the numpy reference (tests/valid_mean_oracle.py),
the exact counts, the identities (no struct = sfm_loss_geometry, groups = S over B*S snippets = S calls, zero-weight
padding), the min_count thresholds, the compositions, reproducibility, CUDA-graph replay and the torch adapter."""

import numpy as np
import pytest

from oracle import sfm_oracle as O
from tests import geometry_oracle as GO
from tests import valid_mean_oracle as VM
from tests.gpu_util import FLAGSETS, make_op, op_args, to_dev, dev_inputs, host, assert_grad_close

pytestmark = pytest.mark.gpu

REG = 0.5


def _case(B, S, H, W, seed, harsh, ns=4):
    d = make_snippets(B, S, H, W, seed=seed, n_scales=ns, harsh=harsh)
    if harsh:
        d['poses'][:, 0, 5] -= np.float32(0.5)
    return d, GO.make_src_disps(B, S, H, W, ns, seed + 7)


def make_snippets(*a, **kw):
    from sfm_learner_chainer_b200.synthetic import make_snippets as m
    return m(*a, **kw)


def _op(flags, ns=4, **kw):
    base = dict(geometry_consistency=True, geometry_reg=REG, valid_mean=True, n_scales=ns)
    base.update(kw)
    return make_op(flags, **base)


def _run(op, g, flags, sd, grads=True, **kw):
    if grads:
        return op.forward_backward(*op_args(g, flags), src_disps=sd, **kw)
    out = op.forward(*op_args(g, flags), src_disps=sd, **kw)
    return out[0], dict(valid_masks=out[-2], valid_counts=out[-1], geometry_diff=out[-3])


def _ref(d, flags, sd, ns, masks=None, **kw):
    cfg = O.LossConfig(n_scales=ns, **flags)
    return VM.loss(*op_args(d, flags)[:5], sd, cfg, geometry_reg=REG, masks=masks, **kw)


def _check_masks(d, flags, sd, ns, gg, automask):
    """The device's masks against the reference's, except at near ties of the auto-mask; counts exactly those of the
    device's masks."""
    L, _ = _ref(d, flags, sd, ns, automask=automask, min_count=0.0, want_grads=False)
    ties = VM.near_ties(*op_args(d, flags)[:5], sd, O.LossConfig(n_scales=ns, **flags)) if automask else None
    dm = [host(m).astype(bool) for m in gg['valid_masks']]
    for s in range(ns):
        off = dm[s] != L['valid_masks'][s]
        if ties is not None:
            off &= ~ties[s]
        assert not off.any(), 'mask[%d]: %d pairs differ' % (s, int(off.sum()))
    cnt = host(gg['valid_counts'])
    G = cnt.shape[2]
    for s in range(ns):
        per_b = dm[s].reshape(dm[s].shape[0], dm[s].shape[1], -1).sum(-1)
        for g in range(G):
            np.testing.assert_array_equal(cnt[s, :, g], per_b[g::G].sum(0))
    return dm


def _check(l, gg, L, G, ns, what='', k=False):
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9, err_msg=what)
    if G is None:
        return
    for s in range(ns):
        assert_grad_close(host(gg['gdisps'][s]), G['gdisp'][s], what='%s gdisp[%d]' % (what, s))
        assert_grad_close(host(gg['gsrc_disps'][s]), G['gsrc_disp'][s], what='%s gsrc_disps[%d]' % (what, s))
    assert_grad_close(host(gg['gposes']), G['gpose'], what=what + ' gposes')
    if k:
        assert_grad_close(host(gg['gintrinsics']), G['gintrinsics'], what=what + ' gintrinsics')


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('automask', [False, True])
@pytest.mark.parametrize('self_mask', [False, True])
def test_parity_with_reference(cfg, ns, S, automask, self_mask):
    flags = FLAGSETS[cfg]
    harsh = (S == 3)
    d, sd = _case(2, S, 128, 416, 6100 + S + 10 * automask, harsh, ns)
    op = _op(flags, ns, valid_automask=automask, self_mask=self_mask, valid_min_count=100.0, intrinsics_grad=True)
    l, gg = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd])
    dm = _check_masks(d, flags, sd, ns, gg, automask)
    L, G = _ref(d, flags, sd, ns, masks=dm, self_mask=self_mask, automask=automask, min_count=100.0,
                want_intrinsics_grad=True)
    _check(l, gg, L, G, ns, '%s ns=%d S=%d auto=%d mask=%d' % (cfg, ns, S, automask, self_mask), k=True)
    # forward only: the losses, masks and counts of the gradient step
    lf, gf = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd], grads=False)
    np.testing.assert_array_equal(host(lf), host(l))
    np.testing.assert_array_equal(host(gf['valid_counts']), host(gg['valid_counts']))
    for s in range(ns):
        np.testing.assert_array_equal(host(gf['valid_masks'][s]), host(gg['valid_masks'][s]))


def test_clamped_pixels():
    """A target 2.5 times brighter: most L1 differences exceed 1 and are clamped."""
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 128, 416, 6201, False)
    d['tgt'] = (d['tgt'] * np.float32(2.5)).astype(np.float32)
    op = _op(flags, self_mask=True)
    l, gg = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd])
    dm = _check_masks(d, flags, sd, 4, gg, True)
    L, G = _ref(d, flags, sd, 4, masks=dm, self_mask=True, automask=True, min_count=10000.0)
    _check(l, gg, L, G, 4, 'clamped')


def test_vm_null_is_sfm_loss_geometry():
    """vm == NULL: bitwise sfm_loss_geometry (the entry point with a descriptor carrying SFM_FLAG_VALID_MEAN), and both
    bitwise the geometry operator without valid_mean."""
    import ctypes as C
    from sfm_learner_chainer_b200 import device as Dv, lib as Lb
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 128, 416, 6301, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    ref = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True)
    lp, gp = _run(ref, g, flags, sdd)
    op = _op(flags, self_mask=True)
    args = op_args(g, flags)
    tgt = args[0]
    desc, inp = op._pack(*args)
    assert desc.flags & Lb.SFM_FLAG_VALID_MEAN
    so, ws, st = op._lib, op._workspace(desc, tgt), C.c_void_p(Dv.current_stream(tgt))
    for name in ('sfm_loss_geometry', 'sfm_loss_geometry_valid_mean'):
        l = Dv.empty(tgt, (5,))
        grads, gg = op._alloc_grads(desc, tgt)
        ge, gg['geometry_diff'], _ = op._geometry(desc, tgt, sdd, True)
        vm = () if name == 'sfm_loss_geometry' else (None,)
        Lb.check(getattr(so, name)(C.byref(desc), C.byref(inp), None, C.byref(ge), *vm, C.c_void_p(Dv.ptr(l)),
                                   C.byref(grads), ws, None, st))
        np.testing.assert_array_equal(host(l), host(lp))
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gp['gdisps'][s]))
            np.testing.assert_array_equal(host(gg['geometry_diff'][s]), host(gp['geometry_diff'][s]))
        np.testing.assert_allclose(host(gg['gposes']), host(gp['gposes']), rtol=1e-5,
                                   atol=1e-6 * np.abs(host(gp['gposes'])).max())


def test_groups_equal_separate_calls():
    """One call with count_groups = S on B*S one-source snippets ordered (b, i) equals S calls of B snippets with
    count_groups = 1 (snippet terms with weights 1: the rows of the one call are those of the separate calls)."""
    flags = FLAGSETS['cfg2']
    B, S = 2, 3
    d, sd = _case(B * S, 1, 128, 416, 6401, False)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    op = _op(flags, self_mask=True, count_groups=S, snippet_terms=True)
    l, gg = _run(op, g, flags, sdd, grads=False, snippet_weights=to_dev(np.ones(B * S, np.float32)))
    tot = np.zeros(5)
    for i in range(S):
        idx = np.arange(B) * S + i
        di = {k: ([x[idx] for x in v] if isinstance(v, list) else v[idx]) for k, v in d.items() if v is not None}
        gi = dev_inputs(di)
        oi = _op(flags, self_mask=True)
        li, gi_ = _run(oi, gi, flags, [to_dev(x[idx]) for x in sd], grads=False)
        np.testing.assert_array_equal(host(gg['valid_counts'])[:, :, i], host(gi_['valid_counts'])[:, :, 0])
        tot += host(li).astype(np.float64)
    # the one call's mean over a group's snippets equals the separate call's mean over its batch up to the batch factor
    # B*S / B in the smoothness (per snippet) -- compared on the photometric and geometry parts, which are per group
    np.testing.assert_allclose(host(l)[[1, 3, 4]], tot[[1, 3, 4]], rtol=1e-6)


def test_zero_weight_padding():
    flags = FLAGSETS['cfg2']
    d, sd = _case(3, 2, 128, 416, 6501, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    op = _op(flags, self_mask=True, snippet_terms=True)
    l, gg = _run(op, g, flags, sdd, snippet_weights=to_dev(np.array([1, 0, 1], np.float32)))
    assert not host(gg['valid_masks'][0])[1].any()
    idx = np.array([0, 2])
    dp = {k: ([x[idx] for x in v] if isinstance(v, list) else v[idx]) for k, v in d.items() if v is not None}
    op2 = _op(flags, self_mask=True, snippet_terms=True)
    l2, g2 = _run(op2, dev_inputs(dp), flags, [to_dev(x[idx]) for x in sd], snippet_weights=to_dev(np.ones(2, np.float32)))
    np.testing.assert_array_equal(host(gg['valid_counts']), host(g2['valid_counts']))
    # the photometric and geometry parts are the valid-pixel means, independent of the batch size; the smoothness and the
    # rows of the kept snippets differ only by the 1 / B of the smoothness
    np.testing.assert_allclose(host(l)[[1, 3, 4]], host(l2)[[1, 3, 4]], rtol=1e-6)
    for s in range(4):
        assert not host(gg['gdisps'][s])[1].any()


def test_min_count_thresholds():
    flags = FLAGSETS['cfg1']
    d, sd = _case(2, 1, 128, 416, 6601, False, ns=1)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    l0, g0 = _run(_op(flags, 1, valid_min_count=0.0), g, flags, sdd, grads=False)
    n = int(host(g0['valid_counts'])[0, 0, 0])
    base = host(l0)
    for mc, photo, geo in ((3 * n - 1, True, False), (3 * n, False, False), (n - 1, True, True), (n, True, False)):
        l, _ = _run(_op(flags, 1, valid_min_count=float(mc)), g, flags, sdd, grads=False)
        l = host(l)
        assert (l[1] == base[1]) if photo else (l[1] == 0.0), mc
        assert (l[3] == base[3]) if geo else (l[3] == 0.0), mc


@pytest.mark.parametrize('what', ['raw', 'axisangle', 'smooth', 'tables'])
def test_compositions(what):
    """Each option composes: the result against the reference (raw inputs: against the activated step; the smoothness
    options: the difference to the step without them is that of the plain steps)."""
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 128, 416, 6701, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    if what == 'axisangle':
        op = _op(flags, self_mask=True, axisangle_pose=True, invert_sources=(0,), intrinsics_grad=True)
        l, gg = _run(op, g, flags, sdd)
        dm = [host(m).astype(bool) for m in gg['valid_masks']]
        L, G = _ref(d, flags, sd, 4, masks=dm, self_mask=True, invert_sources=(0,), want_intrinsics_grad=True)
        _check(l, gg, L, G, 4, 'axisangle', k=True)
    elif what == 'tables':
        op = _op(flags, self_mask=True, intrinsics_grad=True)
        l, gg = _run(op, g, flags, sdd)
        proj, kinv = op.build_tables(g['poses'], g['intrinsics'], 128, 416)
        lt, gt = _run(op, g, flags, sdd, proj=proj, kinv=kinv, intrinsics_grad=False)
        np.testing.assert_array_equal(host(lt), host(l))
        for s in range(4):
            np.testing.assert_array_equal(host(gt['gdisps'][s]), host(gg['gdisps'][s]))
        op.build_pyramid(g['tgt'], g['src'])
        lr, gr = _run(op, g, flags, sdd, reuse_pyramid=True)
        np.testing.assert_array_equal(host(lr), host(l))
        dm = [host(m).astype(bool) for m in gg['valid_masks']]
        L, G = _ref(d, flags, sd, 4, masks=dm, self_mask=True, want_intrinsics_grad=True)
        assert_grad_close(host(gg['gintrinsics']), G['gintrinsics'], what='gintrinsics')
    elif what == 'smooth':
        sm = dict(edge_aware_smooth=True, mean_norm_smooth=True, edge_mean_abs=True)
        off = dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=flags['ssim_rate'])
        la, ga = _run(_op(flags, self_mask=True, **sm), g, flags, sdd)
        lb, gb = _run(_op(off, self_mask=True), g, off, sdd)
        lc, gc = make_op(flags, **sm).forward_backward(*op_args(g, flags))
        ld, gd = make_op(off).forward_backward(*op_args(g, off))
        np.testing.assert_array_equal(host(la)[2], host(lc)[2])
        np.testing.assert_allclose(host(la)[[1, 3, 4]], host(lb)[[1, 3, 4]], rtol=1e-6)
        for s in range(4):
            # a difference of two gradient fields, each rounded where the march adds onto the smoothness: a few entries
            # near zero are off by ~1e-4 of the difference's largest entry
            assert_grad_close(host(ga['gdisps'][s]) - host(gb['gdisps'][s]), host(gc['gdisps'][s]) - host(gd['gdisps'][s]),
                              what='smooth gdisp[%d]' % s, atol_rel=5e-4)
    else:
        from sfm_learner_chainer_b200 import disp_activation, pose_reduce
        from sfm_learner_chainer_b200.synthetic import make_raw_seam
        raw_d, raw_p = make_raw_seam(d, seed=6702)
        rd, rp = [to_dev(x) for x in raw_d], to_dev(raw_p)
        gr_ = dict(g, disps=rd, poses=rp)
        l, gg = _run(_op(flags, self_mask=True, raw_disp_scales=0xF, raw_pose=True), gr_, flags, sdd)
        acts = [disp_activation(x, want_dact=True) for x in rd]
        ga = dict(gr_, disps=[a for a, _ in acts], poses=pose_reduce(rp, 2))
        la, gga = _run(_op(flags, self_mask=True), ga, flags, sdd)
        np.testing.assert_allclose(host(l), host(la), rtol=5e-7, atol=0)
        np.testing.assert_array_equal(host(gg['valid_counts']), host(gga['valid_counts']))
        for s in range(4):
            ref = host(gga['gdisps'][s]).astype(np.float64) * host(acts[s][1]).astype(np.float64)
            assert_grad_close(host(gg['gdisps'][s]), ref, rtol=2e-6, atol_rel=1e-7, what='gdisp[%d]' % s)


def test_reproducibility_and_graph_replay():
    import torch
    flags = FLAGSETS['cfg2']
    d, sd = _case(3, 2, 128, 416, 6801, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    op = _op(flags, self_mask=True)
    l0, g0 = _run(op, g, flags, sdd)
    l0, c0, g0 = host(l0), host(g0['valid_counts']), {s: host(g0['gdisps'][s]) for s in range(4)}
    l1, g1 = _run(op, g, flags, sdd)
    np.testing.assert_array_equal(host(l1), l0)
    for s in range(4):
        np.testing.assert_array_equal(host(g1['gdisps'][s]), g0[s])
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        _run(op, g, flags, sdd)
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l, gg = _run(op, g, flags, sdd)
    for _ in range(3):
        graph.replay()
        torch.cuda.synchronize()
        np.testing.assert_array_equal(host(l), l0)
        np.testing.assert_array_equal(host(gg['valid_counts']), c0)
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), g0[s])


def test_torch_adapter():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 128, 416, 6901, False)
    g = dev_inputs(d)
    op = _op(flags, self_mask=True)
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    srcd = [to_dev(x).requires_grad_(True) for x in sd]
    poses = g['poses'].clone().requires_grad_(True)
    res = view_synthesis_loss(op, g['tgt'], g['src'], g['intrinsics'], disps, poses, src_disps=srcd)
    total, losses, diffs, masks, counts = res
    (2.0 * total).backward()
    assert len(diffs) == 4 and len(masks) == 4 and counts.shape == (4, 2, 1) and counts.dtype == torch.int32
    dm = [host(m).astype(bool) for m in masks]
    L, G = _ref(d, flags, sd, 4, masks=dm, self_mask=True)
    np.testing.assert_allclose(host(losses), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    for s in range(4):
        assert_grad_close(host(srcd[s].grad), 2.0 * G['gsrc_disp'][s], what='src_disps.grad[%d]' % s)
        assert_grad_close(host(disps[s].grad), 2.0 * G['gdisp'][s], what='disps.grad[%d]' % s)
    assert_grad_close(host(poses.grad), 2.0 * G['gpose'], what='poses.grad')


def test_refused_combinations():
    from sfm_learner_chainer_b200 import lib as Lb
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 64, 208, 7001, False)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    with pytest.raises(ValueError):
        _run(_op(flags, count_groups=3), g, flags, sdd)             # G > B
    with pytest.raises(ValueError):
        _op(flags, B_global=4)
    with pytest.raises(ValueError):
        _op(flags, min_reprojection=True)
    assert Lb.SFM_FLAG_VALID_MEAN == 0x2000


def test_cfg5_shape():
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 256, 832, 7101, True)
    op = _op(flags, self_mask=True)
    l, gg = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd])
    dm = _check_masks(d, flags, sd, 4, gg, True)
    L, G = _ref(d, flags, sd, 4, masks=dm, self_mask=True)
    _check(l, gg, L, G, 4, 'cfg5 shape')
