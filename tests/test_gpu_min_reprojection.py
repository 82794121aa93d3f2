"""-m gpu: per-pixel minimum reprojection with auto-masking (sfm_loss_min_reprojection,
ViewSynthesisLoss(min_reprojection=True)) against the reference built on the numpy oracle
(tests/min_reprojection_oracle.py): the selection at every pixel away from near ties, the losses and every gradient for
the exported selection, equality with sfm_loss_weighted given the one-hot weights, the compositions with the other
options, CUDA-graph replay and the torch adapter."""
import ctypes as C

import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests import min_reprojection_oracle as MR
from tests.gpu_util import FLAGSETS, make_op, to_dev, dev_inputs, host, oracle_tables, assert_grad_close

pytestmark = pytest.mark.gpu


def _args(g):
    return g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses']


def _op(flags, **kw):
    return make_op(flags, min_reprojection=True, **kw)


def _check(l, g, L, G, ns=4, k=False):
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    if G is None:
        return
    for s in range(ns):
        assert_grad_close(host(g['gdisps'][s]), G['gdisp'][s], what='gdisp[%d]' % s)
    assert_grad_close(host(g['gposes']), G['gpose'], what='gposes')
    if k:
        assert_grad_close(host(g['gintrinsics']), G['gintrinsics'], what='gintrinsics')


def _sel(g):
    return [host(x) for x in g['selection']]


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('automask', [True, False])
def test_selection_losses_and_gradients_match_oracle(cfg, S, automask):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, S, 128, 416, seed=3100 + S, harsh=True)
    cfg_o = O.LossConfig(**flags)
    l, g = _op(flags, automask=automask, intrinsics_grad=True).forward_backward(*_args(dev_inputs(d)))
    sel = _sel(g)
    # 1. the selection at every pixel whose best and runner-up candidate (identity included) are not within 1e-4
    e, m, e_id = MR.errors(*_args(d), cfg_o)
    amb_n = tot = 0
    for s in range(4):
        ref = MR.select(e[s], m[s], e_id[s], automask)
        amb = MR.ambiguous(e[s], m[s], e_id[s], automask)
        bad = (sel[s] != ref) & ~amb
        assert not bad.any(), 'scale %d: %d of %d pixels selected differently' % (s, int(bad.sum()), bad.size)
        amb_n += int(amb.sum())
        tot += amb.size
    assert amb_n <= 0.005 * tot, amb_n / tot
    # 2. losses and every gradient for the exported selection
    L, G = MR.sfm_loss_min_reprojection(*_args(d), cfg_o, automask=automask, selection=sel, want_intrinsics_grad=True)
    _check(l, g, L, G, k=True)
    # forward only: the same selection and losses
    lf, sf = _op(flags, automask=automask).forward(*_args(dev_inputs(d)))
    for s in range(4):
        np.testing.assert_array_equal(host(sf[s]), sel[s])
    np.testing.assert_allclose(host(lf), host(l), rtol=1e-6, atol=1e-12)


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
def test_same_as_weighted_with_one_hot_weights(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 3, 128, 416, seed=3201, harsh=True)
    g = dev_inputs(d)
    l, gg = _op(flags).forward_backward(*_args(g))
    W = [to_dev(MR.one_hot(s, 3, np.float32)) for s in _sel(gg)]
    lw, gw = make_op(flags, pixel_terms=True).forward_backward(*_args(g), pixel_weights=W)
    np.testing.assert_array_equal(host(l), host(lw))
    for s in range(4):
        np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gw['gdisps'][s]))
    np.testing.assert_allclose(host(gg['gposes']), host(gw['gposes']), rtol=1e-5, atol=1e-6 * np.abs(host(gw['gposes'])).max())


def test_single_source_without_automask_is_the_unit_weighted_step():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 1, 128, 416, seed=3301, harsh=True)
    g = dev_inputs(d)
    l, gg = _op(flags, automask=False).forward_backward(*_args(g))
    lw, gw = make_op(flags, pixel_terms=True).forward_backward(*_args(g))
    np.testing.assert_array_equal(host(l), host(lw))
    for s in range(4):
        np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gw['gdisps'][s]))
        assert set(np.unique(_sel(gg)[s])) <= {-2, 0}


def test_identical_source_is_auto_masked():
    flags = dict(FLAGSETS['cfg2'], smooth_reg=0.0)
    d = make_snippets(3, 2, 128, 416, seed=3401)
    d['src'][:, 1] = d['tgt']
    assert np.abs(d['poses'][:, 1]).max() > 0
    l, g = _op(flags).forward_backward(*_args(dev_inputs(d)))
    sel = _sel(g)
    assert all(np.all(s < 0) for s in sel)
    assert sum(int((s == -1).sum()) for s in sel) >= 0.9 * sum(s.size for s in sel)
    assert not host(l).any()
    assert not host(g['gposes']).any()
    for s in range(4):
        assert not host(g['gdisps'][s]).any()


def test_snippet_weights_do_not_change_the_selection():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=3501, harsh=True)
    g = dev_inputs(d)
    _, g0 = _op(flags).forward_backward(*_args(g))
    wb = np.array([0.7, 0.0, -1.3], np.float32)
    l, gg = _op(flags, snippet_terms=True).forward_backward(*_args(g), snippet_weights=to_dev(wb))
    sel = _sel(gg)
    for s in range(4):
        np.testing.assert_array_equal(sel[s], _sel(g0)[s])
    cfg_b = O.LossConfig(B_global=3, **flags)
    rows = np.zeros((3, 5))
    for b in range(3):
        sl = slice(b, b + 1)
        L, G = MR.sfm_loss_min_reprojection(d['tgt'][sl], d['src'][sl], d['intrinsics'][sl], [x[sl] for x in d['disps']],
                                            d['poses'][sl], cfg_b, selection=[x[sl] for x in sel])
        rows[b] = O.losses_vec(L)
        for s in range(4):
            assert_grad_close(host(gg['gdisps'][s])[sl], wb[b] * G['gdisp'][s].astype(np.float64), what='gdisp[%d]' % s)
    np.testing.assert_allclose(host(gg['snippet_losses']), rows, rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(host(l), (wb[:, None] * rows).sum(0), rtol=1e-5, atol=1e-9)


def test_raw_inputs():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=3601, harsh=True)
    raw_disps, raw_poses = make_raw_seam(d, (1, 4), seed=3602)
    args = (d['tgt'], d['src'], d['intrinsics'], raw_disps, raw_poses)
    op = _op(flags, raw_disp_scales=0xF, raw_pose=True)
    l, g = op.forward_backward(to_dev(d['tgt']), to_dev(d['src']), to_dev(d['intrinsics']), [to_dev(x) for x in raw_disps],
                               to_dev(raw_poses))
    cfg_o = O.LossConfig(**flags)
    e, m, e_id = MR.errors(d['tgt'], d['src'], d['intrinsics'], [O.disp_activation(x)[0] for x in raw_disps],
                           O.pose_from_raw(raw_poses, 2), cfg_o)
    sel = _sel(g)
    for s in range(4):
        ok = (sel[s] == MR.select(e[s], m[s], e_id[s], True)) | MR.ambiguous(e[s], m[s], e_id[s], True)
        assert ok.all()
    L, G = MR.sfm_loss_min_reprojection(*args, cfg_o, selection=sel, raw_disp_scales=0xF, raw_pose=True)
    _check(l, g, L, G)


def test_reused_pyramid_provided_tables_and_edge_smoothness():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=3701, harsh=True)
    g = dev_inputs(d)
    op = _op(flags)
    l0, g0 = op.forward_backward(*_args(g))
    op.build_pyramid(g['tgt'], g['src'])
    l1, g1 = op.forward_backward(*_args(g), reuse_pyramid=True)
    np.testing.assert_array_equal(host(l1), host(l0))
    for s in range(4):
        np.testing.assert_array_equal(host(g1['selection'][s]), host(g0['selection'][s]))
        np.testing.assert_array_equal(host(g1['gdisps'][s]), host(g0['gdisps'][s]))
    proj, kinv = oracle_tables(O, d)
    l2, g2 = op.forward_backward(*_args(g), proj=to_dev(proj), kinv=to_dev(kinv))
    L, G = MR.sfm_loss_min_reprojection(*_args(d), O.LossConfig(**flags), selection=_sel(g2))
    _check(l2, g2, L, G)
    cfg_e = O.LossConfig(edge_aware_smooth=True, **flags)
    l3, g3 = _op(flags, edge_aware_smooth=True).forward_backward(*_args(g))
    L, G = MR.sfm_loss_min_reprojection(*_args(d), cfg_e, selection=_sel(g3))
    _check(l3, g3, L, G)


def test_sharding_and_peer_sum_on_one_rank():
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=3801, harsh=True)
    g = dev_inputs(d)
    l, gg = _op(flags, B_global=5).forward_backward(*_args(g))
    L, G = MR.sfm_loss_min_reprojection(*_args(d), O.LossConfig(B_global=5, **flags), selection=_sel(gg))
    _check(l, gg, L, G)
    peer = PeerLossSum(0, 1)
    try:
        op = _op(flags)
        lr, gr = op.forward_backward(*_args(g))
        lp, gp = op.forward_backward(*_args(g), peer=peer)
        np.testing.assert_allclose(host(lp), host(lr), rtol=1e-6, atol=1e-12)
        for s in range(4):
            np.testing.assert_array_equal(host(gp['gdisps'][s]), host(gr['gdisps'][s]))
            np.testing.assert_array_equal(host(gp['selection'][s]), host(gr['selection'][s]))
    finally:
        torch.cuda.synchronize()
        peer.close()


def test_cuda_graph_capture_and_bitwise_replay():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=3901, harsh=True)
    g = dev_inputs(d)
    op = _op(flags)
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        le, ge = op.forward_backward(*_args(g))
        le, ge = host(le), dict(sel=_sel(ge), gd=[host(x) for x in ge['gdisps']])
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l, gg = op.forward_backward(*_args(g))
    outs = []
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        outs.append((host(l), _sel(gg), [host(x) for x in gg['gdisps']]))
    for lo, so, go in outs:
        np.testing.assert_array_equal(lo, outs[0][0])
        np.testing.assert_allclose(lo, le, rtol=1e-6, atol=1e-12)
        for s in range(4):
            np.testing.assert_array_equal(so[s], ge['sel'][s])
            np.testing.assert_array_equal(go[s], ge['gd'][s])


@pytest.mark.parametrize('cfg,shape', [('cfg1', (4, 2, 128, 416)), ('cfg2', (4, 2, 128, 416)), ('cfg2', (2, 2, 256, 832))])
def test_at_config_shapes(cfg, shape):
    flags = FLAGSETS[cfg]
    d = make_snippets(*shape, seed=4001)
    l, g = _op(flags).forward_backward(*_args(dev_inputs(d)))
    L, G = MR.sfm_loss_min_reprojection(*_args(d), O.LossConfig(**flags), selection=_sel(g))
    _check(l, g, L, G)


def test_explainability_branch_is_unsupported():
    from sfm_learner_chainer_b200 import lib as Lb
    flags = FLAGSETS['cfg4']
    d = make_snippets(2, 2, 64, 208, seed=4101)
    g = dev_inputs(d)
    with pytest.raises(ValueError):
        _op(flags)
    so = Lb.load()
    desc = Lb.SfmDesc(2, 2, 64, 208, 4, 0, flags['smooth_reg'], flags['exp_reg'], flags['ssim_rate'],
                      Lb.SFM_FLAG_MIN_REPROJECTION)
    ws = to_dev(np.zeros(so.sfm_workspace_bytes(C.byref(desc)) // 4 + 64, np.float32))
    inp = Lb.SfmInputs()
    inp.tgt, inp.src, inp.intrinsics, inp.poses = (g[k].data_ptr() for k in ('tgt', 'src', 'intrinsics', 'poses'))
    for s in range(4):
        inp.disps[s] = g['disps'][s].data_ptr()
        inp.logits[s] = g['logits'][s].data_ptr()
    losses = to_dev(np.zeros(5, np.float32))
    mr = Lb.SfmMinReprojection(1, 0)
    rc = so.sfm_loss_min_reprojection(C.byref(desc), C.byref(inp), None, C.byref(mr), C.c_void_p(losses.data_ptr()), None,
                                      C.c_void_p((ws.data_ptr() + 255) // 256 * 256), None, None)
    assert rc == Lb.SFM_E_UNSUPPORTED


def test_torch_adapter():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=4201, harsh=True)
    g = dev_inputs(d)
    gy = 0.37
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    poses = g['poses'].clone().requires_grad_(True)
    total, losses, sel = view_synthesis_loss(_op(flags), g['tgt'], g['src'], g['intrinsics'], disps, poses)
    assert len(sel) == 4 and sel[0].dtype == torch.int8 and not sel[0].requires_grad
    (gy * total).backward()
    L, G = MR.sfm_loss_min_reprojection(*_args(d), O.LossConfig(**flags), selection=[host(x) for x in sel])
    np.testing.assert_allclose(host(losses), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    for s in range(4):
        assert_grad_close(host(disps[s].grad), gy * G['gdisp'][s], what='disps[%d].grad' % s)
    assert_grad_close(host(poses.grad), gy * G['gpose'], what='poses.grad')
