"""-m gpu: per-pixel weights and per-pixel loss maps (sfm_loss_weighted, ViewSynthesisLoss(pixel_terms=True)) against the
weighted reference built on the numpy oracle (tests/pixel_oracle.py), every marching-kernel instance under forced task heights, bitwise equality with the plain
step for unit weights, reproducible maps, the composition with the other options, CUDA-graph replay with changing
weights and the torch adapter."""
import copy

import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests.pixel_oracle import sfm_loss_pixel, sfm_loss_pixel_raw
from tests.gpu_util import (FLAGSETS, make_op, op_args, to_dev, dev_inputs, host, oracle_tables, assert_grad_close,
                            check_same_as_plain)

pytestmark = pytest.mark.gpu


def _pix_weights(d, seed, null_scale=None):
    """Weights in [0, 1] with about 10 % negative ones, scale `null_scale` None (= 1)."""
    rs = np.random.RandomState(seed)
    out = []
    for s, l in enumerate(d['logits']):
        if s == null_scale:
            out.append(None)
            continue
        w = rs.uniform(0.0, 1.0, l.shape).astype(np.float32)
        neg = rs.uniform(0.0, 1.0, l.shape) < 0.1
        w[neg] = -w[neg]
        out.append(w)
    return out


def _dev_w(W):
    return [to_dev(w) if w is not None else None for w in W]


def reference(d_args, cfg, W, snippet_weights=None, raw=None, **kw):
    """-> (losses (5,), rows (B,5) or None, grads dict or None, maps list).  With snippet weights by linearity over the
    one-snippet slices (weights sliced too): losses = sum_b w_b l_b, gradients and maps of snippet b times w_b."""
    tgt, src, K, disps, poses, logits = d_args
    fn = sfm_loss_pixel if raw is None else (lambda *a, **k: sfm_loss_pixel_raw(*a, **raw, **k))
    if snippet_weights is None:
        L, G = fn(tgt, src, K, disps, poses, logits, cfg, pixel_weights=W, **kw)
        return O.losses_vec(L), None, G, L['pixel_losses']
    B = src.shape[0]
    wb = np.asarray(snippet_weights, np.float64)
    cfg_b = copy.copy(cfg)
    cfg_b.B_global = cfg.B_global or B
    rows, per, maps = np.zeros((B, 5)), [], []
    for b in range(B):
        sl = slice(b, b + 1)
        L, G = fn(tgt[sl], src[sl], K[sl], [x[sl] for x in disps], poses[sl], [x[sl] for x in logits] if logits else None,
                  cfg_b, pixel_weights=[w[sl] if w is not None else None for w in W], **kw)
        rows[b] = O.losses_vec(L)
        per.append(G)
        maps.append(L['pixel_losses'])
    grads = None
    if per[0] is not None:
        grads = {}
        for k, v in per[0].items():
            if v is None:
                grads[k] = None
            elif isinstance(v, list):
                grads[k] = [np.concatenate([wb[b] * per[b][k][s].astype(np.float64) for b in range(B)]) for s in range(len(v))]
            else:
                grads[k] = np.concatenate([wb[b] * per[b][k].astype(np.float64) for b in range(B)])
    maps = [np.concatenate([wb[b] * maps[b][s] for b in range(B)]) for s in range(len(maps[0]))]
    return (wb[:, None] * rows).sum(0), rows, grads, maps


def _check(l, g, maps, ref, ns, exp):
    L, rows, G, M = ref
    np.testing.assert_allclose(host(l), L, rtol=1e-5, atol=1e-9)
    if rows is not None:
        np.testing.assert_allclose(host(g['snippet_losses']), rows, rtol=1e-5, atol=1e-9)
    for s in range(ns):
        assert_grad_close(host(maps[s]), M[s], what='map[%d]' % s)
    if G is None:
        return
    for s in range(ns):
        assert_grad_close(host(g['gdisps'][s]), G['gdisp'][s], what='gdisp[%d]' % s)
        if exp:
            assert_grad_close(host(g['glogits'][s]), G['glogits'][s], what='glogits[%d]' % s)
    assert_grad_close(host(g['gposes']), G['gpose'], what='gposes')


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('ns', [1, 4])
def test_kernels_match_oracle(cfg, S, ns):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, S, 128, 416, seed=1200 + S + 10 * ns, n_scales=ns, harsh=True)
    W = _pix_weights(d, 3 + S, null_scale=2 if ns > 1 else None)
    ref = reference(op_args(d, flags), O.LossConfig(n_scales=ns, **flags), W)
    l, g = make_op(flags, n_scales=ns, pixel_terms=True).forward_backward(*op_args(dev_inputs(d), flags), pixel_weights=_dev_w(W))
    _check(l, g, g['pixel_losses'], ref, ns, bool(flags['exp_reg']))


@pytest.mark.parametrize('cfg,shape', [('cfg4', (4, 2, 128, 416)), ('cfg2', (2, 2, 256, 832))])
def test_kernels_match_oracle_at_cfg4_and_cfg5_shapes(cfg, shape):
    flags = FLAGSETS[cfg]
    d = make_snippets(*shape, seed=1231)
    W = _pix_weights(d, 5)
    ref = reference(op_args(d, flags), O.LossConfig(**flags), W)
    l, g = make_op(flags, pixel_terms=True).forward_backward(*op_args(dev_inputs(d), flags), pixel_weights=_dev_w(W))
    _check(l, g, g['pixel_losses'], ref, 4, bool(flags['exp_reg']))


# 72 rows: scale heights 72 / 36 / 18 / 9; L1 tasks are runs of 32 pixels.  Per-pixel terms run the SSIM march with one
# warp per CTA and shared-memory records only.
FORCED = [('cfg2', h) for h in (8, 9, 10, 64)] + [(c, h) for c in ('cfg1', 'cfg4') for h in (1, 3, 8)]
_CACHE = {}


@pytest.mark.parametrize('cfg,hseg', FORCED)
@pytest.mark.parametrize('accum', [True, False])
@pytest.mark.parametrize('raw', [False, True])
def test_every_new_instance_under_forced_task_heights(cfg, hseg, accum, raw, monkeypatch):
    flags = dict(FLAGSETS[cfg], smooth_reg=0.1 if accum else 0.0)
    key = (cfg, accum, raw)
    if key not in _CACHE:
        d = make_snippets(3, 3, 72, 136, seed=1301, harsh=True)
        raw_disps, raw_poses = make_raw_seam(d, (1, 4), seed=1302)
        disps, poses = (raw_disps, raw_poses) if raw else (d['disps'], d['poses'])
        W = _pix_weights(d, 7, null_scale=1)
        args = (d['tgt'], d['src'], d['intrinsics'], disps, poses, d['logits'] if flags['exp_reg'] else None)
        ref = reference(args, O.LossConfig(**flags), W, raw=dict(raw_disp_scales=0xF if raw else 0, raw_pose=raw))
        _CACHE[key] = (d, disps, poses, W, ref)
    d, disps, poses, W, ref = _CACHE[key]
    monkeypatch.setenv('SFM_HSEG', str(hseg))
    args = (to_dev(d['tgt']), to_dev(d['src']), to_dev(d['intrinsics']), [to_dev(x) for x in disps], to_dev(poses),
            [to_dev(x) for x in d['logits']] if flags['exp_reg'] else None)
    op = make_op(flags, pixel_terms=True, raw_disp_scales=0xF if raw else 0, raw_pose=raw)
    l, g = op.forward_backward(*args, pixel_weights=_dev_w(W))
    _check(l, g, g['pixel_losses'], ref, 4, bool(flags['exp_reg']))
    # the forward-only instance of the same plan
    lf, mf = op.forward(*args, pixel_weights=_dev_w(W))
    _check(lf, None, mf, (ref[0], None, None, ref[3]), 4, False)


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
@pytest.mark.parametrize('unit', [False, True])
def test_unit_weights_are_bitwise_the_plain_step(cfg, unit, monkeypatch):
    flags = FLAGSETS[cfg]
    # the same plan for both: per-pixel terms run the SSIM march with one warp per CTA and shared-memory records, where
    # the plain step may pick the register-record or source-split instances
    for k, v in {'SFM_HSEG': '16', 'SFM_SSIM_NW': '1', 'SFM_SSIM_SREC': '1'}.items():
        monkeypatch.setenv(k, v)
    d = make_snippets(3, 2, 128, 416, seed=1401, harsh=True)
    g = dev_inputs(d)
    W = [to_dev(np.ones_like(x)) for x in d['logits']] if unit else None
    l, gg = make_op(flags, pixel_terms=True).forward_backward(*op_args(g, flags), pixel_weights=W)
    lp, gp = make_op(flags).forward_backward(*op_args(g, flags))
    if flags['ssim_rate']:
        # the SSIM instance with per-pixel terms is compiled separately: the losses are bitwise, gdisps agree to the last
        # bits (about 5 % of the entries differ, by at most 3e-4 relative, on entries where terms cancel)
        np.testing.assert_array_equal(host(l), host(lp))
        for s in range(4):
            assert_grad_close(host(gg['gdisps'][s]), host(gp['gdisps'][s]), rtol=1e-5, atol_rel=1e-6, what='gdisp[%d]' % s)
    else:
        check_same_as_plain(l, gg, lp, gp, 4, bool(flags['exp_reg']))
    # the maps are each pixel's share of the photometric loss
    r = flags['ssim_rate']
    tot = sum(float(host(m).astype(np.float64).sum()) for m in gg['pixel_losses'])
    ref = (1 - r) * float(host(lp)[1]) + r * float(host(lp)[4])
    assert abs(tot - ref) <= 1e-5 * abs(ref)


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
def test_forward_maps_are_those_of_forward_backward_and_reproducible(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 128, 416, seed=1501, harsh=True)
    g = dev_inputs(d)
    W = _dev_w(_pix_weights(d, 11, null_scale=3))
    op = make_op(flags, pixel_terms=True)
    _, gg = op.forward_backward(*op_args(g, flags), pixel_weights=W)
    l1, m1 = op.forward(*op_args(g, flags), pixel_weights=W)
    l2, m2 = op.forward(*op_args(g, flags), pixel_weights=W)
    for s in range(4):
        np.testing.assert_array_equal(host(m1[s]), host(gg['pixel_losses'][s]))
        np.testing.assert_array_equal(host(m1[s]), host(m2[s]))
    with pytest.raises(ValueError):
        make_op(flags).forward(*op_args(g, flags), pixel_weights=W)
    with pytest.raises(ValueError):
        op.forward(*op_args(g, flags), debug=True)
    with pytest.raises(ValueError):
        make_op(flags, pixel_terms=True, image_grads=True)


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_with_snippet_weights(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 128, 416, seed=1601, harsh=True)
    W = _pix_weights(d, 13)
    wb = np.array([0.7, 0.0, -1.3], np.float32)
    ref = reference(op_args(d, flags), O.LossConfig(**flags), W, snippet_weights=wb)
    op = make_op(flags, pixel_terms=True, snippet_terms=True)
    l, g = op.forward_backward(*op_args(dev_inputs(d), flags), pixel_weights=_dev_w(W), snippet_weights=to_dev(wb))
    _check(l, g, g['pixel_losses'], ref, 4, bool(flags['exp_reg']))
    lf, rows, maps = op.forward(*op_args(dev_inputs(d), flags), pixel_weights=_dev_w(W), snippet_weights=to_dev(wb))
    np.testing.assert_allclose(host(rows), ref[1], rtol=1e-5, atol=1e-9)
    for s in range(4):
        np.testing.assert_array_equal(host(maps[s]), host(g['pixel_losses'][s]))


def test_peer_sum_on_one_rank():
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=1701, harsh=True)
    g = dev_inputs(d)
    W = _dev_w(_pix_weights(d, 17))
    peer = PeerLossSum(0, 1)
    try:
        op = make_op(flags, pixel_terms=True)
        lr, gr = op.forward_backward(*op_args(g, flags), pixel_weights=W)
        lp, gp = op.forward_backward(*op_args(g, flags), pixel_weights=W, peer=peer)
        np.testing.assert_allclose(host(lp), host(lr), rtol=1e-6, atol=1e-12)
        for s in range(4):
            np.testing.assert_array_equal(host(gp['gdisps'][s]), host(gr['gdisps'][s]))
            np.testing.assert_array_equal(host(gp['pixel_losses'][s]), host(gr['pixel_losses'][s]))
    finally:
        torch.cuda.synchronize()
        peer.close()


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_intrinsics_grad_under_weights(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 128, 416, seed=1801, harsh=True)
    W = _pix_weights(d, 19)
    ref = reference(op_args(d, flags), O.LossConfig(**flags), W, want_intrinsics_grad=True)
    l, g = make_op(flags, pixel_terms=True, intrinsics_grad=True).forward_backward(*op_args(dev_inputs(d), flags),
                                                                                    pixel_weights=_dev_w(W))
    _check(l, g, g['pixel_losses'], ref, 4, bool(flags['exp_reg']))
    assert_grad_close(host(g['gintrinsics']), ref[2]['gintrinsics'], what='gintrinsics')


def test_edge_aware_smoothness():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=1901, harsh=True)
    W = _pix_weights(d, 23)
    ref = reference(op_args(d, flags), O.LossConfig(edge_aware_smooth=True, **flags), W)
    l, g = make_op(flags, pixel_terms=True, edge_aware_smooth=True).forward_backward(*op_args(dev_inputs(d), flags),
                                                                                    pixel_weights=_dev_w(W))
    _check(l, g, g['pixel_losses'], ref, 4, False)


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_tables_provided_and_reused_pyramid(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 64, 208, seed=2001, harsh=True)
    W = _pix_weights(d, 29)
    proj, kinv = oracle_tables(O, d)
    ref = reference(op_args(d, flags), O.LossConfig(**flags), W,
                    proj_override=np.concatenate([proj, np.zeros_like(proj[..., :1, :])], -2), kinv_override=kinv)
    g = dev_inputs(d)
    op = make_op(flags, pixel_terms=True)
    l, gg = op.forward_backward(*op_args(g, flags), proj=to_dev(proj), kinv=to_dev(kinv), pixel_weights=_dev_w(W))
    _check(l, gg, gg['pixel_losses'], ref, 4, bool(flags['exp_reg']))
    ref2 = reference(op_args(d, flags), O.LossConfig(**flags), W)
    op.build_pyramid(g['tgt'], g['src'])
    l2, g2 = op.forward_backward(*op_args(g, flags), reuse_pyramid=True, pixel_weights=_dev_w(W))
    _check(l2, g2, g2['pixel_losses'], ref2, 4, bool(flags['exp_reg']))


def test_cuda_graph_replay_with_changing_weights():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=2101, harsh=True)
    g = dev_inputs(d)
    op = make_op(flags, pixel_terms=True)
    W = [to_dev(np.ones_like(x)) for x in d['logits']]
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        op.forward_backward(*op_args(g, flags), pixel_weights=W)
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l, gg = op.forward_backward(*op_args(g, flags), pixel_weights=W)
    for k in range(3):
        Wk = _pix_weights(d, 200 + k)
        for s in range(4):
            W[s].copy_(torch.from_numpy(Wk[s]))
        graph.replay()
        torch.cuda.synchronize()
        _check(l, gg, gg['pixel_losses'], reference(op_args(d, flags), O.LossConfig(**flags), Wk), 4, False)


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_torch_adapter(cfg):
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 64, 208, seed=2201, harsh=True)
    Wn = _pix_weights(d, 31, null_scale=1)
    L, _, G, M = reference(op_args(d, flags), O.LossConfig(**flags), Wn)
    g = dev_inputs(d)
    gy = 0.37
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    poses = g['poses'].clone().requires_grad_(True)
    W = [to_dev(w).requires_grad_(s != 3) if w is not None else None for s, w in enumerate(Wn)]
    op = make_op(flags, pixel_terms=True)
    total, losses, maps = view_synthesis_loss(op, g['tgt'], g['src'], g['intrinsics'], disps, poses, g['logits'],
                                              pixel_weights=W)
    (gy * total).backward()
    np.testing.assert_allclose(host(losses), L, rtol=1e-5, atol=1e-9)
    for s in range(4):
        assert_grad_close(host(maps[s]), M[s], what='map[%d]' % s)
        if W[s] is not None and s != 3:
            np.testing.assert_allclose(host(W[s].grad), gy * host(maps[s]), rtol=1e-6)
        assert_grad_close(host(disps[s].grad), gy * G['gdisp'][s], what='disps[%d].grad' % s)
    assert W[3].grad is None
    assert_grad_close(host(poses.grad), gy * G['gpose'], what='poses.grad')
    # with snippet terms too: (total, losses, rows, maps)
    op2 = make_op(flags, pixel_terms=True, snippet_terms=True)
    out = view_synthesis_loss(op2, g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], g['logits'])
    assert len(out) == 4 and len(out[3]) == 4
    with pytest.raises(ValueError):
        view_synthesis_loss(make_op(flags), g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], g['logits'],
                            pixel_weights=W)
