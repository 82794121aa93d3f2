"""-m gpu: per-snippet weights and per-snippet loss values (sfm_loss_snippets, ViewSynthesisLoss(snippet_terms=True))
against the weighted reference (tests/snippet_oracle.py), bitwise equality of the gradients with the plain step for
all-ones weights, every marching-kernel plan under forced task heights, the composition with the other options, the
padding recipe of a captured batch, CUDA-graph replay with changing weights, the torch adapter and the peer sum."""
import os
import sys

import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests.gpu_util import FLAGSETS, make_op, op_args, to_dev, dev_inputs, host, oracle_tables, assert_grad_close
from tests.snippet_oracle import sfm_loss_snippets

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _weights(B, seed):
    w = np.random.RandomState(seed).uniform(-0.5, 2.0, B).astype(np.float32)
    w[1 % B] = 0.0
    return w


def _check(l, g, L, rows, G, ns, exp, rows_dev=None, images=False):
    np.testing.assert_allclose(host(l), L, rtol=1e-5, atol=1e-9)
    if rows_dev is None:
        rows_dev = g['snippet_losses']
    np.testing.assert_allclose(host(rows_dev), rows, rtol=1e-5, atol=1e-9)
    if g is None:
        return
    for s in range(ns):
        assert_grad_close(host(g['gdisps'][s]), G['gdisp'][s], what='gdisp[%d]' % s)
        if exp:
            assert_grad_close(host(g['glogits'][s]), G['glogits'][s], what='glogits[%d]' % s)
    assert_grad_close(host(g['gposes']), G['gpose'], what='gposes')
    if images:
        assert_grad_close(host(g['gtgt']), G['gtgt'], what='gtgt')
        assert_grad_close(host(g['gsrc']), G['gsrc'], what='gsrc')


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_snippets_match_oracle(cfg, S, ns, harsh):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, S, 128, 416, seed=700 + S + 10 * ns + harsh, n_scales=ns, harsh=harsh)
    w = _weights(3, 7 + S)
    L, rows, G = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(n_scales=ns, **flags), w)
    l, g = make_op(flags, n_scales=ns, snippet_terms=True).forward_backward(*op_args(dev_inputs(d), flags),
                                                                            snippet_weights=to_dev(w))
    _check(l, g, L, rows, G, ns, bool(flags['exp_reg']))


def test_snippets_match_oracle_at_cfg5_shape(monkeypatch):
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 256, 832, seed=771)
    w = np.array([1.7, -0.4], np.float32)
    L, rows, G = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(**flags), w)
    g = dev_inputs(d)
    for k, v in {'SFM_HSEG': '128', 'SFM_SSIM_NW': '1', 'SFM_SSIM_SREC': '1'}.items():
        monkeypatch.setenv(k, v)
    l, gg = make_op(flags, snippet_terms=True).forward_backward(*op_args(g, flags), snippet_weights=to_dev(w))
    _check(l, gg, L, rows, G, 4, False)


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
@pytest.mark.parametrize('null_weights', [False, True])
def test_all_ones_gradients_are_bitwise_those_of_the_plain_step(cfg, null_weights):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 128, 416, seed=781, harsh=True)
    g = dev_inputs(d)
    w = None if null_weights else to_dev(np.ones(3, np.float32))
    ls, gs = make_op(flags, snippet_terms=True, image_grads=True).forward_backward(*op_args(g, flags), snippet_weights=w)
    lp, gp = make_op(flags, image_grads=True).forward_backward(*op_args(g, flags))
    for s in range(4):
        np.testing.assert_array_equal(host(gs['gdisps'][s]), host(gp['gdisps'][s]))
        if flags['exp_reg']:
            np.testing.assert_array_equal(host(gs['glogits'][s]), host(gp['glogits'][s]))
    np.testing.assert_array_equal(host(gs['gtgt']), host(gp['gtgt']))
    np.testing.assert_allclose(host(ls), host(lp), rtol=1e-6, atol=1e-12)
    np.testing.assert_allclose(host(gs['snippet_losses']).sum(0), host(ls), rtol=1e-6, atol=1e-12)


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
def test_forward_only(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 128, 416, seed=791, harsh=True)
    w = _weights(3, 3)
    L, rows, _ = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(**flags), w, want_grads=False)
    l, r = make_op(flags, snippet_terms=True).forward(*op_args(dev_inputs(d), flags), snippet_weights=to_dev(w))
    _check(l, None, L, rows, None, 4, False, rows_dev=r)
    with pytest.raises(ValueError):
        make_op(flags, snippet_terms=True).forward(*op_args(dev_inputs(d), flags), debug=True)


# 72 rows: scale heights 72 / 36 / 18 / 9; L1 tasks are runs of 32 pixels
FORCED = ([('cfg2', h, nw, srec) for h in (8, 9, 10, 64) for nw, srec in ((1, 1), (1, 0), (2, 1), (2, 0))]
          + [(c, h, None, None) for c in ('cfg1', 'cfg4') for h in (1, 3, 8)])
_CACHE = {}


@pytest.mark.parametrize('cfg,hseg,nw,srec', FORCED)
@pytest.mark.parametrize('accum', [True, False])
@pytest.mark.parametrize('raw', [False, True])
def test_every_plan_under_forced_task_heights(cfg, hseg, nw, srec, accum, raw, monkeypatch):
    flags = dict(FLAGSETS[cfg], smooth_reg=0.1 if accum else 0.0)
    key = (cfg, accum, raw)
    if key not in _CACHE:
        d = make_snippets(3, 3, 72, 136, seed=801, harsh=True)
        raw_disps, raw_poses = make_raw_seam(d, (1, 4), seed=802)
        disps, poses = (raw_disps, raw_poses) if raw else (d['disps'], d['poses'])
        w = _weights(3, 5)
        L, rows, G = sfm_loss_snippets(d['tgt'], d['src'], d['intrinsics'], disps, poses, d['logits'], O.LossConfig(**flags), w,
                                       raw=dict(raw_disp_scales=0xF if raw else 0, raw_pose=raw))
        _CACHE[key] = (d, disps, poses, w, L, rows, G)
    d, disps, poses, w, L, rows, G = _CACHE[key]
    monkeypatch.setenv('SFM_HSEG', str(hseg))
    if nw is not None:
        monkeypatch.setenv('SFM_SSIM_NW', str(nw))
        monkeypatch.setenv('SFM_SSIM_SREC', str(srec))
    args = (to_dev(d['tgt']), to_dev(d['src']), to_dev(d['intrinsics']), [to_dev(x) for x in disps], to_dev(poses),
            [to_dev(x) for x in d['logits']] if flags['exp_reg'] else None)
    op = make_op(flags, snippet_terms=True, raw_disp_scales=0xF if raw else 0, raw_pose=raw)
    l, g = op.forward_backward(*args, snippet_weights=to_dev(w))
    _check(l, g, L, rows, G, 4, bool(flags['exp_reg']))


FORCED_IMG = [('cfg2', h) for h in (8, 9, 10, 64)] + [(c, h) for c in ('cfg1', 'cfg4') for h in (1, 3, 8)]
_CACHE_IMG = {}


@pytest.mark.parametrize('cfg,hseg', FORCED_IMG)
@pytest.mark.parametrize('accum', [True, False])
@pytest.mark.parametrize('raw', [False, True])
def test_every_image_gradient_plan_under_forced_task_heights(cfg, hseg, accum, raw, monkeypatch):
    flags = dict(FLAGSETS[cfg], smooth_reg=0.1 if accum else 0.0)
    key = (cfg, accum, raw)
    if key not in _CACHE_IMG:
        d = make_snippets(3, 3, 72, 136, seed=901, harsh=True)
        raw_disps, _ = make_raw_seam(d, (1, 4), seed=902)
        disps = raw_disps if raw else d['disps']
        w = _weights(3, 9)
        L, rows, G = sfm_loss_snippets(d['tgt'], d['src'], d['intrinsics'], disps, d['poses'], d['logits'], O.LossConfig(**flags), w,
                                       raw=dict(raw_disp_scales=0xF if raw else 0), want_image_grads=True)
        _CACHE_IMG[key] = (d, disps, w, L, rows, G)
    d, disps, w, L, rows, G = _CACHE_IMG[key]
    monkeypatch.setenv('SFM_HSEG', str(hseg))
    args = (to_dev(d['tgt']), to_dev(d['src']), to_dev(d['intrinsics']), [to_dev(x) for x in disps], to_dev(d['poses']),
            [to_dev(x) for x in d['logits']] if flags['exp_reg'] else None)
    op = make_op(flags, snippet_terms=True, image_grads=True, raw_disp_scales=0xF if raw else 0)
    l, g = op.forward_backward(*args, snippet_weights=to_dev(w))
    _check(l, g, L, rows, G, 4, bool(flags['exp_reg']), images=True)


def test_peer_sum_with_image_gradients_and_forward_only_on_one_rank():
    """The peer sum of a world of one rank runs the epilogue's exchange on a single GPU: with weights, together with
    image gradients and forward only (grads == NULL through the C ABI), it gives the result of the step without it."""
    import ctypes as C
    import torch
    from sfm_learner_chainer_b200 import lib as L
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=911, harsh=True)
    g = dev_inputs(d)
    w = to_dev(_weights(3, 21))
    peer = PeerLossSum(0, 1)
    try:
        op = make_op(flags, snippet_terms=True, image_grads=True)
        lr, gr = op.forward_backward(*op_args(g, flags), snippet_weights=w)
        lp, gp = op.forward_backward(*op_args(g, flags), snippet_weights=w, peer=peer)
        np.testing.assert_allclose(host(lp), host(lr), rtol=1e-6, atol=1e-12)
        np.testing.assert_allclose(host(gp['snippet_losses']), host(gr['snippet_losses']), rtol=1e-6, atol=1e-12)
        for k in ('gtgt',):
            np.testing.assert_array_equal(host(gp[k]), host(gr[k]))
        for s in range(4):
            np.testing.assert_array_equal(host(gp['gdisps'][s]), host(gr['gdisps'][s]))
        assert_grad_close(host(gp['gsrc']), host(gr['gsrc']), rtol=1e-5, what='gsrc')
        # the plain operator through the same entry point: peer + image gradients used to be refused
        lpi, gpi = make_op(flags, image_grads=True).forward_backward(*op_args(g, flags), peer=peer)
        lri, gri = make_op(flags, image_grads=True).forward_backward(*op_args(g, flags))
        np.testing.assert_allclose(host(lpi), host(lri), rtol=1e-6, atol=1e-12)
        np.testing.assert_array_equal(host(gpi['gtgt']), host(gri['gtgt']))
        # forward only with the peer sum
        desc, inp = op._pack(*op_args(g, flags))
        losses = torch.empty(5, device='cuda')
        rows = torch.empty(3, 5, device='cuda')
        terms = L.SfmSnippetTerms(w.data_ptr(), rows.data_ptr())
        L.check(op._lib.sfm_loss_snippets(C.byref(desc), C.byref(inp), C.byref(terms), C.c_void_p(losses.data_ptr()), None, None,
                                          op._workspace(desc, g['tgt']), peer.handle,
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        lf, rf = op.forward(*op_args(g, flags), snippet_weights=w)
        torch.cuda.synchronize()
        np.testing.assert_allclose(host(losses), host(lf), rtol=1e-6, atol=1e-12)
        np.testing.assert_allclose(host(rows), host(rf), rtol=1e-6, atol=1e-12)
    finally:
        torch.cuda.synchronize()
        peer.close()


def test_edge_aware_smoothness():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=811, harsh=True)
    w = _weights(3, 11)
    L, rows, G = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(edge_aware_smooth=True, **flags), w)
    l, g = make_op(flags, snippet_terms=True, edge_aware_smooth=True).forward_backward(*op_args(dev_inputs(d), flags),
                                                                                      snippet_weights=to_dev(w))
    _check(l, g, L, rows, G, 4, False)


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_tables_provided_reused_pyramid_images_and_intrinsics(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 2, 64, 208, seed=821, harsh=True)
    w = _weights(3, 13)
    proj, kinv = oracle_tables(O, d)
    L, rows, G = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(**flags), w, want_image_grads=True,
                                   proj_override=np.concatenate([proj, np.zeros_like(proj[..., :1, :])], -2), kinv_override=kinv)
    g = dev_inputs(d)
    op = make_op(flags, snippet_terms=True, image_grads=True, intrinsics_grad=True)
    l, gg = op.forward_backward(*op_args(g, flags), proj=to_dev(proj), kinv=to_dev(kinv), snippet_weights=to_dev(w),
                                intrinsics_grad=False)
    _check(l, gg, L, rows, G, 4, bool(flags['exp_reg']), images=True)
    # the pyramid built ahead of the loss call, and the intrinsics gradient read from the same cells afterwards
    L2, rows2, G2 = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(**flags), w, want_image_grads=True,
                                      want_intrinsics_grad=True)
    op.build_pyramid(g['tgt'], g['src'])
    l2, g2 = op.forward_backward(*op_args(g, flags), reuse_pyramid=True, snippet_weights=to_dev(w))
    _check(l2, g2, L2, rows2, G2, 4, bool(flags['exp_reg']), images=True)
    assert_grad_close(host(g2['gintrinsics']), G2['gintrinsics'], what='gintrinsics')


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_shard_is_the_slice_of_the_full_weighted_batch(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(4, 2, 64, 208, seed=831)
    g = dev_inputs(d)
    w = to_dev(_weights(4, 17))
    _, full = make_op(flags, snippet_terms=True).forward_backward(*op_args(g, flags), snippet_weights=w)
    sl = slice(2, 4)
    gs = {k: (v[sl].contiguous() if not isinstance(v, list) else [x[sl].contiguous() for x in v]) for k, v in g.items()}
    _, shard = make_op(flags, snippet_terms=True, B_global=4).forward_backward(*op_args(gs, flags),
                                                                               snippet_weights=w[sl].contiguous())
    for s in range(4):
        np.testing.assert_array_equal(host(shard['gdisps'][s]), host(full['gdisps'][s])[sl])
    # the rows are sums of fp64 atomics: equal up to their order
    np.testing.assert_allclose(host(shard['snippet_losses']), host(full['snippet_losses'])[sl], rtol=1e-6, atol=1e-12)
    assert_grad_close(host(shard['gposes']), host(full['gposes'])[sl], rtol=1e-5, what='gposes')


def test_padding_recipe_and_zero_weight():
    """B_real = 3 real snippets run in a batch of B = 4: the padding is a copy of snippet 0 with weight 0, the real
    snippets weigh B / B_real, B_global stays B; the result is the loss and gradients of the 3-snippet batch."""
    flags = FLAGSETS['cfg4']
    d = make_snippets(3, 2, 128, 416, seed=841, harsh=True)
    L, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags))
    pad = {k: (np.concatenate([v, v[:1]]) if not isinstance(v, list) else [np.concatenate([x, x[:1]]) for x in v])
           for k, v in d.items()}
    w = np.array([4 / 3, 4 / 3, 4 / 3, 0.0], np.float32)
    l, g = make_op(flags, snippet_terms=True, image_grads=True).forward_backward(*op_args(dev_inputs(pad), flags),
                                                                                 snippet_weights=to_dev(w))
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    for s in range(4):
        assert_grad_close(host(g['gdisps'][s])[:3], G['gdisp'][s], what='gdisp[%d]' % s)
        assert_grad_close(host(g['glogits'][s])[:3], G['glogits'][s], what='glogits[%d]' % s)
        assert not host(g['gdisps'][s])[3].any() and not host(g['glogits'][s])[3].any()
    assert_grad_close(host(g['gposes'])[:3], G['gpose'], what='gposes')
    assert not host(g['gposes'])[3].any() and not host(g['gtgt'])[3].any()


def test_cuda_graph_replay_with_changing_weights():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=851, harsh=True)
    g = dev_inputs(d)
    op = make_op(flags, snippet_terms=True)
    w = to_dev(np.ones(3, np.float32))
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        op.forward_backward(*op_args(g, flags), snippet_weights=w)
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l, gg = op.forward_backward(*op_args(g, flags), snippet_weights=w)
    for k in range(3):
        wk = _weights(3, 100 + k)
        w.copy_(torch.from_numpy(wk))
        graph.replay()
        torch.cuda.synchronize()
        L, rows, G = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(**flags), wk)
        _check(l, gg, L, rows, G, 4, False)


def test_torch_adapter():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg4']
    d = make_snippets(3, 2, 64, 208, seed=861, harsh=True)
    wn = _weights(3, 19)
    L, rows, G = sfm_loss_snippets(*op_args(d, flags), O.LossConfig(**flags), wn, want_image_grads=True)
    g = dev_inputs(d)
    gy = 0.37
    tgt = g['tgt'].clone().requires_grad_(True)
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    poses = g['poses'].clone().requires_grad_(True)
    w = to_dev(wn).requires_grad_(True)
    op = make_op(flags, snippet_terms=True, image_grads=True)
    total, losses, rows_dev = view_synthesis_loss(op, tgt, g['src'], g['intrinsics'], disps, poses, g['logits'], snippet_weights=w)
    (gy * total).backward()
    np.testing.assert_allclose(host(losses), L, rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(host(w.grad), gy * host(rows_dev)[:, 0], rtol=1e-6)
    np.testing.assert_allclose(host(rows_dev)[:, 0], rows[:, 0], rtol=1e-5, atol=1e-9)
    assert_grad_close(host(tgt.grad), gy * G['gtgt'], what='tgt.grad')
    assert_grad_close(host(poses.grad), gy * G['gpose'], what='poses.grad')
    for s in range(4):
        assert_grad_close(host(disps[s].grad), gy * G['gdisp'][s], what='disps[%d].grad' % s)
    # without the option the return arity is unchanged
    out = view_synthesis_loss(make_op(flags), g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], g['logits'])
    assert len(out) == 2
    with pytest.raises(ValueError):
        view_synthesis_loss(make_op(flags), g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], g['logits'],
                            snippet_weights=w)


FLAGS2 = dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15)


def _worker(rank, world, out_dir, B, w_all):
    sys.path.insert(0, ROOT)
    import pickle
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum, ShardedViewSynthesisLoss, shard_arrays, shard_range

    def gather(b):                       # the handles through files: no process group needed
        with open(os.path.join(out_dir, 'h%d' % rank), 'wb') as f:
            pickle.dump(b, f)
        os.replace(os.path.join(out_dir, 'h%d' % rank), os.path.join(out_dir, 'handle%d' % rank))
        import time
        paths = [os.path.join(out_dir, 'handle%d' % r) for r in range(world)]
        while not all(os.path.exists(p) for p in paths):
            time.sleep(0.05)
        return [pickle.load(open(p, 'rb')) for p in paths]

    def barrier():
        import time
        open(os.path.join(out_dir, 'b%d_%d' % (rank, barrier.n)), 'w').close()
        while not all(os.path.exists(os.path.join(out_dir, 'b%d_%d' % (r, barrier.n))) for r in range(world)):
            time.sleep(0.05)
        barrier.n += 1
    barrier.n = 0

    torch.cuda.set_device(rank)
    d = make_snippets(B, 2, 128, 416, seed=890)
    mine = shard_arrays(dict(tgt=d['tgt'], src=d['src'], intrinsics=d['intrinsics'], disps=d['disps'], poses=d['poses'],
                             logits=d['logits']), B, rank, world)
    lo, hi = shard_range(B, rank, world)
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    args = (dev(mine['tgt']), dev(mine['src']), dev(mine['intrinsics']), [dev(x) for x in mine['disps']], dev(mine['poses']), None)
    w = dev(w_all[lo:hi])
    peer = PeerLossSum(rank, world, gather=gather, barrier=barrier)
    op = ShardedViewSynthesisLoss(peer=peer, B_global=B, snippet_terms=True, **FLAGS2)
    l, g, _ = op.forward_backward(*args, snippet_weights=w)
    op_i = ShardedViewSynthesisLoss(peer=peer, B_global=B, snippet_terms=True, image_grads=True, **FLAGS2)
    li, gi, _ = op_i.forward_backward(*args, snippet_weights=w)
    torch.cuda.synchronize()
    res = dict(losses=l.cpu().numpy(), rows=g['snippet_losses'].cpu().numpy(), gdisp0=g['gdisps'][0].cpu().numpy(),
               losses_img=li.cpu().numpy(), gtgt=gi['gtgt'].cpu().numpy(), lo=lo, hi=hi)
    barrier()
    peer.close()
    np.savez(os.path.join(out_dir, 'rank%d.npz' % rank), **res)


def test_two_gpus_uneven_shards_with_weights_and_peer(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip('needs >= 2 GPUs')
    import time
    import torch.multiprocessing as mp
    world, B = 2, 5                                   # uneven shards: 3 + 2
    w_all = _weights(B, 23)
    ctx = mp.spawn(_worker, args=(world, str(tmp_path), B, w_all), nprocs=world, join=False)
    deadline = time.time() + 240
    while not ctx.join(timeout=5):
        if time.time() > deadline:
            for pr in ctx.processes:
                pr.kill()
            pytest.fail('multi-GPU workers did not finish within 240 s')
    d = make_snippets(B, 2, 128, 416, seed=890)
    g = dev_inputs(d)
    lf, gf = make_op(FLAGS2, snippet_terms=True, image_grads=True).forward_backward(g['tgt'], g['src'], g['intrinsics'],
                                                                                  g['disps'], g['poses'], None,
                                                                                  snippet_weights=to_dev(w_all))
    z = [np.load(tmp_path / ('rank%d.npz' % r)) for r in range(world)]
    np.testing.assert_array_equal(z[0]['losses'], z[1]['losses'])
    for r in range(world):
        sl = slice(int(z[r]['lo']), int(z[r]['hi']))
        np.testing.assert_allclose(z[r]['losses'], host(lf), rtol=2e-6, atol=1e-9)
        np.testing.assert_allclose(z[r]['losses_img'], host(lf), rtol=2e-6, atol=1e-9)
        np.testing.assert_allclose(z[r]['rows'], host(gf['snippet_losses'])[sl], rtol=1e-6, atol=1e-12)
        np.testing.assert_array_equal(z[r]['gdisp0'], host(gf['gdisps'][0])[sl])
        np.testing.assert_array_equal(z[r]['gtgt'], host(gf['gtgt'])[sl])
