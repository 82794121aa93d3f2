"""-m gpu: Monodepth2's image borders (SFM_FLAG_BORDER_PADDING, ViewSynthesisLoss(border_padding=True)) against the
reference (tests/border_oracle.py: the weighted, min-reprojection and full-resolution references under the flag):
losses and every gradient at the configuration shapes, the edge shapes of the SSIM strips and task segments, per-pixel
and per-snippet terms, minimum reprojection, Monodepth2's full configuration against the torch restatement of its code,
sfm_intrinsics_grad, the peer step, CUDA-graph replay, the torch adapter and the unsupported combinations."""
import ctypes as C

import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests import border_oracle as BO
from tests import min_reprojection_oracle as MR
from tests.gpu_util import FLAGSETS, make_op, to_dev, dev_inputs, host, assert_grad_close

pytestmark = pytest.mark.gpu


def _args(g):
    return g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses']


def _op(flags, **kw):
    return make_op(flags, border_padding=True, **kw)


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


@pytest.mark.parametrize('cfg,shape', [('cfg1', (4, 2, 128, 416)), ('cfg2', (4, 2, 128, 416)), ('cfg2', (2, 2, 256, 832)),
                                       ('cfg2', (2, 4, 128, 416))])
def test_at_config_shapes(cfg, shape):
    """cfg2 / cfg5 shapes: the three step kinds, losses rtol 1e-5 and every gradient rtol 1e-4; with intrinsics_grad."""
    flags = FLAGSETS[cfg]
    d = make_snippets(*shape, seed=5001, harsh=True)
    g = dev_inputs(d)
    L, G = BO.loss_pixel(*_args(d), O.LossConfig(**flags), want_intrinsics_grad=True)
    l, gg = _op(flags, intrinsics_grad=True).forward_backward(*_args(g))
    _check(l, gg, L, G, k=True)
    np.testing.assert_allclose(host(_op(flags).forward(*_args(g))), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    gb = _op(flags).backward(*_args(g), gy=to_dev(np.float32([0.5])))
    for s in range(4):
        assert_grad_close(host(gb['gdisps'][s]), 0.5 * G['gdisp'][s], what='backward gdisp[%d]' % s)


@pytest.mark.parametrize('W', [56, 57, 58, 55])          # W mod 28 = 0, 1, 2, 27: the last strips and their halos
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
def test_edge_widths(W, cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(2, 2, 20, W, seed=5100 + W, n_scales=1, harsh=True)
    L, G = BO.loss_pixel(*_args(d), O.LossConfig(n_scales=1, **flags))
    l, g = _op(flags, n_scales=1).forward_backward(*_args(dev_inputs(d)))
    _check(l, g, L, G, ns=1)


@pytest.mark.parametrize('raw', [False, True])
def test_four_row_coarsest_scale(raw):
    """A 4 x 14 coarsest scale under minimum reprojection with a fixed selection (source 0 everywhere), given as the
    one-hot per-pixel weights; with `raw` the disparity of scales 1 and 3 and the pose are the pre-activation maps."""
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 32, 116, seed=5201, harsh=True)                  # scale 3: 4 x 14
    rb = 0b1010 if raw else 0
    disps, poses = d['disps'], d['poses']
    if raw:
        rd, poses = make_raw_seam(d, (1, 4), seed=5202)
        disps = [rd[s] if (rb >> s) & 1 else disps[s] for s in range(4)]
    a = dict(d, disps=disps, poses=poses)
    L, G = BO.loss_min_reprojection(*_args(a), O.LossConfig(**flags), selection=[
        np.zeros((2, 32 >> s, 116 >> s), np.int8) for s in range(4)], raw_disp_scales=rb, raw_pose=raw)
    W1 = [to_dev(np.concatenate([np.ones((2, 1, 32 >> s, 116 >> s)), np.zeros((2, 1, 32 >> s, 116 >> s))], 1).astype(np.float32))
          for s in range(4)]
    l, g = _op(flags, pixel_terms=True, raw_disp_scales=rb, raw_pose=raw).forward_backward(*_args(dev_inputs(a)),
                                                                                          pixel_weights=W1)
    _check(l, g, L, G)


@pytest.mark.parametrize('hseg', ['1', '17'])            # task boundaries on rows 1 and h-2 (h = 19)
@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
def test_task_boundaries_at_rows_1_and_h_minus_2(monkeypatch, hseg, cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(2, 2, 19, 61, seed=5300, n_scales=1, harsh=True)
    L, G = BO.loss_pixel(*_args(d), O.LossConfig(n_scales=1, **flags))
    monkeypatch.setenv('SFM_HSEG', hseg)
    l, g = _op(flags, n_scales=1).forward_backward(*_args(dev_inputs(d)))
    _check(l, g, L, G, ns=1)


def test_pixel_weights_and_maps():
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=5401, harsh=True)
    rs = np.random.RandomState(4)
    W = [rs.rand(3, 2, 128 >> s, 416 >> s).astype(np.float32) for s in range(4)]
    W[2] = None
    L, G = BO.loss_pixel(*_args(d), O.LossConfig(**flags), pixel_weights=W)
    l, g = _op(flags, pixel_terms=True).forward_backward(*_args(dev_inputs(d)),
                                                         pixel_weights=[None if w is None else to_dev(w) for w in W])
    _check(l, g, L, G)
    for s in range(4):
        ref = L['pixel_losses'][s]
        np.testing.assert_allclose(host(g['pixel_losses'][s]), ref, rtol=1e-4, atol=1e-5 * np.abs(ref).max())


def test_snippet_terms():
    """sum_b w_b l_b with the rows l_b of the reference on each snippet alone (B_global = B)."""
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 128, 416, seed=5501, harsh=True)
    wb = np.array([0.7, -1.3], np.float32)
    l, g = _op(flags, snippet_terms=True).forward_backward(*_args(dev_inputs(d)), snippet_weights=to_dev(wb))
    rows = host(g['snippet_losses'])
    tot = 0.0
    for b in range(2):
        db = dict(d, tgt=d['tgt'][b:b + 1], src=d['src'][b:b + 1], intrinsics=d['intrinsics'][b:b + 1],
                  disps=[x[b:b + 1] for x in d['disps']], poses=d['poses'][b:b + 1])
        L, G = BO.loss_pixel(*_args(db), O.LossConfig(B_global=2, **flags))
        np.testing.assert_allclose(rows[b], O.losses_vec(L), rtol=1e-5, atol=1e-9)
        tot = tot + wb[b] * O.losses_vec(L)
        for s in range(4):
            assert_grad_close(host(g['gdisps'][s])[b:b + 1], wb[b] * G['gdisp'][s], what='gdisp[%d] b=%d' % (s, b))
    np.testing.assert_allclose(host(l), tot, rtol=1e-5, atol=1e-9)


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
@pytest.mark.parametrize('full_res', [False, True])
def test_min_reprojection(cfg, full_res):
    flags = FLAGSETS[cfg]
    d = make_snippets(3, 3, 128, 416, seed=5601, harsh=True)
    cfg_o = O.LossConfig(**flags)
    l, g = _op(flags, min_reprojection=True, full_res_multiscale=full_res).forward_backward(*_args(dev_inputs(d)))
    sel = _sel(g)
    if not full_res:
        e, m, e_id = BO.errors(*_args(d), cfg_o)
        amb_n = tot = 0
        for s in range(4):
            ref = MR.select(e[s], m[s], e_id[s], True)
            amb = MR.ambiguous(e[s], m[s], e_id[s], True)
            bad = (sel[s] != ref) & ~amb
            assert not bad.any(), 'scale %d: %d of %d pixels selected differently' % (s, int(bad.sum()), bad.size)
            amb_n += int(amb.sum())
            tot += amb.size
        assert amb_n <= 0.005 * tot, amb_n / tot
        assert all((x >= -1).all() for x in sel)                  # no pixel without a candidate at the borders
        L, G = BO.loss_min_reprojection(*_args(d), cfg_o, selection=sel)
    else:
        L, G = BO.loss_full_res(*_args(d), cfg_o, min_reprojection=True, selection=sel)
    _check(l, g, L, G)


def test_monodepth2_configuration_against_torch_restatement():
    """Monodepth2's loss (min reprojection + automask, full resolution, mean-normalised edge-aware smoothness with its
    edge weight, border padding) against the torch fp64 restatement of its code."""
    import torch
    from tests.torch_border_restatement import torch_border
    from tests.torch_mean_norm_smooth_restatement import torch_smoothness
    flags = dict(smooth_reg=1e-3, exp_reg=0.0, ssim_rate=0.85)
    d = make_snippets(2, 2, 64, 208, seed=5701, harsh=True)
    l, g = _op(flags, min_reprojection=True, full_res_multiscale=True, mean_norm_smooth=True, edge_aware_smooth=True,
               edge_mean_abs=True).forward_backward(*_args(dev_inputs(d)))
    d64 = {k: (v.astype(np.float64) if isinstance(v, np.ndarray) else [x.astype(np.float64) for x in v])
           for k, v in d.items() if k != 'logits'}
    disps = [torch.from_numpy(x) for x in d64['disps']]
    phot, pixel, ssim, sels = torch_border(d64, O.LossConfig(**flags), disps, torch.from_numpy(d64['poses']),
                                           min_reprojection=True, full_res=True)
    smooth, _ = torch_smoothness(torch.from_numpy(d64['tgt']), disps, flags['smooth_reg'], edge=True, edge_mean_abs=True)
    lh = host(l)
    same = sum(int((host(a) == b.numpy()).sum()) for a, b in zip(g['selection'], sels))
    assert same >= 0.999 * sum(b.numel() for b in sels)
    np.testing.assert_allclose(lh[1], pixel.item(), rtol=2e-4)
    np.testing.assert_allclose(lh[4], ssim.item(), rtol=2e-4)
    np.testing.assert_allclose(lh[2], smooth.item(), rtol=1e-4)
    np.testing.assert_allclose(lh[0], (phot + smooth).item(), rtol=2e-4)


def test_intrinsics_grad_and_peer_step_on_one_rank():
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=5801, harsh=True)
    g = dev_inputs(d)
    l, gg = _op(flags, B_global=5, intrinsics_grad=True, min_reprojection=True).forward_backward(*_args(g))
    L, G = BO.loss_min_reprojection(*_args(d), O.LossConfig(B_global=5, **flags), selection=_sel(gg),
                                        want_intrinsics_grad=True)
    _check(l, gg, L, G, k=True)
    peer = PeerLossSum(0, 1)
    try:
        op = _op(flags, min_reprojection=True)
        lr, gr = op.forward_backward(*_args(g))
        lp, gp = op.forward_backward(*_args(g), peer=peer)
        np.testing.assert_allclose(host(lp), host(lr), rtol=1e-6, atol=1e-12)
        for s in range(4):
            np.testing.assert_array_equal(host(gp['gdisps'][s]), host(gr['gdisps'][s]))
    finally:
        torch.cuda.synchronize()
        peer.close()


def test_cuda_graph_capture_and_bitwise_replay():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=5901, harsh=True)
    g = dev_inputs(d)
    op = _op(flags)
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        le, ge = op.forward_backward(*_args(g))
        le, ge = host(le), [host(x) for x in ge['gdisps']]
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l, gg = op.forward_backward(*_args(g))
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        np.testing.assert_array_equal(host(l), le)
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), ge[s])


def test_torch_adapter():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=6001, harsh=True)
    g = dev_inputs(d)
    gy = 0.37
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    poses = g['poses'].clone().requires_grad_(True)
    total, losses = view_synthesis_loss(_op(flags), g['tgt'], g['src'], g['intrinsics'], disps, poses)[:2]
    (gy * total).backward()
    L, G = BO.loss_pixel(*_args(d), O.LossConfig(**flags))
    np.testing.assert_allclose(host(losses), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    for s in range(4):
        assert_grad_close(host(disps[s].grad), gy * G['gdisp'][s], what='disps[%d].grad' % s)
    assert_grad_close(host(poses.grad), gy * G['gpose'], what='poses.grad')


def test_unsupported_combinations():
    from sfm_learner_chainer_b200 import lib as Lb
    flags = FLAGSETS['cfg4']
    d = make_snippets(2, 2, 64, 208, seed=6101)
    g = dev_inputs(d)
    with pytest.raises(ValueError):
        _op(flags)
    with pytest.raises(ValueError):
        _op(FLAGSETS['cfg2'], image_grads=True)
    with pytest.raises(ValueError):
        _op(FLAGSETS['cfg2']).forward(*_args(g), debug=True)
    so = Lb.load()
    desc = Lb.SfmDesc(2, 2, 64, 208, 4, 0, flags['smooth_reg'], flags['exp_reg'], flags['ssim_rate'], Lb.SFM_FLAG_BORDER_PADDING)
    ws = to_dev(np.zeros(so.sfm_workspace_bytes(C.byref(desc)) // 4 + 64, np.float32))
    inp = Lb.SfmInputs()
    inp.tgt, inp.src, inp.intrinsics, inp.poses = (g[k].data_ptr() for k in ('tgt', 'src', 'intrinsics', 'poses'))
    for s in range(4):
        inp.disps[s] = g['disps'][s].data_ptr()
        inp.logits[s] = g['logits'][s].data_ptr()
    losses = to_dev(np.zeros(5, np.float32))
    rc = so.sfm_loss_forward(C.byref(desc), C.byref(inp), C.c_void_p(losses.data_ptr()), None,
                             C.c_void_p((ws.data_ptr() + 255) // 256 * 256), None)
    assert rc == Lb.SFM_E_UNSUPPORTED
