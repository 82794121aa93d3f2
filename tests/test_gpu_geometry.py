"""-m gpu: SC-SfMLearner's geometry consistency term and self-discovered mask (sfm_loss_geometry,
ViewSynthesisLoss(geometry_consistency=True)) against the numpy reference (tests/geometry_oracle.py), bitwise identities
with the plain and the weighted step, the compositions with the other options, reproducibility, CUDA-graph replay, the
reverse-direction recipe against the torch restatement and the torch adapter."""

import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests import geometry_oracle as GO
from tests.gpu_util import FLAGSETS, make_op, op_args, to_dev, dev_inputs, host, assert_grad_close

pytestmark = pytest.mark.gpu

REG = 0.5


def _case(B, S, H, W, seed, harsh, ns=4):
    d = make_snippets(B, S, H, W, seed=seed, n_scales=ns, harsh=harsh)
    if harsh:
        d['poses'][:, 0, 5] -= np.float32(0.5)          # near points behind source 0's camera, some still in view
    return d, GO.make_src_disps(B, S, H, W, ns, seed + 7)


def _run(op, g, flags, sd, grads=True, **kw):
    if grads:
        return op.forward_backward(*op_args(g, flags), src_disps=sd, **kw)
    out = op.forward(*op_args(g, flags), src_disps=sd, **kw)
    return out[0], dict(geometry_diff=out[-1], snippet_losses=out[1] if len(out) > 2 else None)


def _check(l, gg, L, G, ns, what='', k=False):
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9, err_msg=what)
    for s in range(ns):
        np.testing.assert_allclose(host(gg['geometry_diff'][s]), L['geometry_diff'][s], rtol=1e-5, atol=1e-6,
                                   err_msg='%s diff[%d]' % (what, s))
    if G is None:
        return
    for s in range(ns):
        assert_grad_close(host(gg['gdisps'][s]), G['gdisp'][s], what='%s gdisp[%d]' % (what, s))
        assert_grad_close(host(gg['gsrc_disps'][s]), G['gsrc_disp'][s], what='%s gsrc_disps[%d]' % (what, s))
    assert_grad_close(host(gg['gposes']), G['gpose'], what=what + ' gposes')
    if k:
        assert_grad_close(host(gg['gintrinsics']), G['gintrinsics'], what=what + ' gintrinsics')


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('harsh', [False, True])
@pytest.mark.parametrize('self_mask', [False, True])
def test_parity_with_reference(cfg, S, harsh, self_mask):
    flags = FLAGSETS[cfg]
    d, sd = _case(2, S, 128, 416, 4100 + S + 10 * harsh, harsh)
    op = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=self_mask, intrinsics_grad=True)
    l, gg = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd])
    L, G = GO.loss(*op_args(d, flags)[:5], sd, O.LossConfig(**flags), geometry_reg=REG, self_mask=self_mask,
                   want_intrinsics_grad=True)
    _check(l, gg, L, G, 4, '%s S=%d harsh=%d mask=%d' % (cfg, S, harsh, self_mask), k=True)
    # forward only: the losses and maps of the gradient step
    lf, gf = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd], grads=False)
    np.testing.assert_array_equal(host(lf), host(l))
    for s in range(4):
        np.testing.assert_array_equal(host(gf['geometry_diff'][s]), host(gg['geometry_diff'][s]))


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
def test_zero_reg_without_mask_is_the_plain_step(cfg):
    flags = FLAGSETS[cfg]
    d, sd = _case(3, 2, 128, 416, 4201, True)
    g = dev_inputs(d)
    op = make_op(flags, geometry_consistency=True, geometry_reg=0.0, snippet_terms=True)
    w = to_dev(np.array([1.0, 0.5, -2.0], np.float32))
    l, gg = _run(op, g, flags, [to_dev(x) for x in sd], snippet_weights=w)
    lp, gp = make_op(flags, snippet_terms=True).forward_backward(*op_args(g, flags), snippet_weights=w)
    np.testing.assert_array_equal(host(l), host(lp))
    np.testing.assert_array_equal(host(gg['snippet_losses']), host(gp['snippet_losses']))
    for s in range(4):
        np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gp['gdisps'][s]))
        assert not host(gg['gsrc_disps'][s]).any()
    np.testing.assert_allclose(host(gg['gposes']), host(gp['gposes']), rtol=1e-5, atol=1e-6 * np.abs(host(gp['gposes'])).max())


@pytest.mark.parametrize('cfg', ['cfg1', 'cfg2'])
def test_self_mask_losses_are_the_weighted_step(cfg):
    flags = FLAGSETS[cfg]
    d, sd = _case(3, 2, 128, 416, 4301, True)
    g = dev_inputs(d)
    l, gg = _run(make_op(flags, geometry_consistency=True, geometry_reg=0.0, self_mask=True), g, flags,
                 [to_dev(x) for x in sd])
    M = [1.0 - x for x in gg['geometry_diff']]
    lw, gw = make_op(flags, pixel_terms=True).forward_backward(*op_args(g, flags), pixel_weights=M)
    np.testing.assert_array_equal(host(l), host(lw))


def test_snippet_weights_peer_and_reproducibility():
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d, sd = _case(3, 2, 128, 416, 4401, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    wb = np.array([1.5, 0.0, -0.75], np.float32)
    op = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True, snippet_terms=True)
    l, gg = _run(op, g, flags, sdd, snippet_weights=to_dev(wb))
    # the reference by linearity over the one-snippet slices
    cfg = O.LossConfig(B_global=3, **flags)
    tot = np.zeros(5)
    for b in range(3):
        sl = slice(b, b + 1)
        L, G = GO.loss(d['tgt'][sl], d['src'][sl], d['intrinsics'][sl], [x[sl] for x in d['disps']], d['poses'][sl],
                       [x[sl] for x in sd], cfg, geometry_reg=REG, self_mask=True)
        row = O.losses_vec(L)
        np.testing.assert_allclose(host(gg['snippet_losses'])[b], row, rtol=1e-5, atol=1e-9)
        tot += wb[b] * row
        for s in range(4):
            assert_grad_close(host(gg['gdisps'][s])[sl], wb[b] * G['gdisp'][s], what='gdisp[%d] b=%d' % (s, b))
            assert_grad_close(host(gg['gsrc_disps'][s])[sl], wb[b] * G['gsrc_disp'][s], what='gsrc[%d] b=%d' % (s, b))
        assert_grad_close(host(gg['gposes'])[sl], wb[b] * G['gpose'], what='gposes b=%d' % b)
    np.testing.assert_allclose(host(l), tot, rtol=1e-5, atol=1e-9)
    # gdisps are bitwise reproducible from run to run; the peer sum on one rank gives the same step
    l2, g2 = _run(op, g, flags, sdd, snippet_weights=to_dev(wb))
    peer = PeerLossSum(0, 1)
    try:
        l3, g3 = _run(op, g, flags, sdd, snippet_weights=to_dev(wb), peer=peer)
        torch.cuda.synchronize()
    finally:
        peer.close()
    np.testing.assert_allclose(host(l3), host(l), rtol=1e-6, atol=1e-12)
    for s in range(4):
        np.testing.assert_array_equal(host(g2['gdisps'][s]), host(gg['gdisps'][s]))
        np.testing.assert_array_equal(host(g3['gdisps'][s]), host(gg['gdisps'][s]))
        np.testing.assert_array_equal(host(g2['geometry_diff'][s]), host(gg['geometry_diff'][s]))
        np.testing.assert_allclose(host(g2['gsrc_disps'][s]), host(gg['gsrc_disps'][s]), rtol=1e-5,
                                   atol=1e-6 * np.abs(host(gg['gsrc_disps'][s])).max())


def test_raw_disparity_and_pose():
    """raw disparity and raw pose: the step equals the activation and pose stages followed by the plain geometry step
    (D_diff bit for bit, losses to summation order, gradients to rounding), and that step matches the reference fed the
    device's activation.  numpy's tanh differs from CUDA's in the last bit; where the source disparity is rough D' moves
    by many ulp with the target's disparity, so the reference is not fed its own activation."""
    from sfm_learner_chainer_b200 import disp_activation, pose_reduce
    flags = FLAGSETS['cfg2']
    B, S = 3, 2
    d, sd = _case(B, S, 72, 136, 4501, True)
    raw_d, raw_p = make_raw_seam(d, seed=4501)
    sdd = [to_dev(x) for x in sd]
    rd, rp = [to_dev(x) for x in raw_d], to_dev(raw_p)
    g = dict(tgt=to_dev(d['tgt']), src=to_dev(d['src']), intrinsics=to_dev(d['intrinsics']), disps=rd, poses=rp,
             logits=None)
    geo = dict(geometry_consistency=True, geometry_reg=REG, self_mask=True)
    l, gg = _run(make_op(flags, raw_disp_scales=0xF, raw_pose=True, **geo), g, flags, sdd)
    acts = [disp_activation(x, want_dact=True) for x in rd]
    gp_in = dict(g, disps=[a for a, _ in acts], poses=pose_reduce(rp, S))
    lp, gp = _run(make_op(flags, **geo), gp_in, flags, sdd)
    np.testing.assert_allclose(host(l), host(lp), rtol=5e-7, atol=0)
    for s in range(4):
        np.testing.assert_array_equal(host(gg['geometry_diff'][s]), host(gp['geometry_diff'][s]))
        ref = host(gp['gdisps'][s]).astype(np.float64) * host(acts[s][1]).astype(np.float64)
        assert_grad_close(host(gg['gdisps'][s]), ref, rtol=2e-6, atol_rel=1e-7, what='gdisp[%d]' % s)
        assert_grad_close(host(gg['gsrc_disps'][s]), host(gp['gsrc_disps'][s]), rtol=1e-5, atol_rel=1e-6,
                          what='gsrc_disps[%d]' % s)
    n = int(np.prod(raw_p.shape[2:]))
    gpr = host(gp['gposes']).astype(np.float64).reshape(B, 6 * S, 1, 1) * (0.01 / n)
    assert tuple(gg['gposes'].shape) == raw_p.shape
    assert_grad_close(host(gg['gposes']), np.broadcast_to(gpr, raw_p.shape), rtol=2e-6, atol_rel=1e-7, what='gposes')
    L, G = GO.loss(d['tgt'], d['src'], d['intrinsics'], [host(a) for a, _ in acts], host(gp_in['poses']), sd,
                   O.LossConfig(**flags), geometry_reg=REG, self_mask=True)
    _check(lp, gp, L, G, 4, 'device activation')


@pytest.mark.parametrize('inv', [(), (0,), (0, 1)])
def test_axisangle_pose_with_invert_bits(inv):
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 128, 416, 4601, False)
    d['poses'][:, :, :3] *= 5.0
    op = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True, axisangle_pose=True,
                 invert_sources=inv, intrinsics_grad=True)
    l, gg = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd])
    L, G = GO.loss(*op_args(d, flags)[:5], sd, O.LossConfig(**flags), geometry_reg=REG, self_mask=True,
                   want_intrinsics_grad=True, invert_sources=inv)
    _check(l, gg, L, G, 4, 'axisangle %r' % (inv,), k=True)


def test_mean_norm_edge_smoothness():
    """The smoothness options add the same term as on the plain step: the difference of the geometry steps with and
    without them is that of the plain steps."""
    flags = FLAGSETS['cfg2']
    d, sd = _case(3, 2, 128, 416, 4701, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    sm = dict(edge_aware_smooth=True, mean_norm_smooth=True, edge_mean_abs=True)
    off = dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=flags['ssim_rate'])
    geo = dict(geometry_consistency=True, geometry_reg=REG, self_mask=True)
    la, ga = _run(make_op(flags, **geo, **sm), g, flags, sdd)
    lb, gb = _run(make_op(off, **geo), g, off, sdd)
    lc, gc = make_op(flags, **sm).forward_backward(*op_args(g, flags))
    ld, gd = make_op(off).forward_backward(*op_args(g, off))
    np.testing.assert_array_equal(host(la)[2], host(lc)[2])
    np.testing.assert_allclose(host(la)[[1, 3, 4]], host(lb)[[1, 3, 4]], rtol=1e-6)
    for s in range(4):
        assert_grad_close(host(ga['gdisps'][s]) - host(gb['gdisps'][s]), host(gc['gdisps'][s]) - host(gd['gdisps'][s]),
                          what='smooth gdisp[%d]' % s, atol_rel=1e-4)


def test_tables_provided_and_intrinsics_grad():
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 128, 416, 4801, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    op = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True, intrinsics_grad=True)
    l, gg = _run(op, g, flags, sdd)
    proj, kinv = op.build_tables(g['poses'], g['intrinsics'], 128, 416)
    lt, gt = _run(op, g, flags, sdd, proj=proj, kinv=kinv, intrinsics_grad=False)
    np.testing.assert_array_equal(host(lt), host(l))
    for s in range(4):
        np.testing.assert_array_equal(host(gt['gdisps'][s]), host(gg['gdisps'][s]))
        np.testing.assert_array_equal(host(gt['geometry_diff'][s]), host(gg['geometry_diff'][s]))
    L, G = GO.loss(*op_args(d, flags)[:5], sd, O.LossConfig(**flags), geometry_reg=REG, self_mask=True,
                   want_intrinsics_grad=True)
    assert_grad_close(host(gg['gintrinsics']), G['gintrinsics'], what='gintrinsics')


def test_cuda_graph_replay_is_bitwise():
    import torch
    flags = FLAGSETS['cfg2']
    d, sd = _case(3, 2, 128, 416, 4901, True)
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    op = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True)
    l0, g0 = _run(op, g, flags, sdd)
    l0, g0 = host(l0), {s: host(g0['gdisps'][s]) for s in range(4)}
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
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), g0[s])


def test_reverse_direction_recipe():
    """INTEGRATION.md §6: the reverse direction is a second call on B*S snippets with S = 1 (target = source i, source =
    the target, disparities swapped, the axis-angle pose with its invert bit flipped, snippet weights S so that the
    means are per pair).  The two calls together give the restatement's two-direction loss and gradients.

    Every entry is checked at the default bar against the two calls of the per-pixel reference (fp32 arithmetic, the
    device's decisions), and against the torch fp64 restatement wherever the two references agree.  At this seed they
    disagree, on the CPU, at 2 of 26624 entries of gdisp[0], in the photometric part alone (they disagree there with
    geometry_reg = 0 and no mask too): a pixel on a kink of the photometric term that fp32 and fp64 resolve differently."""
    import torch
    from tests.torch_axisangle_restatement import transform_rows
    from tests.torch_geometry_restatement import torch_total_geometry
    flags = dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.15)
    B, S, H, W = 2, 2, 64, 208
    d, sd = _case(B, S, H, W, 5001, False)
    d['poses'][:, :, :3] *= 5.0
    g = dev_inputs(d)
    sdd = [to_dev(x) for x in sd]
    fwd = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True, axisangle_pose=True)
    lf, gf = _run(fwd, g, flags, sdd)
    rev = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True, axisangle_pose=True,
                  invert_sources=(0,), snippet_terms=True)
    tgt_r = g['src'].reshape(B * S, 3, H, W).contiguous()
    src_r = g['tgt'][:, None].expand(B, S, 3, H, W).reshape(B * S, 1, 3, H, W).contiguous()
    K_r = g['intrinsics'][:, None].expand(B, S, 4, 3, 3).reshape(B * S, 4, 3, 3).contiguous()
    disps_r = [x.reshape(B * S, 1, H >> s, W >> s).contiguous() for s, x in enumerate(sdd)]
    sd_r = [x.expand(B, S, H >> s, W >> s).reshape(B * S, 1, H >> s, W >> s).contiguous() for s, x in enumerate(g['disps'])]
    poses_r = g['poses'].reshape(B * S, 1, 6).contiguous()
    w = torch.full((B * S,), float(S), device='cuda')
    lr, gr = rev.forward_backward(tgt_r, src_r, K_r, disps_r, poses_r, None, src_disps=sd_r, snippet_weights=w)
    total = float(host(lf)[0] + host(lr)[0])
    # the restatement: every pair in both directions, means over B h w
    t = lambda a: torch.from_numpy(np.asarray(a, np.float64)).requires_grad_(True)
    disps = [t(x) for x in d['disps']]
    srcd = [t(x) for x in sd]
    poses = t(d['poses'])
    K = torch.from_numpy(d['intrinsics'].astype(np.float64))
    tgt64, src64 = torch.from_numpy(d['tgt'].astype(np.float64)), torch.from_numpy(d['src'].astype(np.float64))
    cfg = O.LossConfig(**flags)
    ref, _ = torch_total_geometry(tgt64, src64, K, disps, poses, srcd, cfg, REG, True,
                                  rot=lambda p, i: transform_rows(p, False))
    for i in range(S):
        r, _ = torch_total_geometry(src64[:, i], tgt64[:, None], K, [x[:, i:i + 1] for x in srcd], poses[:, i:i + 1],
                                    [x for x in disps], cfg, REG, True, rot=lambda p, j: transform_rows(p, True))
        ref = ref + r
    ref.backward()
    np.testing.assert_allclose(total, float(ref.detach()), rtol=1e-4)
    # the per-pixel reference of the two calls (the reverse one with B_global = B: weights S over B*S snippets)
    Lf, Gf = GO.loss(*op_args(d, flags)[:5], sd, cfg, geometry_reg=REG, self_mask=True, invert_sources=())
    bc = lambda x, shape: np.ascontiguousarray(np.broadcast_to(x, shape))
    Lr, Gr = GO.loss(d['src'].reshape(B * S, 3, H, W), bc(d['tgt'][:, None], (B, S, 3, H, W)).reshape(B * S, 1, 3, H, W),
                     bc(d['intrinsics'][:, None], (B, S, 4, 3, 3)).reshape(B * S, 4, 3, 3),
                     [x.reshape(B * S, 1, H >> s, W >> s) for s, x in enumerate(sd)], d['poses'].reshape(B * S, 1, 6),
                     [bc(x, (B, S, H >> s, W >> s)).reshape(B * S, 1, H >> s, W >> s) for s, x in enumerate(d['disps'])],
                     O.LossConfig(B_global=B, **flags), geometry_reg=REG, self_mask=True, invert_sources=(0,))
    np.testing.assert_allclose(total, Lf['total_loss'] + Lr['total_loss'], rtol=1e-5)
    off = lambda got, r: np.abs(got - r) > 5e-4 * np.abs(r).max() + 2e-3 * np.abs(r)
    for s in range(4):
        sh = (B, S, H >> s, W >> s)
        pairs = ((host(gf['gdisps'][s]) + host(gr['gsrc_disps'][s]).reshape(sh).sum(1)[:, None],
                  Gf['gdisp'][s] + Gr['gsrc_disp'][s].reshape(sh).sum(1)[:, None], disps[s].grad.numpy(), 'gdisp[%d]' % s),
                 (host(gf['gsrc_disps'][s]) + host(gr['gdisps'][s]).reshape(sh),
                  Gf['gsrc_disp'][s] + Gr['gdisp'][s].reshape(sh), srcd[s].grad.numpy(), 'gsrc[%d]' % s))
        for got, ref_o, ref_t, what in pairs:
            assert_grad_close(got, ref_o, what=what)
            agree = ~off(ref_o, ref_t)
            assert (~agree).sum() <= 4, '%s: the references disagree at %d of %d entries' % (what, (~agree).sum(), agree.size)
            bad = off(got, ref_t) & agree
            assert not bad.any(), '%s: %d entries off the torch restatement' % (what, int(bad.sum()))
    gp = host(gf['gposes']) + host(gr['gposes']).reshape(B, S, 6)
    assert_grad_close(gp, Gf['gpose'] + Gr['gpose'].reshape(B, S, 6), what='gposes')
    assert_grad_close(gp, poses.grad.numpy(), rtol=2e-3, atol_rel=5e-4, what='gposes vs torch autograd')


def test_torch_adapter_src_disps_grad():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 128, 416, 5101, True)
    g = dev_inputs(d)
    op = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True)
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    srcd = [to_dev(x).requires_grad_(True) for x in sd]
    poses = g['poses'].clone().requires_grad_(True)
    res = view_synthesis_loss(op, g['tgt'], g['src'], g['intrinsics'], disps, poses, src_disps=srcd)
    total, losses, diffs = res[0], res[1], res[-1]
    (3.0 * total).backward()
    L, G = GO.loss(*op_args(d, flags)[:5], sd, O.LossConfig(**flags), geometry_reg=REG, self_mask=True)
    np.testing.assert_allclose(host(losses), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert len(diffs) == 4 and not diffs[0].requires_grad
    for s in range(4):
        assert_grad_close(host(srcd[s].grad), 3.0 * G['gsrc_disp'][s], what='src_disps.grad[%d]' % s)
        assert_grad_close(host(disps[s].grad), 3.0 * G['gdisp'][s], what='disps.grad[%d]' % s)
    assert_grad_close(host(poses.grad), 3.0 * G['gpose'], what='poses.grad')


def test_cfg5_shape():
    flags = FLAGSETS['cfg2']
    d, sd = _case(2, 2, 256, 832, 5201, True)
    op = make_op(flags, geometry_consistency=True, geometry_reg=REG, self_mask=True)
    l, gg = _run(op, dev_inputs(d), flags, [to_dev(x) for x in sd])
    L, G = GO.loss(*op_args(d, flags)[:5], sd, O.LossConfig(**flags), geometry_reg=REG, self_mask=True)
    _check(l, gg, L, G, 4, 'cfg5 shape')
