"""-m gpu: Monodepth2's axis-angle pose (SFM_FLAG_AXISANGLE_POSE, ViewSynthesisLoss(axisangle_pose=True,
invert_sources=...)).  The device tables against the numpy tables of tests/axisangle_oracle.py, the step against the same
step on those tables given as SFM_FLAG_TABLES_PROVIDED (bitwise), gposes and gintrinsics against the reference, the raw
poseout map, the compositions with the other options, Monodepth2's whole configuration against the torch restatement of
its code, CUDA-graph replay and the torch adapter."""
import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests import axisangle_oracle as AA
from tests.gpu_util import FLAGSETS, make_op, to_dev, dev_inputs, host, assert_grad_close

pytestmark = pytest.mark.gpu

SHAPES = [('cfg1', (4, 2, 128, 416)), ('cfg2', (4, 2, 128, 416)), ('cfg4', (4, 2, 128, 416)),
          ('cfg5', (2, 2, 256, 832)), ('cfg2', (2, 4, 128, 416))]


def _flags(cfg):
    return FLAGSETS['cfg2' if cfg == 'cfg5' else cfg]


def _with_angles(d, seed):
    """Axis-angle rows over the theta cases of the CPU tests (0, 1e-8, 1e-7, 1e-3, 0.1, > pi), the rest as made."""
    p = d['poses'].copy()
    rs = np.random.RandomState(seed)
    flat = p.reshape(-1, 6)
    for k, th in enumerate([0.0, 1e-8, 1e-7, 1e-3, 0.1, 3.5]):
        if k < flat.shape[0]:
            ax = rs.standard_normal(3)
            flat[k, :3] = th * ax / np.linalg.norm(ax)
    return dict(d, poses=p)


def _masks(S):
    return [(), (0,), tuple(range(S))]


def _args(g, exp=False):
    return (g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses']) + ((g['logits'],) if exp else ())


def _op(flags, inv, **kw):
    return make_op(flags, axisangle_pose=True, invert_sources=inv, **kw)


def _ulp(a, b):
    return np.abs(a.astype(np.float32).view(np.int32).astype(np.int64) - b.astype(np.float32).view(np.int32).astype(np.int64))


@pytest.mark.parametrize('cfg,shape', SHAPES)
def test_build_tables_match_numpy_bitwise(cfg, shape):
    """sin / cos are evaluated in fp64 by CUDA's sincos and by the host libm; they may differ in the last fp64 bit, which
    can move an fp32 rounding of R by one ulp.  Every other operation is individually rounded on both sides, so the
    tables must be bitwise equal except for such entries, and those are at most 1 ulp of R (a few ulp of P) off."""
    d = _with_angles(make_snippets(*shape, seed=7001), 7002)
    B, S, H, W = shape
    for inv in _masks(S):
        proj, kinv = AA.tables(d['poses'], d['intrinsics'], inv)
        gp, gk = _op(_flags(cfg), inv).build_tables(to_dev(d['poses']), to_dev(d['intrinsics']), H, W)
        np.testing.assert_array_equal(host(gk), kinv)
        got = host(gp)
        same = float(np.mean(got == proj))
        print('tables %s %s inv=%s: %.6f bitwise equal' % (cfg, shape, inv, same))
        assert same >= 0.999
        assert _ulp(got, proj).max() <= 4


@pytest.mark.parametrize('cfg,shape', SHAPES)
def test_step_against_tables_provided_and_reference(cfg, shape):
    """The step with the flag equals the step on the device-built tables bitwise (losses, gdisps, glogits); gposes and
    gintrinsics match the reference (gposes vary with the order of the fp64 atomics of the dL/dP cells)."""
    flags = _flags(cfg)
    exp = bool(flags['exp_reg'])
    d = _with_angles(make_snippets(*shape, seed=7101, harsh=True), 7102)
    g = dev_inputs(d)
    B, S, H, W = shape
    for inv in _masks(S):
        l, gg = _op(flags, inv, intrinsics_grad=True).forward_backward(*_args(g, exp))
        proj, kinv = _op(flags, inv).build_tables(g['poses'], g['intrinsics'], H, W)
        lt, gt = _op(flags, inv).forward_backward(*_args(g, exp), proj=proj, kinv=kinv)
        np.testing.assert_array_equal(host(l), host(lt))
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gt['gdisps'][s]))
            if exp:
                np.testing.assert_array_equal(host(gg['glogits'][s]), host(gt['glogits'][s]))
        L, G = AA.loss(*_args(d), O.LossConfig(**flags), invert_sources=inv, want_intrinsics_grad=True,
                       logits=d['logits'] if exp else None)
        np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9)
        for s in range(4):
            assert_grad_close(host(gg['gdisps'][s]), G['gdisp'][s], what='gdisp[%d]' % s)
        assert_grad_close(host(gg['gposes']), G['gpose'], what='gposes inv=%s' % (inv,))
        assert_grad_close(host(gt['gposes']), G['gpose'], what='gposes (tables provided) inv=%s' % (inv,))
        assert_grad_close(host(gg['gintrinsics']), G['gintrinsics'], what='gintrinsics inv=%s' % (inv,))


def test_raw_poseout_map_equals_reduce_then_plain_step():
    from sfm_learner_chainer_b200.functions import pose_reduce
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=7201, harsh=True)
    _, xp = make_raw_seam(d, (1, 4), seed=7202)
    g = dev_inputs(d)
    xpd = to_dev(xp)
    inv = (0,)
    l, gg = _op(flags, inv, raw_pose=True).forward_backward(g['tgt'], g['src'], g['intrinsics'], g['disps'], xpd)
    pv = pose_reduce(xpd, 2)
    lp, gp = _op(flags, inv).forward_backward(g['tgt'], g['src'], g['intrinsics'], g['disps'], pv)
    np.testing.assert_array_equal(host(l), host(lp))
    for s in range(4):
        np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gp['gdisps'][s]))
    gpv = host(gp['gposes']).astype(np.float64) * (0.01 / 4)
    assert_grad_close(host(gg['gposes']), np.broadcast_to(gpv.reshape(3, 12, 1, 1), xp.shape), what='raw gposes')


COMPOSITIONS = {
    'snippet': dict(snippet_terms=True),
    'pixel': dict(pixel_terms=True),
    'minrep_automask': dict(min_reprojection=True),
    'full_res': dict(min_reprojection=True, full_res_multiscale=True),
    'mean_norm': dict(mean_norm_smooth=True, edge_aware_smooth=True, edge_mean_abs=True),
    'border': dict(border_padding=True, min_reprojection=True),
}


@pytest.mark.parametrize('name', sorted(COMPOSITIONS))
def test_compositions_equal_tables_provided(name):
    """With every other option the flag only changes the tables and the pose chain: the step equals the same step on the
    device-built tables bitwise (losses, gdisps, selections, per-pixel maps, per-snippet rows), gposes to the atomics'
    order."""
    flags = FLAGSETS['cfg2']
    kw = COMPOSITIONS[name]
    d = _with_angles(make_snippets(3, 2, 128, 416, seed=7301, harsh=True), 7302)
    g = dev_inputs(d)
    inv = (0,)
    extra = {}
    if kw.get('snippet_terms'):
        extra['snippet_weights'] = to_dev(np.float32([0.5, 1.0, -2.0]))
    if kw.get('pixel_terms'):
        rs = np.random.RandomState(3)
        extra['pixel_weights'] = [to_dev(rs.rand(3, 2, 128 >> s, 416 >> s).astype(np.float32)) for s in range(4)]
    op = _op(flags, inv, **kw)
    l, gg = op.forward_backward(*_args(g), **extra)
    proj, kinv = op.build_tables(g['poses'], g['intrinsics'], 128, 416)
    if kw.get('full_res_multiscale'):               # every scale's table is built from K_0
        proj, kinv = _op(flags, inv).build_tables(g['poses'], g['intrinsics'][:, :1].repeat(1, 4, 1, 1).contiguous(), 128, 416)
    lt, gt = op.forward_backward(*_args(g), proj=proj, kinv=kinv, **extra)
    np.testing.assert_array_equal(host(l), host(lt))
    for s in range(4):
        np.testing.assert_array_equal(host(gg['gdisps'][s]), host(gt['gdisps'][s]))
    for key in ('selection', 'pixel_losses'):
        if key in gg:
            for a, b in zip(gg[key], gt[key]):
                np.testing.assert_array_equal(host(a), host(b))
    if 'snippet_losses' in gg:
        np.testing.assert_array_equal(host(gg['snippet_losses']), host(gt['snippet_losses']))
    ref = host(gt['gposes'])
    np.testing.assert_allclose(host(gg['gposes']), ref, rtol=1e-5, atol=1e-6 * np.abs(ref).max())


def test_pixel_terms_against_reference():
    flags = FLAGSETS['cfg2']
    d = _with_angles(make_snippets(3, 2, 128, 416, seed=7401, harsh=True), 7402)
    rs = np.random.RandomState(4)
    W = [rs.rand(3, 2, 128 >> s, 416 >> s).astype(np.float32) for s in range(4)]
    inv = (1,)
    L, G = AA.loss(*_args(d), O.LossConfig(**flags), invert_sources=inv, pixel_weights=W)
    l, g = _op(flags, inv, pixel_terms=True).forward_backward(*_args(dev_inputs(d)), pixel_weights=[to_dev(w) for w in W])
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert_grad_close(host(g['gposes']), G['gpose'], what='gposes')


def test_peer_step_on_one_rank():
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=7501, harsh=True)
    g = dev_inputs(d)
    peer = PeerLossSum(0, 1)
    try:
        op = _op(flags, (0,), min_reprojection=True)
        lr, gr = op.forward_backward(*_args(g))
        lp, gp = op.forward_backward(*_args(g), peer=peer)
        np.testing.assert_allclose(host(lp), host(lr), rtol=1e-6, atol=1e-12)
        for s in range(4):
            np.testing.assert_array_equal(host(gp['gdisps'][s]), host(gr['gdisps'][s]))
        ref = host(gr['gposes'])
        np.testing.assert_allclose(host(gp['gposes']), ref, rtol=1e-5, atol=1e-6 * np.abs(ref).max())
    finally:
        torch.cuda.synchronize()
        peer.close()


def test_monodepth2_configuration_against_torch_restatement():
    """Monodepth2's whole loss (min reprojection + automask, full resolution, mean-normalised edge-aware smoothness with
    its edge weight, border padding, axis-angle pose with the preceding source inverted) against the torch fp64
    restatement of its code; gposes against torch autograd with the poses as a leaf.  A pose gradient is a sum of about
    10^5 per-pixel terms of both signs, which the step accumulates in fp32 within each task and the restatement in fp64;
    on a B200 the two differed by 0.37 % of the largest entry with every selection equal (not broken down further), hence
    0.5 % of the largest entry.  A pixel whose selection differs near a tie would add its whole share.  The chain itself
    is checked to 1e-4 against the per-pixel reference above."""
    import torch
    from tests.torch_mean_norm_smooth_restatement import torch_smoothness
    from tests.torch_axisangle_restatement import torch_border_axisangle
    flags = dict(smooth_reg=1e-3, exp_reg=0.0, ssim_rate=0.85)
    d = make_snippets(2, 2, 64, 208, seed=7601, harsh=True)
    inv = (0,)
    l, g = _op(flags, inv, min_reprojection=True, full_res_multiscale=True, mean_norm_smooth=True, edge_aware_smooth=True,
               edge_mean_abs=True, border_padding=True).forward_backward(*_args(dev_inputs(d)))
    d64 = {k: (v.astype(np.float64) if isinstance(v, np.ndarray) else [x.astype(np.float64) for x in v])
           for k, v in d.items() if k != 'logits'}
    disps = [torch.from_numpy(x) for x in d64['disps']]
    poses = torch.from_numpy(d64['poses']).requires_grad_(True)
    phot, pixel, ssim, sels = torch_border_axisangle(d64, O.LossConfig(**flags), disps, poses, invert_sources=inv,
                                                     min_reprojection=True, full_res=True)
    smooth, _ = torch_smoothness(torch.from_numpy(d64['tgt']), disps, flags['smooth_reg'], edge=True, edge_mean_abs=True)
    lh = host(l)
    same = sum(int((host(a) == b.numpy()).sum()) for a, b in zip(g['selection'], sels))
    n = sum(b.numel() for b in sels)
    print('selection: %d of %d pixels differ' % (n - same, n))
    assert same >= 0.999 * n
    np.testing.assert_allclose(lh[1], pixel.item(), rtol=2e-4)
    np.testing.assert_allclose(lh[4], ssim.item(), rtol=2e-4)
    np.testing.assert_allclose(lh[2], smooth.item(), rtol=1e-4)
    np.testing.assert_allclose(lh[0], (phot + smooth).item(), rtol=2e-4)
    (phot + smooth).backward()
    ref = poses.grad.numpy()
    got = host(g['gposes'])
    print('gposes vs torch autograd: max abs err %.3e, max |ref| %.3e' % (np.abs(got - ref).max(), np.abs(ref).max()))
    assert_grad_close(got, ref, rtol=2e-3, atol_rel=5e-3, what='gposes vs torch autograd')


def test_cuda_graph_capture_and_bitwise_replay():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=7701, harsh=True)
    g = dev_inputs(d)
    op = _op(flags, (0,))
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
    d = _with_angles(make_snippets(3, 2, 64, 208, seed=7801, harsh=True), 7802)
    g = dev_inputs(d)
    gy = 0.37
    inv = (0, 1)
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    poses = g['poses'].clone().requires_grad_(True)
    total, losses = view_synthesis_loss(_op(flags, inv), g['tgt'], g['src'], g['intrinsics'], disps, poses)[:2]
    (gy * total).backward()
    L, G = AA.loss(*_args(d), O.LossConfig(**flags), invert_sources=inv)
    np.testing.assert_allclose(host(losses), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert_grad_close(host(poses.grad), gy * G['gpose'], what='poses.grad')


def test_invert_source_out_of_range_raises():
    d = make_snippets(2, 2, 64, 208, seed=7901)
    with pytest.raises(ValueError):
        _op(FLAGSETS['cfg2'], (2,)).forward_backward(*_args(dev_inputs(d)))
