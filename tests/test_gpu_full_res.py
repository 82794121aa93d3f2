"""-m gpu: the full-resolution multi-scale loss (SFM_FLAG_FULL_RES_MULTISCALE, ViewSynthesisLoss(full_res_multiscale=True))
against the reference composed from the existing ones (tests/full_res_oracle.py): the upsample stage against
F.interpolate, the warp bit for bit, losses and every gradient at the configuration shapes, Monodepth2's configuration
(minimum reprojection with auto-masking), the compositions with the other options, CUDA-graph replay, the torch adapter
and the unsupported combinations."""
import ctypes as C

import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.functions import upsample_disparity, disp_activation
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests import full_res_oracle as FR
from tests import min_reprojection_oracle as MR
from tests.gpu_util import FLAGSETS, make_op, to_dev, dev_inputs, host, oracle_tables, assert_grad_close

pytestmark = pytest.mark.gpu

NOEXP = dict(FLAGSETS['cfg4'], exp_reg=0.0)       # cfg4's flags without the explainability branch


def _args(g):
    return g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses']


def _op(flags, **kw):
    return make_op(flags, full_res_multiscale=True, **kw)


def _check(l, g, L, G, ns=4, k=False):
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    if G is None:
        return
    for s in range(ns):
        assert tuple(g['gdisps'][s].shape) == G['gdisp'][s].shape
        assert_grad_close(host(g['gdisps'][s]), G['gdisp'][s], what='gdisp[%d]' % s)
    assert_grad_close(host(g['gposes']), G['gpose'], what='gposes')
    if k:
        assert_grad_close(host(g['gintrinsics']), G['gintrinsics'], what='gintrinsics')
        assert not host(g['gintrinsics'])[:, 1:].any()


@pytest.mark.parametrize('hw,HW', [((64, 208), (128, 416)), ((16, 52), (128, 416)), ((4, 6), (36, 52)), ((32, 104), (256, 832))])
def test_upsample_stage(hw, HW):
    import torch
    import torch.nn.functional as F
    x = np.random.RandomState(7).uniform(0.01, 10, (3, 1) + hw).astype(np.float32)
    y = host(upsample_disparity(to_dev(x), *HW))
    np.testing.assert_array_equal(y, FR.upsample(x, *HW))        # the numpy pair is the device arithmetic
    ref64 = F.interpolate(torch.from_numpy(x.astype(np.float64)), size=HW, mode='bilinear', align_corners=False).numpy()
    np.testing.assert_allclose(y, ref64, rtol=1e-6)
    # torch's CUDA kernel does not round as the unfused arithmetic above does: on a B200 64-84 % of the values were bitwise
    # equal and 97.4-99.99 % within 2 ulp (the 4x6 -> 36x52 case lowest, max 1.1e-6 relative).  The shares are reported,
    # and every value must agree to 2e-6 relative
    ref = host(F.interpolate(to_dev(x), size=HW, mode='bilinear', align_corners=False))
    ulp = np.spacing(np.abs(ref).astype(np.float32))
    within = np.abs(y - ref) <= 2 * ulp
    print('upsample %s -> %s vs F.interpolate on the GPU: %.5f bitwise equal, %.5f within 2 ulp, max rel diff %.2e'
          % (hw, HW, np.mean(y == ref), np.mean(within), float(np.max(np.abs(y - ref) / np.abs(ref)))))
    np.testing.assert_allclose(y, ref, rtol=2e-6)


def _k0_tables(d):
    d0 = dict(d, intrinsics=np.repeat(d['intrinsics'][:, :1], d['intrinsics'].shape[1], 1))
    return oracle_tables(O, d0)


def test_warp_bit_exact_with_k0_tables():
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 128, 416, seed=5100, harsh=True)
    g = dev_inputs(d)
    proj, kinv = _k0_tables(d)
    l, dbg = _op(flags).forward(*_args(g), proj=to_dev(proj), kinv=to_dev(kinv), debug=True)
    cfg1 = O.LossConfig(ssim_rate=flags['ssim_rate'], n_scales=1)
    for s in range(4):
        u = d['disps'][0] if s == 0 else host(upsample_disparity(g['disps'][s], 128, 416))
        pov = np.concatenate([proj[:, :, :1], np.zeros_like(proj[:, :, :1, :1, :])], -2)
        _, _, ref = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'][:, :1], [u], d['poses'], None, cfg1, want_grads=False,
                               want_debug=True, proj_override=pov, kinv_override=kinv[:, :1])
        np.testing.assert_array_equal(host(dbg['u0'][s]), ref['u0'][0], err_msg='u0 scale %d' % s)
        np.testing.assert_array_equal(host(dbg['v0'][s]), ref['v0'][0], err_msg='v0 scale %d' % s)
        np.testing.assert_array_equal(host(dbg['inb'][s]).astype(bool), ref['inb'][0], err_msg='inb scale %d' % s)
        np.testing.assert_array_equal(host(dbg['P'][s]), ref['P'][0], err_msg='warped image scale %d' % s)
    L, _ = FR.sfm_loss_full_res(*_args(d), O.LossConfig(**flags), want_grads=False)
    np.testing.assert_allclose(host(l), O.losses_vec(L), rtol=1e-5, atol=1e-9)


@pytest.mark.parametrize('name,flags,shape,extra', [
    ('cfg1', FLAGSETS['cfg1'], (4, 2, 128, 416), {}),
    ('cfg2', FLAGSETS['cfg2'], (4, 2, 128, 416), {}),
    ('cfg4_noexp_S4', NOEXP, (3, 4, 128, 416), {}),
    ('cfg5_shape', FLAGSETS['cfg2'], (2, 2, 256, 832), {}),
    ('edge', FLAGSETS['cfg2'], (3, 2, 128, 416), dict(edge_aware_smooth=True)),
    ('l1_smooth', dict(FLAGSETS['cfg1'], smooth_reg=0.1), (3, 2, 72, 200), {}),
])
def test_losses_and_gradients_match_oracle(name, flags, shape, extra):
    d = make_snippets(*shape, seed=5200 + shape[1], harsh=True)
    l, g = _op(flags, intrinsics_grad=True, **extra).forward_backward(*_args(dev_inputs(d)))
    L, G = FR.sfm_loss_full_res(*_args(d), O.LossConfig(**flags, **extra), want_intrinsics_grad=True)
    _check(l, g, L, G, k=True)
    lf = _op(flags, **extra).forward(*_args(dev_inputs(d)))
    np.testing.assert_allclose(host(lf), host(l), rtol=1e-6, atol=1e-12)


@pytest.mark.parametrize('cfg,shape', [('cfg1', (3, 2, 128, 416)), ('cfg2', (3, 3, 128, 416)), ('cfg2', (2, 2, 256, 832))])
def test_monodepth2_configuration(cfg, shape):
    """minimum reprojection with auto-masking at full resolution: the selection away from near ties, and the losses and
    gradients of the exported selection."""
    flags = FLAGSETS[cfg]
    d = make_snippets(*shape, seed=5300, harsh=True)
    g = dev_inputs(d)
    l, gg = _op(flags, min_reprojection=True, automask=True, intrinsics_grad=True).forward_backward(*_args(g))
    sel = [host(x) for x in gg['selection']]
    B, S, _, H, W = d['src'].shape
    cfg1 = O.LossConfig(ssim_rate=flags['ssim_rate'], n_scales=1)
    amb_n = tot = 0
    for s in range(4):
        assert sel[s].shape == (B, H, W)
        u = d['disps'][0] if s == 0 else host(upsample_disparity(g['disps'][s], H, W))
        e, m, e_id = MR.errors(d['tgt'], d['src'], d['intrinsics'][:, :1], [u], d['poses'], cfg1)
        ref = MR.select(e[0], m[0], e_id[0], True)
        amb = MR.ambiguous(e[0], m[0], e_id[0], True)
        bad = (sel[s] != ref) & ~amb
        assert not bad.any(), 'scale %d: %d of %d pixels selected differently' % (s, int(bad.sum()), bad.size)
        amb_n += int(amb.sum())
        tot += amb.size
    assert amb_n <= 0.005 * tot, amb_n / tot
    assert any((x == -1).any() for x in sel)
    L, G = FR.sfm_loss_full_res(*_args(d), O.LossConfig(**flags), min_reprojection=True, selection=sel,
                                want_intrinsics_grad=True)
    _check(l, gg, L, G, k=True)


def test_snippet_and_pixel_terms():
    flags = FLAGSETS['cfg2']
    B, S, H, W = 3, 2, 64, 208
    d = make_snippets(B, S, H, W, seed=5400, harsh=True)
    g = dev_inputs(d)
    rs = np.random.RandomState(5401)
    pw = [rs.uniform(-0.5, 2.0, (B, S, H, W)).astype(np.float32) for _ in range(4)]
    pw[1] = None
    wb = np.array([0.7, 0.0, -1.3], np.float32)
    op = _op(flags, snippet_terms=True, pixel_terms=True)
    l, gg = op.forward_backward(*_args(g), snippet_weights=to_dev(wb), pixel_weights=[None if w is None else to_dev(w) for w in pw])
    cfg_b = O.LossConfig(B_global=B, **flags)
    rows = np.zeros((B, 5))
    for b in range(B):
        sl = slice(b, b + 1)
        L, G = FR.sfm_loss_full_res(d['tgt'][sl], d['src'][sl], d['intrinsics'][sl], [x[sl] for x in d['disps']],
                                    d['poses'][sl], cfg_b, pixel_weights=[None if w is None else w[sl] for w in pw])
        rows[b] = O.losses_vec(L)
        for s in range(4):
            assert gg['pixel_losses'][s].shape == (B, S, H, W)
            np.testing.assert_allclose(host(gg['pixel_losses'][s])[sl], wb[b] * L['pixel_losses'][s], rtol=1e-4,
                                       atol=1e-6 * np.abs(L['pixel_losses'][s]).max() + 1e-30)
            assert_grad_close(host(gg['gdisps'][s])[sl], wb[b] * G['gdisp'][s].astype(np.float64), what='gdisp[%d]' % s)
    np.testing.assert_allclose(host(gg['snippet_losses']), rows, rtol=1e-5, atol=1e-9)
    np.testing.assert_allclose(host(l), (wb[:, None] * rows).sum(0), rtol=1e-5, atol=1e-9)


def test_raw_inputs_equal_the_stages():
    """raw disparity (bits 0 and 1-3) and raw pose: the step equals the activation stage, then the upsample stage, then
    the plain full-resolution step."""
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 128, 416, seed=5500, harsh=True)
    raw_disps, raw_poses = make_raw_seam(d, (1, 4), seed=5501)
    g = dev_inputs(d)
    rd = [to_dev(x) for x in raw_disps]
    l, gg = _op(flags, raw_disp_scales=0xF).forward_backward(g['tgt'], g['src'], g['intrinsics'], rd, g['poses'])
    acts = [disp_activation(x, want_dact=True) for x in rd]
    lp, gp = _op(flags).forward_backward(g['tgt'], g['src'], g['intrinsics'], [a for a, _ in acts], g['poses'])
    np.testing.assert_array_equal(host(l), host(lp))
    for s in range(4):
        ref = host(gp['gdisps'][s]) * host(acts[s][1])
        np.testing.assert_allclose(host(gg['gdisps'][s]), ref, rtol=2e-6, atol=2e-6 * np.abs(ref).max())
    # the upsample stage of the activated map is what the step marches on
    for s in range(1, 4):
        np.testing.assert_array_equal(host(upsample_disparity(acts[s][0], 128, 416)),
                                      FR.upsample(host(acts[s][0]), 128, 416))
    # bits 1-3 with raw pose against the reference, fed the device's activation (numpy's tanh differs in the last bit,
    # which moves a few full-resolution pixels across a tap boundary)
    lr, gr = _op(flags, raw_disp_scales=0xE, raw_pose=True).forward_backward(
        g['tgt'], g['src'], g['intrinsics'], [g['disps'][0]] + rd[1:], to_dev(raw_poses))
    L, G = FR.sfm_loss_full_res(d['tgt'], d['src'], d['intrinsics'], [d['disps'][0]] + [host(a) for a, _ in acts[1:]],
                                raw_poses, O.LossConfig(**flags), raw_pose=True)
    G['gdisp'] = [G['gdisp'][0]] + [G['gdisp'][s].astype(np.float64) * host(acts[s][1]) for s in range(1, 4)]
    _check(lr, gr, L, G)


def test_reused_pyramid_tables_peer_and_recomputing_backward():
    import torch
    from sfm_learner_chainer_b200.distributed import PeerLossSum
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=5600, harsh=True)
    g = dev_inputs(d)
    for extra in ({}, dict(edge_aware_smooth=True)):
        op = _op(flags, **extra)
        l0, g0 = op.forward_backward(*_args(g))
        op.build_pyramid(g['tgt'], g['src'])
        l1, g1 = op.forward_backward(*_args(g), reuse_pyramid=True)
        np.testing.assert_array_equal(host(l1), host(l0))
        for s in range(4):
            np.testing.assert_array_equal(host(g1['gdisps'][s]), host(g0['gdisps'][s]))
    op = _op(flags)
    l0, g0 = op.forward_backward(*_args(g))
    proj, kinv = _k0_tables(d)
    l2, g2 = op.forward_backward(*_args(g), proj=to_dev(proj), kinv=to_dev(kinv))
    L, G = FR.sfm_loss_full_res(*_args(d), O.LossConfig(**flags))
    _check(l2, g2, L, G)
    gy = 0.37
    gb = op.backward(*_args(g), gy=to_dev(np.array([gy], np.float32)))
    for s in range(4):
        assert_grad_close(host(gb['gdisps'][s]), gy * G['gdisp'][s].astype(np.float64), what='backward gdisp[%d]' % s)
    assert_grad_close(host(gb['gposes']), gy * G['gpose'].astype(np.float64), what='backward gposes')
    peer = PeerLossSum(0, 1)
    try:
        lp, gp = op.forward_backward(*_args(g), peer=peer)
        np.testing.assert_allclose(host(lp), host(l0), rtol=1e-6, atol=1e-12)
        for s in range(4):
            np.testing.assert_array_equal(host(gp['gdisps'][s]), host(g0['gdisps'][s]))
    finally:
        torch.cuda.synchronize()
        peer.close()


def test_intrinsics_grad_central_differences():
    """gintrinsics[:, 0] against central differences of the device's own total (fp64 sums of fp32 terms)."""
    flags = dict(FLAGSETS['cfg2'], smooth_reg=0.0)
    d = make_snippets(1, 2, 32, 48, seed=5700, harsh=False)
    g = dev_inputs(d)
    op = _op(flags, intrinsics_grad=True)
    _, gg = op.forward_backward(*_args(g))
    gk = host(gg['gintrinsics'])
    L, G = FR.sfm_loss_full_res(*_args(d), O.LossConfig(**flags), want_intrinsics_grad=True)
    assert_grad_close(gk, G['gintrinsics'], what='gintrinsics')
    K = d['intrinsics'].astype(np.float64)
    for ix in ((0, 0, 0, 0), (0, 0, 1, 1), (0, 0, 0, 2), (0, 0, 1, 2)):
        eps = 1e-6 * abs(K[ix])
        vals = []
        for sgn in (1, -1):
            k = K.copy()
            k[ix] += sgn * eps
            Lk, _ = FR.sfm_loss_full_res(d['tgt'].astype(np.float64), d['src'].astype(np.float64), k,
                                         [x.astype(np.float64) for x in d['disps']], d['poses'].astype(np.float64),
                                         O.LossConfig(**flags), want_grads=False)
            vals.append(Lk['total_loss'])
        fd = (vals[0] - vals[1]) / (2 * eps)
        assert abs(fd - gk[ix]) <= 1e-2 * abs(fd) + 1e-3 * np.abs(gk).max(), (ix, fd, gk[ix])


def test_graph_replay_determinism_and_one_scale():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(3, 2, 64, 208, seed=5800, harsh=True)
    g = dev_inputs(d)
    op = _op(flags)
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        le, ge = op.forward_backward(*_args(g))
        le, gde = host(le), [host(x) for x in ge['gdisps']]
        la, ga = op.forward_backward(*_args(g))
        for s in range(4):
            np.testing.assert_array_equal(host(ga['gdisps'][s]), gde[s])     # two runs: bitwise equal gdisps
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l, gg = op.forward_backward(*_args(g))
    for _ in range(2):
        graph.replay()
        torch.cuda.synchronize()
        np.testing.assert_allclose(host(l), le, rtol=1e-6, atol=1e-12)
        for s in range(4):
            np.testing.assert_array_equal(host(gg['gdisps'][s]), gde[s])
    # n_scales = 1: the flag changes nothing
    g1 = dict(g, intrinsics=g['intrinsics'][:, :1].contiguous(), disps=g['disps'][:1])
    l1, gg1 = _op(flags, n_scales=1).forward_backward(*_args(g1))
    lp, gp = make_op(flags, n_scales=1).forward_backward(*_args(g1))
    np.testing.assert_array_equal(host(l1), host(lp))
    np.testing.assert_array_equal(host(gg1['gdisps'][0]), host(gp['gdisps'][0]))


def test_torch_adapter_matches_the_restatement():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    from tests.torch_full_res_restatement import torch_full_res
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 64, 208, seed=5900, harsh=True)
    g = dev_inputs(d)
    gy = 0.37
    disps = [x.clone().requires_grad_(True) for x in g['disps']]
    poses = g['poses'].clone().requires_grad_(True)
    total, losses, sel = view_synthesis_loss(_op(flags, min_reprojection=True), g['tgt'], g['src'], g['intrinsics'],
                                             disps, poses)
    assert all(tuple(x.shape) == (2, 64, 208) for x in sel)
    (gy * total).backward()
    d64 = {k: (v.astype(np.float64) if isinstance(v, np.ndarray) else [x.astype(np.float64) for x in v]) for k, v in d.items()}
    rd = [torch.from_numpy(x).requires_grad_(True) for x in d64['disps']]
    rp = torch.from_numpy(d64['poses']).requires_grad_(True)
    ref, _, _, _, rsel = torch_full_res(d64, O.LossConfig(**flags), rd, rp, torch.from_numpy(d64['intrinsics']),
                                        min_reprojection=True)
    (gy * ref).backward()
    same = all(np.array_equal(host(a), b.numpy()) for a, b in zip(sel, rsel))
    np.testing.assert_allclose(host(losses)[0], float(ref.detach()), rtol=1e-4 if same else 1e-3)
    for s in range(4):
        assert tuple(disps[s].grad.shape) == tuple(g['disps'][s].shape)
        if same:
            assert_grad_close(host(disps[s].grad), rd[s].grad.numpy(), what='disps[%d].grad' % s)
    if same:
        assert_grad_close(host(poses.grad), rp.grad.numpy(), what='poses.grad')


def test_unsupported_combinations():
    from sfm_learner_chainer_b200 import lib as Lb
    with pytest.raises(ValueError):
        _op(FLAGSETS['cfg4'])
    with pytest.raises(ValueError):
        _op(FLAGSETS['cfg2'], image_grads=True)
    flags = FLAGSETS['cfg4']
    d = make_snippets(2, 2, 64, 208, seed=6000)
    g = dev_inputs(d)
    so = Lb.load()
    desc = Lb.SfmDesc(2, 2, 64, 208, 4, 0, flags['smooth_reg'], flags['exp_reg'], flags['ssim_rate'],
                      Lb.SFM_FLAG_FULL_RES_MULTISCALE | Lb.SFM_FLAG_MIN_REPROJECTION)
    ws = to_dev(np.zeros(so.sfm_workspace_bytes(C.byref(desc)) // 4 + 64, np.float32))
    wsp = C.c_void_p((ws.data_ptr() + 255) // 256 * 256)
    inp = Lb.SfmInputs()
    inp.tgt, inp.src, inp.intrinsics, inp.poses = (g[k].data_ptr() for k in ('tgt', 'src', 'intrinsics', 'poses'))
    for s in range(4):
        inp.disps[s] = g['disps'][s].data_ptr()
        inp.logits[s] = g['logits'][s].data_ptr()
    losses = to_dev(np.zeros(5, np.float32))
    lp = C.c_void_p(losses.data_ptr())
    assert so.sfm_loss_forward(C.byref(desc), C.byref(inp), lp, None, wsp, None) == Lb.SFM_E_UNSUPPORTED
    assert b'exp_reg' in so.sfm_last_error()
    assert so.sfm_loss_weighted(C.byref(desc), C.byref(inp), None, None, lp, None, None, wsp, None, None) == Lb.SFM_E_UNSUPPORTED
    mr = Lb.SfmMinReprojection(1, 0)
    assert so.sfm_loss_min_reprojection(C.byref(desc), C.byref(inp), None, C.byref(mr), lp, None, wsp, None,
                                        None) == Lb.SFM_E_UNSUPPORTED
