"""-m gpu: gradient of the fused loss w.r.t. the camera intrinsics (sfm_intrinsics_grad,
ViewSynthesisLoss(intrinsics_grad=True)) against the numpy oracle, bitwise equality of everything else with the same
operator without the option, the supported input modes and combinations, backward(gy), sharding, CUDA-graph capture and
the torch adapter."""
import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests.gpu_util import FLAGSETS, make_op, op_args, check_same_as_plain, to_dev, dev_inputs, host, assert_grad_close

pytestmark = pytest.mark.gpu

@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_intrinsics_grad_matches_oracle(cfg, S, ns, harsh):
    flags = FLAGSETS[cfg]
    d = make_snippets(2, S, 128, 416, seed=700 + S + 10 * ns + harsh, n_scales=ns, harsh=harsh)
    L, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(n_scales=ns, **flags), want_intrinsics_grad=True)
    g = dev_inputs(d)
    lk, gk = make_op(flags, n_scales=ns, intrinsics_grad=True).forward_backward(*op_args(g, flags))
    lp, gp = make_op(flags, n_scales=ns).forward_backward(*op_args(g, flags))
    np.testing.assert_allclose(host(lk), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert tuple(gk['gintrinsics'].shape) == (2, ns, 3, 3)
    assert_grad_close(host(gk['gintrinsics']), G['gintrinsics'], what='gintrinsics')
    check_same_as_plain(lk, gk, lp, gp, ns, bool(flags['exp_reg']))


def test_intrinsics_grad_matches_oracle_at_cfg5_shape():
    flags = FLAGSETS['cfg2']
    d = make_snippets(1, 2, 256, 832, seed=771)
    L, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_intrinsics_grad=True)
    g = dev_inputs(d)
    lk, gk = make_op(flags, intrinsics_grad=True).forward_backward(*op_args(g, flags))
    np.testing.assert_allclose(host(lk), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert_grad_close(host(gk['gintrinsics']), G['gintrinsics'], what='gintrinsics')


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
def test_raw_disparity_and_raw_pose(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(2, 2, 128, 416, seed=781, harsh=True)
    raw_disps, raw_poses = make_raw_seam(d, (2, 3), seed=782)
    L, G, _ = O.sfm_loss_raw(d['tgt'], d['src'], d['intrinsics'], raw_disps, raw_poses, d['logits'], O.LossConfig(**flags),
                             raw_disp_scales=0xF, raw_pose=True, want_intrinsics_grad=True)
    args = (to_dev(d['tgt']), to_dev(d['src']), to_dev(d['intrinsics']), [to_dev(x) for x in raw_disps], to_dev(raw_poses),
            [to_dev(x) for x in d['logits']] if flags['exp_reg'] else None)
    lk, gk = make_op(flags, intrinsics_grad=True, raw_disp_scales=0xF, raw_pose=True).forward_backward(*args)
    np.testing.assert_allclose(host(lk), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert_grad_close(host(gk['gintrinsics']), G['gintrinsics'], what='gintrinsics (raw inputs)')


def test_edge_aware_smoothness():
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 128, 416, seed=791)
    L, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(edge_aware_smooth=True, **flags), want_intrinsics_grad=True)
    g = dev_inputs(d)
    lk, gk = make_op(flags, intrinsics_grad=True, edge_aware_smooth=True).forward_backward(*op_args(g, flags))
    lp, gp = make_op(flags, edge_aware_smooth=True).forward_backward(*op_args(g, flags))
    np.testing.assert_allclose(host(lk), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert_grad_close(host(gk['gintrinsics']), G['gintrinsics'], what='gintrinsics (edge-aware smoothness)')
    check_same_as_plain(lk, gk, lp, gp, 4, False)


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_together_with_image_grads(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(2, 2, 128, 416, seed=801, harsh=True)
    _, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_intrinsics_grad=True)
    g = dev_inputs(d)
    lk, gk = make_op(flags, intrinsics_grad=True, image_grads=True).forward_backward(*op_args(g, flags))
    li, gi = make_op(flags, image_grads=True).forward_backward(*op_args(g, flags))
    assert_grad_close(host(gk['gintrinsics']), G['gintrinsics'], what='gintrinsics (with image gradients)')
    check_same_as_plain(lk, gk, li, gi, 4, bool(flags['exp_reg']))
    np.testing.assert_array_equal(host(gk['gtgt']), host(gi['gtgt']))
    assert_grad_close(host(gk['gsrc']), host(gi['gsrc']), rtol=1e-5, what='gsrc')


def test_backward_with_gy_and_per_call_opt_out():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 3, 128, 416, seed=811)
    _, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_intrinsics_grad=True)
    g = dev_inputs(d)
    op = make_op(flags, intrinsics_grad=True)
    gy = 0.37
    out = op.backward(*op_args(g, flags), gy=torch.full((1,), gy, device='cuda'))
    assert_grad_close(host(out['gintrinsics']), gy * G['gintrinsics'], what='gintrinsics (backward, gy)')
    assert op.backward(*op_args(g, flags), intrinsics_grad=False)['gintrinsics'] is None
    _, fb = op.forward_backward(*op_args(g, flags))
    op.scale_grads(fb, torch.full((1,), gy, device='cuda'), 2, 3, 128, 416)
    assert_grad_close(host(fb['gintrinsics']), gy * G['gintrinsics'], what='gintrinsics (scale_grads)')
    assert op.forward_backward(*op_args(g, flags), intrinsics_grad=False)[1]['gintrinsics'] is None


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_shard_intrinsics_grad_is_the_slice_of_the_full_batch(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(4, 2, 64, 208, seed=821)
    g = dev_inputs(d)
    _, full = make_op(flags, intrinsics_grad=True).forward_backward(*op_args(g, flags))
    sl = slice(2, 4)
    gs = {k: (v[sl].contiguous() if not isinstance(v, list) else [x[sl].contiguous() for x in v]) for k, v in g.items()}
    _, shard = make_op(flags, intrinsics_grad=True, B_global=4).forward_backward(*op_args(gs, flags))
    assert_grad_close(host(shard['gintrinsics']), host(full['gintrinsics'])[sl], rtol=1e-5, what='gintrinsics shard')


def test_cuda_graph_replay():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 64, 208, seed=831, harsh=True)
    _, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_intrinsics_grad=True)
    g = dev_inputs(d)
    op = make_op(flags, intrinsics_grad=True)
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        op.forward_backward(*op_args(g, flags))
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            _, g2 = op.forward_backward(*op_args(g, flags))
    g2['gintrinsics'].fill_(float('nan'))
    for _ in range(3):                      # the cells are reset by every replayed step: replays do not accumulate
        graph.replay()
    torch.cuda.synchronize()
    assert_grad_close(host(g2['gintrinsics']), G['gintrinsics'], what='gintrinsics after replay')


def test_torch_adapter():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 128, 416, seed=841, harsh=True)
    g = dev_inputs(d)
    gy = 0.37

    def run(op, K):
        disps = [x.clone().requires_grad_(True) for x in g['disps']]
        loss, _ = view_synthesis_loss(op, g['tgt'], g['src'], K, disps, g['poses'])
        (gy * loss).backward()

    # intrinsics as a leaf
    _, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_intrinsics_grad=True)
    K = g['intrinsics'].clone().requires_grad_(True)
    run(make_op(flags, intrinsics_grad=True), K)
    assert_grad_close(host(K.grad), gy * G['gintrinsics'], what='intrinsics.grad')
    # the multi-scale intrinsics built from one (B,3,3) camera (get_multi_scale_intrinsics): the gradient chains on
    K0 = g['intrinsics'][:, 0].clone().requires_grad_(True)
    scale = torch.tensor([1.0, 1.0, 0.0], device='cuda')[:, None]
    Ks = torch.stack([K0 * (scale / 2 ** s + (1 - scale)) for s in range(4)], 1)
    d2 = dict(d, intrinsics=host(Ks))
    _, G2, _ = O.sfm_loss(*op_args(d2, flags), O.LossConfig(**flags), want_intrinsics_grad=True)
    run(make_op(flags, intrinsics_grad=True), Ks)
    ref0 = sum(G2['gintrinsics'][:, s] * np.array([1.0 / 2 ** s, 1.0 / 2 ** s, 1.0])[:, None] for s in range(4))
    assert_grad_close(host(K0.grad), gy * ref0, what='K0.grad')
    # not requested: the operator without the option, or intrinsics that do not require grad
    K = g['intrinsics'].clone().requires_grad_(True)
    run(make_op(flags), K)
    assert K.grad is None
    op = make_op(flags, intrinsics_grad=True)
    run(op, g['intrinsics'])
    assert g['intrinsics'].grad is None
