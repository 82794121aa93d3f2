"""-m gpu: gradients of the fused loss w.r.t. the target and source images (sfm_loss_forward_backward_images,
ViewSynthesisLoss(image_grads=True)) against the numpy oracle, bitwise equality of everything else with the plain fused
pass, every new marching-kernel instance under forced task heights, the supported input modes, run-to-run behaviour,
CUDA-graph capture and the torch adapter."""
import ctypes as C

import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests.gpu_util import (FLAGSETS, make_op, op_args, check_same_as_plain, to_dev, dev_inputs, host, oracle_tables,
                            assert_grad_close)

pytestmark = pytest.mark.gpu


def _check_images(grads, G):
    assert_grad_close(host(grads['gtgt']), G['gtgt'], what='gtgt')
    assert_grad_close(host(grads['gsrc']), G['gsrc'], what='gsrc')


@pytest.mark.parametrize('cfg', sorted(FLAGSETS))
@pytest.mark.parametrize('S', [1, 3])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_image_grads_match_oracle(cfg, S, ns, harsh):
    flags = FLAGSETS[cfg]
    d = make_snippets(2, S, 128, 416, seed=500 + S + 10 * ns + harsh, n_scales=ns, harsh=harsh)
    L, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(n_scales=ns, **flags), want_image_grads=True)
    g = dev_inputs(d)
    li, gi = make_op(flags, n_scales=ns, image_grads=True).forward_backward(*op_args(g, flags))
    lp, gp = make_op(flags, n_scales=ns).forward_backward(*op_args(g, flags))
    np.testing.assert_allclose(host(li), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    _check_images(gi, G)
    check_same_as_plain(li, gi, lp, gp, ns, bool(flags['exp_reg']))


def test_image_grads_match_oracle_at_cfg5_shape(monkeypatch):
    flags = FLAGSETS['cfg2']
    d = make_snippets(1, 2, 256, 832, seed=571)
    L, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_image_grads=True)
    g = dev_inputs(d)
    for forced in (True, False):          # the cfg5 plan, then whatever the policy picks for this batch
        for k, v in {'SFM_HSEG': '128', 'SFM_SSIM_NW': '1', 'SFM_SSIM_SREC': '1'}.items():
            monkeypatch.setenv(k, v) if forced else monkeypatch.delenv(k, raising=False)
        li, gi = make_op(flags, image_grads=True).forward_backward(*op_args(g, flags))
        np.testing.assert_allclose(host(li), O.losses_vec(L), rtol=1e-5, atol=1e-9)
        _check_images(gi, G)


# 72 rows: scale heights 72 / 36 / 18 / 9 (see test_gpu_ssim_rows.py for the head / tail shapes each hseg exercises).
# L1 tasks are runs of 32 pixels: 1, 3 and 8 runs per task.
FORCED = [('cfg2', h) for h in (8, 9, 10, 64)] + [(c, h) for c in ('cfg1', 'cfg4') for h in (1, 3, 8)]
_CACHE = {}


@pytest.mark.parametrize('cfg,hseg', FORCED)
@pytest.mark.parametrize('accum', [True, False])
@pytest.mark.parametrize('raw', [False, True])
def test_every_new_instance_under_forced_task_heights(cfg, hseg, accum, raw, monkeypatch):
    flags = dict(FLAGSETS[cfg], smooth_reg=0.1 if accum else 0.0)       # accum: the smoothness term initialises gdisp
    key = (cfg, accum, raw)
    if key not in _CACHE:
        d = make_snippets(2, 3, 72, 136, seed=601, harsh=True)
        raw_disps, _ = make_raw_seam(d, (1, 4), seed=602)
        disps = raw_disps if raw else d['disps']
        L, G, _ = O.sfm_loss_raw(d['tgt'], d['src'], d['intrinsics'], disps, d['poses'], d['logits'], O.LossConfig(**flags),
                                 raw_disp_scales=0xF if raw else 0, want_image_grads=True)
        _CACHE[key] = (d, disps, L, G)
    d, disps, L, G = _CACHE[key]
    monkeypatch.setenv('SFM_HSEG', str(hseg))
    args = (to_dev(d['tgt']), to_dev(d['src']), to_dev(d['intrinsics']), [to_dev(x) for x in disps], to_dev(d['poses']),
            [to_dev(x) for x in d['logits']] if flags['exp_reg'] else None)
    li, gi = make_op(flags, image_grads=True, raw_disp_scales=0xF if raw else 0).forward_backward(*args)
    np.testing.assert_allclose(host(li), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    _check_images(gi, G)
    # the rest against the existing instance under the same task height (its own oracle bar is test_gpu_ssim_rows.py)
    lp, gp = make_op(flags, raw_disp_scales=0xF if raw else 0).forward_backward(*args)
    check_same_as_plain(li, gi, lp, gp, 4, bool(flags['exp_reg']))


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_tables_provided_and_reused_pyramid(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(2, 2, 64, 208, seed=611, harsh=True)
    proj, kinv = oracle_tables(O, d)
    L, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_image_grads=True,
                         proj_override=np.concatenate([proj, np.zeros_like(proj[..., :1, :])], -2), kinv_override=kinv)
    g = dev_inputs(d)
    op = make_op(flags, image_grads=True)
    li, gi = op.forward_backward(*op_args(g, flags), proj=to_dev(proj), kinv=to_dev(kinv))
    np.testing.assert_allclose(host(li), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    _check_images(gi, G)
    # the pyramid built ahead of the loss call
    L2, G2, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_image_grads=True)
    op.build_pyramid(g['tgt'], g['src'])
    l2, g2 = op.forward_backward(*op_args(g, flags), reuse_pyramid=True)
    np.testing.assert_allclose(host(l2), O.losses_vec(L2), rtol=1e-5, atol=1e-9)
    _check_images(g2, G2)


@pytest.mark.parametrize('cfg', ['cfg2', 'cfg4'])
def test_shard_image_grads_are_the_slice_of_the_full_batch(cfg):
    flags = FLAGSETS[cfg]
    d = make_snippets(4, 2, 64, 208, seed=621)
    g = dev_inputs(d)
    _, full = make_op(flags, image_grads=True).forward_backward(*op_args(g, flags))
    sl = slice(2, 4)
    gs = {k: (v[sl].contiguous() if not isinstance(v, list) else [x[sl].contiguous() for x in v]) for k, v in g.items()}
    _, shard = make_op(flags, image_grads=True, B_global=4).forward_backward(*op_args(gs, flags))
    np.testing.assert_array_equal(host(shard['gtgt']), host(full['gtgt'])[sl])
    assert_grad_close(host(shard['gsrc']), host(full['gsrc'])[sl], rtol=1e-5, what='gsrc')


def test_one_image_only_and_run_to_run():
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 128, 416, seed=631, harsh=True)
    g = dev_inputs(d)
    op = make_op(flags, image_grads=True)
    _, a = op.forward_backward(*op_args(g, flags))
    _, b = op.forward_backward(*op_args(g, flags))
    np.testing.assert_array_equal(host(a['gtgt']), host(b['gtgt']))            # owned: no atomics
    assert_grad_close(host(a['gsrc']), host(b['gsrc']), rtol=1e-5, what='gsrc run to run')
    _, t = op.forward_backward(*op_args(g, flags), image_grads=('tgt',))
    _, s = op.forward_backward(*op_args(g, flags), image_grads=('src',))
    assert t['gsrc'] is None and s['gtgt'] is None
    np.testing.assert_array_equal(host(t['gtgt']), host(a['gtgt']))
    assert_grad_close(host(s['gsrc']), host(a['gsrc']), rtol=1e-5, what='gsrc alone')


def test_cuda_graph_replay():
    import torch
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 64, 208, seed=641)
    g = dev_inputs(d)
    op = make_op(flags, image_grads=True)
    ref_l, ref = op.forward_backward(*op_args(g, flags))
    torch.cuda.synchronize()
    ref = {k: host(ref[k]) for k in ('gtgt', 'gsrc')}
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        op.forward_backward(*op_args(g, flags))
        side.synchronize()
        with torch.cuda.graph(graph, stream=side):
            l2, g2 = op.forward_backward(*op_args(g, flags))
    for _ in range(3):                      # gsrc is re-zeroed inside the graph: replays do not accumulate
        graph.replay()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(host(l2), host(ref_l))
    np.testing.assert_array_equal(host(g2['gtgt']), ref['gtgt'])
    assert_grad_close(host(g2['gsrc']), ref['gsrc'], rtol=1e-5, what='gsrc after replay')


def test_unsupported_combination_returns_its_code():
    import torch
    from sfm_learner_chainer_b200 import lib as L
    with pytest.raises(ValueError):
        make_op(FLAGSETS['cfg2'], image_grads=True, edge_aware_smooth=True)
    so = L.load()
    d = L.SfmDesc(1, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, L.SFM_FLAG_IMAGE_GRADS | L.SFM_FLAG_EDGE_AWARE_SMOOTH)
    buf = torch.zeros(16, device='cuda')
    ig = L.SfmImageGrads(buf.data_ptr(), None)
    rc = so.sfm_loss_forward_backward_images(C.byref(d), C.byref(L.SfmInputs()), C.c_void_p(buf.data_ptr()),
                                             C.byref(L.SfmGrads()), C.byref(ig), C.c_void_p(buf.data_ptr()), None)
    assert rc == L.SFM_E_UNSUPPORTED


def test_torch_adapter():
    import torch
    from sfm_learner_chainer_b200.torch_adapter import view_synthesis_loss
    flags = FLAGSETS['cfg2']
    d = make_snippets(2, 2, 64, 208, seed=651, harsh=True)
    _, G, _ = O.sfm_loss(*op_args(d, flags), O.LossConfig(**flags), want_image_grads=True)
    g = dev_inputs(d)
    gy = 0.37

    def run(op, want_tgt, want_src):
        tgt = g['tgt'].clone().requires_grad_(want_tgt)
        src = g['src'].clone().requires_grad_(want_src)
        disps = [x.clone().requires_grad_(True) for x in g['disps']]
        loss, _ = view_synthesis_loss(op, tgt, src, g['intrinsics'], disps, g['poses'])
        (gy * loss).backward()
        return tgt, src

    tgt, src = run(make_op(flags, image_grads=True), True, True)
    assert_grad_close(host(tgt.grad), gy * G['gtgt'], what='tgt.grad')
    assert_grad_close(host(src.grad), gy * G['gsrc'], what='src.grad')
    tgt, src = run(make_op(flags, image_grads=True), False, True)
    assert tgt.grad is None
    assert_grad_close(host(src.grad), gy * G['gsrc'], what='src.grad alone')
    tgt, src = run(make_op(flags), True, True)
    assert tgt.grad is None and src.grad is None
