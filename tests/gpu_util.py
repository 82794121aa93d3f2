"""Helpers for the -m gpu parity tests: torch is used purely as the device-memory allocator."""
import numpy as np


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def dev_inputs(d):
    return dict(tgt=to_dev(d['tgt']), src=to_dev(d['src']), intrinsics=to_dev(d['intrinsics']),
                disps=[to_dev(x) for x in d['disps']], poses=to_dev(d['poses']),
                logits=[to_dev(x) for x in d['logits']])


def host(x):
    return x.detach().cpu().numpy()


def oracle_tables(O, d, n_scales=4):
    """proj (B,S,ns,3,4) and kinv (B,ns,3,3) from the oracle's canonical host arithmetic."""
    B, S = d['poses'].shape[:2]
    proj = np.zeros((B, S, n_scales, 3, 4), np.float32)
    kinv = np.zeros((B, n_scales, 3, 3), np.float32)
    for s in range(n_scales):
        K = d['intrinsics'][:, s]
        kinv[:, s] = O.batch_inv3(K)
        for i in range(S):
            proj[:, i, s] = O.proj_tgt_to_src(d['poses'][:, i], K)[:, :3, :]
    return proj, kinv


FLAGSETS = {
    'cfg1': dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0),
    'cfg2': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
    'cfg4': dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0),
}


def make_op(flags, **kw):
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    return ViewSynthesisLoss(flags['smooth_reg'], flags['exp_reg'], flags['ssim_rate'], **kw)


def op_args(g, flags):
    """The loss arguments from a dict of inputs (device tensors or host arrays); logits only with the
    explainability term."""
    return (g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], g['logits'] if flags['exp_reg'] else None)


def check_same_as_plain(l, g, lp, gp, ns, exp):
    """Losses, gdisps, glogits of an operator with an opt-in gradient bitwise those of the operator without it; gposes
    to the order of the fp64 atomics (they vary from run to run in either operator)."""
    np.testing.assert_array_equal(host(l), host(lp))
    for s in range(ns):
        np.testing.assert_array_equal(host(g['gdisps'][s]), host(gp['gdisps'][s]))
        if exp:
            np.testing.assert_array_equal(host(g['glogits'][s]), host(gp['glogits'][s]))
    np.testing.assert_allclose(host(g['gposes']), host(gp['gposes']), rtol=1e-5, atol=1e-6 * np.abs(host(gp['gposes'])).max())
    assert 'gintrinsics' not in gp


def assert_grad_close(got, ref, rtol=1e-4, atol_rel=5e-5, what=''):
    """fp32 gradient bar of the north star: rtol 1e-4, plus an absolute floor relative to the largest
    reference entry (sums with different association, fp64 atomics)."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    atol = atol_rel * float(np.max(np.abs(ref))) + 1e-30
    bad = np.abs(got - ref) > (atol + rtol * np.abs(ref))
    assert not bad.any(), '%s: %d / %d entries off, max abs err %.3e (max |ref| %.3e)' % (
        what, int(bad.sum()), bad.size, float(np.max(np.abs(got - ref))), float(np.max(np.abs(ref))))
