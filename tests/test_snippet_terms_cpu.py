"""-m "not gpu": per-snippet weights and per-snippet loss values (sfm_loss_snippets).

The weighted reference (tests/snippet_oracle.py, linearity over the oracle's one-snippet slices) is checked against
torch fp64 autograd of the independent restatement with the weights as a leaf, including d total / d w_b = l_b, and
against the plain oracle for all-ones weights.  The C ABI additions are checked for their struct size, workspace bytes
and argument errors without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests.snippet_oracle import sfm_loss_snippets
from tests.torch_restatement import torch_total

FLAGS = {
    'l1': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.0),
    'exp': dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
}
WEIGHTS = np.array([0.7, 0.0, -1.3])


def _args(d):
    return d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits']


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 2, 4])
@pytest.mark.parametrize('ns', [1, 4])
def test_weighted_reference_matches_torch_autograd(flags, S, ns):
    d = make_snippets(3, S, 32, 64, seed=40 + S + 10 * ns, n_scales=ns, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L, rows, G = sfm_loss_snippets(*_args(d), cfg, WEIGHTS, want_image_grads=True, want_intrinsics_grad=True)
    tgt = torch.from_numpy(d['tgt']).requires_grad_(True)
    src = torch.from_numpy(d['src']).requires_grad_(True)
    K = torch.from_numpy(d['intrinsics']).requires_grad_(True)
    w = torch.from_numpy(WEIGHTS).requires_grad_(True)
    B = 3
    # snippet b's image-dependent terms with the 1/B_global means: the restatement of the one-snippet slice over B
    tot = sum(w[b] * torch_total({k: (v[b:b + 1] if not isinstance(v, list) else [x[b:b + 1] for x in v]) for k, v in d.items()},
                                 cfg, tgt[b:b + 1], src[b:b + 1], K[b:b + 1]) / B for b in range(B))
    tot.backward()
    r = cfg.ssim_rate
    part = (1 - r) * rows[:, 1] + r * rows[:, 4]            # what the restatement covers of l_b
    np.testing.assert_allclose(tot.item(), (WEIGHTS * part).sum(), rtol=1e-9, atol=1e-12)
    np.testing.assert_allclose(w.grad.numpy(), part, rtol=1e-9, atol=1e-12)
    # d total / d w_b = l_b[0], and l_b[0] is formed from the row like the batch total
    np.testing.assert_allclose(rows[:, 0], part + rows[:, 2] + rows[:, 3], rtol=1e-12)
    np.testing.assert_allclose(L, WEIGHTS @ rows, rtol=1e-12)
    for got, ref in ((G['gtgt'], tgt.grad.numpy()), (G['gsrc'], src.grad.numpy()), (G['gintrinsics'], K.grad.numpy())):
        np.testing.assert_allclose(got, ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())
    assert not np.any(G['gtgt'][1]) and not np.any(G['gsrc'][1])    # weight 0
    for s in range(ns):
        assert not np.any(G['gdisp'][s][1])


@pytest.mark.parametrize('flags', sorted(FLAGS) + ['edge'])
@pytest.mark.parametrize('ns', [1, 4])
def test_all_ones_weights_equal_the_plain_oracle(flags, ns):
    edge = flags == 'edge'
    d = make_snippets(3, 2, 32, 64, seed=70 + ns, n_scales=ns, harsh=True, dtype=np.float64)
    cfg = O.LossConfig(n_scales=ns, edge_aware_smooth=edge, **FLAGS['ssim' if edge else flags])
    kw = dict(want_intrinsics_grad=True) if edge else dict(want_image_grads=True, want_intrinsics_grad=True)
    L0, G0, _ = O.sfm_loss(*_args(d), cfg, **kw)
    L, rows, G = sfm_loss_snippets(*_args(d), cfg, None, **kw)
    np.testing.assert_allclose(L, O.losses_vec(L0), rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(rows.sum(0), O.losses_vec(L0), rtol=1e-12, atol=1e-15)
    for k in ('gpose', 'gtgt', 'gsrc', 'gintrinsics', 'dP'):
        if k in G0:
            np.testing.assert_allclose(G[k], G0[k], rtol=1e-12, atol=1e-15 * np.abs(G0[k]).max())
    for k in ('gdisp', 'glogits'):
        if G0[k] is not None:
            for a, b in zip(G[k], G0[k]):
                np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-15 * np.abs(b).max())


def test_edge_aware_weighted_gradient_is_the_weighted_sum():
    """Edge-aware smoothness: gdisp of the weighted loss against central differences of the weighted total."""
    d = make_snippets(3, 1, 16, 32, seed=81, n_scales=2, dtype=np.float64)
    cfg = O.LossConfig(n_scales=2, edge_aware_smooth=True, smooth_reg=0.1)
    _, _, G = sfm_loss_snippets(*_args(d), cfg, WEIGHTS)

    def total(disps):
        return sfm_loss_snippets(d['tgt'], d['src'], d['intrinsics'], disps, d['poses'], d['logits'], cfg, WEIGHTS,
                                 want_grads=False)[0][0]
    rs = np.random.RandomState(2)
    eps = 1e-7
    for _ in range(12):
        s = rs.randint(0, 2)
        ix = tuple(rs.randint(0, n) for n in d['disps'][s].shape)
        vals = []
        for sgn in (1, -1):
            disps = [x.copy() for x in d['disps']]
            disps[s][ix] += sgn * eps
            vals.append(total(disps))
        fd = (vals[0] - vals[1]) / (2 * eps)
        assert abs(fd - G['gdisp'][s][ix]) <= 1e-4 * abs(G['gdisp'][s][ix]) + 1e-8, (s, ix, fd, G['gdisp'][s][ix])


def _lib():
    from sfm_learner_chainer_b200 import lib as L
    try:
        return L, L.load()
    except ImportError:
        pytest.skip('libsfmloss.so not built')


def _smooth_tasks(B, ns, H, W):
    hseg = 64
    while True:
        n = sum(B * -(-(W >> s) // 28) * -(-(H >> s) // hseg) for s in range(ns))
        if n >= 148 * 4 * 8 or hseg <= 8:
            return n
        hseg >>= 1


def test_abi_struct_size_and_workspace_bytes():
    L, so = _lib()
    assert C.sizeof(L.SfmSnippetTerms) == 16
    for B in (1, 3, 8, 40):
        d = L.SfmDesc(B, 2, 128, 416, 4, 0, 0.1, 0.0, 0.15, 0)
        plain = so.sfm_workspace_bytes(C.byref(d))
        d.flags = L.SFM_FLAG_SNIPPET_TERMS
        snip = so.sfm_workspace_bytes(C.byref(d))
        # the fp64 cells end on a 256-byte boundary; the snippet cells follow the dL/dP cells inside that block.  Then one
        # float per smoothness task (sfm_smooth_plan of common.cuh), also rounded to 256 bytes
        cells = (4 + B * 2 * 4 * 12) * 8
        grow = -(-(cells + 32 * B) // 256) * 256 - -(-cells // 256) * 256
        assert snip - plain == grow + -(-4 * _smooth_tasks(B, 4, 128, 416) // 256) * 256


def test_abi_argument_errors():
    L, so = _lib()
    buf = (C.c_float * 64)()
    ptr = C.cast(buf, C.c_void_p)
    terms = L.SfmSnippetTerms(ptr, None)
    d = L.SfmDesc(2, 2, 64, 208, 4, 0, 0.1, 0.0, 0.15, 0)
    # a non-NULL member without the flag
    rc = so.sfm_loss_snippets(C.byref(d), C.byref(L.SfmInputs()), C.byref(terms), ptr, None, None, ptr, None, None)
    assert rc == L.SFM_E_INVALID_DESC
    terms = L.SfmSnippetTerms(None, ptr)
    rc = so.sfm_loss_snippets(C.byref(d), C.byref(L.SfmInputs()), C.byref(terms), ptr, None, None, ptr, None, None)
    assert rc == L.SFM_E_INVALID_DESC
    # edge-aware smoothness with image gradients
    d.flags = L.SFM_FLAG_SNIPPET_TERMS | L.SFM_FLAG_IMAGE_GRADS | L.SFM_FLAG_EDGE_AWARE_SMOOTH
    ig = L.SfmImageGrads(ptr, None)
    rc = so.sfm_loss_snippets(C.byref(d), C.byref(L.SfmInputs()), C.byref(terms), ptr, C.byref(L.SfmGrads()), C.byref(ig),
                              ptr, None, None)
    assert rc == L.SFM_E_UNSUPPORTED
    # image gradients without the flag that sizes their workspace
    d.flags = L.SFM_FLAG_SNIPPET_TERMS
    rc = so.sfm_loss_snippets(C.byref(d), C.byref(L.SfmInputs()), C.byref(terms), ptr, C.byref(L.SfmGrads()), C.byref(ig),
                              ptr, None, None)
    assert rc == L.SFM_E_INVALID_DESC
    # losses_out is required
    rc = so.sfm_loss_snippets(C.byref(d), C.byref(L.SfmInputs()), C.byref(terms), None, None, None, ptr, None, None)
    assert rc == L.SFM_E_NULL_POINTER
