"""-m "not gpu": image gradients of the fused loss (d total / d tgt_img, d total / d src_imgs).

The oracle's analytic gtgt / gsrc (O.sfm_loss(want_image_grads=True)) are checked against torch fp64 autograd through
an independent restatement of the forward (tests/torch_restatement.py), against central differences of the oracle
itself, and the resize adjoint against <Rx, y> = <x, R^T y>.  The C ABI additions are checked for their argument
errors without a device."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests.torch_restatement import torch_total

FLAGS = {
    'l1': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.0),
    'exp': dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
}


def _data(B, S, H, W, ns, harsh, seed=0):
    d = make_snippets(B, S, H, W, seed=seed, n_scales=ns, harsh=harsh, dtype=np.float64)
    return d


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 2, 4])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_oracle_image_grads_match_torch_autograd(flags, S, ns, harsh):
    d = _data(2, S, 32, 64, ns, harsh, seed=S + 10 * ns)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L, G, _ = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg, want_image_grads=True)
    tgt = torch.from_numpy(d['tgt']).requires_grad_(True)
    src = torch.from_numpy(d['src']).requires_grad_(True)
    tot = torch_total(d, cfg, tgt, src, torch.from_numpy(d['intrinsics']))
    tot.backward()
    # the restatement leaves out only image-independent terms
    np.testing.assert_allclose(tot.item(), L['total_loss'] - L['smooth_loss'] - L['exp_loss'], rtol=1e-9, atol=1e-12)
    for got, ref in ((G['gtgt'], tgt.grad.numpy()), (G['gsrc'], src.grad.numpy())):
        assert got.dtype == np.float64
        np.testing.assert_allclose(got, ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())
    assert np.abs(G['gsrc']).max() > 0 and np.abs(G['gtgt']).max() > 0


@pytest.mark.parametrize('flags', sorted(FLAGS))
def test_oracle_image_grads_central_differences(flags):
    """fp64 central differences of the reported total on sampled entries away from kinks (floor flips cannot
    happen: the grid does not depend on the images; |P - T|, the SSIM clip and the all-zero mask can)."""
    d = _data(1, 2, 32, 64, 4, True, seed=7)
    cfg = O.LossConfig(n_scales=4, **FLAGS[flags])

    def total(tgt, src):
        return O.sfm_loss(tgt, src, d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg, want_grads=False)[0]['total_loss']

    _, G, _ = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg, want_image_grads=True)
    rs = np.random.RandomState(1)
    eps = 1e-6
    mid = total(d['tgt'], d['src'])
    checked = 0
    for which in ('tgt', 'src'):
        arr = d[which]
        ref = G['g' + which]
        idx = [tuple(rs.randint(0, n) for n in arr.shape) for _ in range(40)]
        idx += [np.unravel_index(k, arr.shape) for k in np.argsort(-np.abs(ref).ravel())[:10]]
        for ix in idx:
            vals = []
            for sgn in (1, -1):
                a = arr.copy()
                a[ix] += sgn * eps
                vals.append(total(a, d['src']) if which == 'tgt' else total(d['tgt'], a))
            fd = (vals[0] - vals[1]) / (2 * eps)
            # a kink inside [-eps, eps] shows as a one-sided difference that disagrees with the other side
            if abs((vals[0] - mid) - (mid - vals[1])) > 1e-3 * abs(vals[0] - vals[1]) + 1e-15:
                continue
            # the difference of two totals of order 1 carries ~1e-16 / eps of rounding
            assert abs(fd - ref[ix]) <= 1e-5 * abs(ref[ix]) + 1e-9, (which, ix, fd, ref[ix])
            checked += 1
    assert checked >= 60


def test_resize_adjoint_is_the_transpose():
    rs = np.random.RandomState(0)
    for (H, W), (h, w) in (((32, 64), (16, 32)), ((128, 416), (32, 104)), ((37, 53), (9, 13))):
        x = rs.standard_normal((2, 3, H, W))
        y = rs.standard_normal((2, 3, h, w))
        lhs = np.sum(O.resize_images(x, (h, w)) * y)
        rhs = np.sum(x * O.resize_images_adjoint(y, (H, W), np.float64))
        assert abs(lhs - rhs) <= 1e-12 * (abs(lhs) + np.sum(np.abs(x)) * np.abs(y).max())


# ---- C ABI, without a device ---------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sfm_learner_chainer_b200 import lib as L
    return L


def test_image_grad_symbols_and_struct(lib):
    so = lib.load()
    for name in ('sfm_loss_forward_backward_images', 'sfm_scale_image_grads'):
        assert name in lib.SYMBOLS and getattr(so, name) is not None
    assert C.sizeof(lib.SfmImageGrads) == 16
    assert lib.SFM_FLAG_IMAGE_GRADS == 0x10


@pytest.mark.parametrize('shape', [(4, 2, 128, 416, 4), (3, 3, 64, 200, 3), (2, 1, 32, 64, 1)])
def test_image_grad_flag_adds_the_level_bytes(lib, shape):
    so = lib.load()
    B, S, H, W, ns = shape
    d = lib.SfmDesc(B, S, H, W, ns, 0, 0.1, 0.0, 0.15, 0)
    n0 = so.sfm_workspace_bytes(C.byref(d))
    d.flags = lib.SFM_FLAG_IMAGE_GRADS
    n1 = so.sfm_workspace_bytes(C.byref(d))
    up = lambda n: (n + 255) // 256 * 256
    lv = sum(up(4 * B * 3 * (H >> s) * (W >> s)) + up(4 * B * S * 3 * (H >> s) * (W >> s)) for s in range(1, ns))
    assert n0 > 0 and n1 - n0 == lv


def test_image_grad_argument_errors(lib):
    so = lib.load()
    d = lib.SfmDesc(4, 2, 128, 416, 4, 0, 0.1, 0.0, 0.15, 0)
    inp, g = lib.SfmInputs(), lib.SfmGrads()
    buf = (C.c_float * 4)()
    ig = lib.SfmImageGrads(C.cast(buf, C.c_void_p), None)
    call = lambda desc, igr: so.sfm_loss_forward_backward_images(C.byref(desc), C.byref(inp), C.c_void_p(256), C.byref(g),
                                                                 igr, C.c_void_p(256), None)
    assert call(d, C.byref(ig)) == lib.SFM_E_INVALID_DESC                          # flag missing
    assert b'SFM_FLAG_IMAGE_GRADS' in so.sfm_last_error()
    d.flags = lib.SFM_FLAG_IMAGE_GRADS | lib.SFM_FLAG_EDGE_AWARE_SMOOTH
    assert call(d, C.byref(ig)) == lib.SFM_E_UNSUPPORTED                           # edge-aware smoothness
    d.flags = lib.SFM_FLAG_IMAGE_GRADS
    assert call(d, C.byref(lib.SfmImageGrads(None, None))) == lib.SFM_E_NULL_POINTER   # both NULL
    assert call(d, None) == lib.SFM_E_NULL_POINTER
    assert so.sfm_scale_image_grads(C.byref(d), None, C.byref(ig), None) == lib.SFM_E_NULL_POINTER
    assert so.sfm_scale_image_grads(C.byref(d), C.c_void_p(256), C.byref(lib.SfmImageGrads(None, None)), None) == lib.SFM_E_NULL_POINTER
