"""-m "not gpu": image gradients of the fused loss (d total / d tgt_img, d total / d src_imgs).

The oracle's analytic gtgt / gsrc (tests/image_grad_oracle.py) are checked against torch fp64 autograd through an independent restatement of the
image-dependent part of the forward (the projection grid does not depend on the images and is taken from the oracle),
against central differences of the oracle itself, and the resize adjoint against <Rx, y> = <x, R^T y>.  The C ABI
additions are checked for their argument errors without a device."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import image_grad_oracle as IO

FLAGS = {
    'l1': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.0),
    'exp': dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
}


def _data(B, S, H, W, ns, harsh, seed=0):
    d = make_snippets(B, S, H, W, seed=seed, n_scales=ns, harsh=harsh, dtype=np.float64)
    return d


def _torch_total(d, cfg, tgt, src):
    """(1 - r) * pixel + r * ssim of base_model.py:64-118 with the images as torch leaves; the terms that do not
    depend on the images (smoothness, explainability regulariser) are left out."""
    B, S, _, H, W = d['src'].shape
    Bg = B
    use_exp = bool(cfg.exp_reg)
    use_ssim = not use_exp and bool(cfg.ssim_rate)
    rate = cfg.ssim_rate or 0.0
    pixel = ssim = 0.0
    for ns in range(cfg.n_scales):
        h, w = H >> ns, W >> ns
        if ns == 0:
            ct, cs = tgt, src.reshape(B, 3 * S, H, W)
        else:
            ct = F.interpolate(tgt, size=(h, w), mode='bilinear', align_corners=True)
            cs = F.interpolate(src.reshape(B, 3 * S, H, W), size=(h, w), mode='bilinear', align_corners=True)
        depth = 1.0 / d['disps'][ns].reshape(B, h * w)
        K = d['intrinsics'][:, ns]
        _, cam = O.pixel2cam(depth, O.batch_inv3(K), h, w)
        n3 = Bg * 3 * h * w
        for i in range(S):
            gr = O.cam2pixel(cam, O.proj_tgt_to_src(d['poses'][:, i], K), h, w)
            grid = torch.from_numpy(np.stack([gr['xn'], gr['yn']], -1).reshape(B, h, w, 2))
            P = F.grid_sample(cs[:, 3 * i:3 * i + 3], grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            m = (P == 0).all(dim=1, keepdim=True).detach()
            err = torch.where(m, torch.zeros_like(P), (P - ct).abs())
            if use_exp:
                sg = torch.sigmoid(torch.from_numpy(d['logits'][ns][:, i:i + 1]))
                pixel = pixel + (err * sg).sum() / n3
            else:
                pixel = pixel + err.sum() / n3
            if use_ssim:
                pool = lambda x: F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)
                a, my = pool(P), pool(ct)
                sx, sy, sxy = pool(P * P) - a * a, pool(ct * ct) - my * my, pool(P * ct) - a * my
                n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
                dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
                e = torch.clamp((1 - n / dd) / 2, 0, 1) * (~m)
                ssim = ssim + e.sum() / n3
    return (1 - rate) * pixel + rate * ssim


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 2, 4])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_oracle_image_grads_match_torch_autograd(flags, S, ns, harsh):
    d = _data(2, S, 32, 64, ns, harsh, seed=S + 10 * ns)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L, G, _ = IO.sfm_loss_with_image_grads(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg)
    tgt = torch.from_numpy(d['tgt']).requires_grad_(True)
    src = torch.from_numpy(d['src']).requires_grad_(True)
    tot = _torch_total(d, cfg, tgt, src)
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

    _, G, _ = IO.sfm_loss_with_image_grads(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg)
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
        rhs = np.sum(x * IO.resize_images_adjoint(y, (H, W), np.float64))
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
