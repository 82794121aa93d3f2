"""-m "not gpu": gradient of the fused loss w.r.t. the camera intrinsics (d total / d intrinsics).

The oracle's gintrinsics (tests/intrinsics_grad_oracle.py) is checked against torch fp64 autograd through an independent
restatement of the whole K-dependent path (K a leaf through torch.linalg.inv and K @ [R|t], the grid with the x2 rule,
grid_sample, the L1 / explainability / SSIM terms), against central differences of the numpy oracle, and on the poses
where the formula has a closed form.  The C ABI additions are checked for their argument errors without a device."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets
from tests import intrinsics_grad_oracle as KO

FLAGS = {
    'l1': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.0),
    'exp': dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0),
    'ssim': dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
}


def _data(B, S, H, W, ns, harsh, seed=0):
    return make_snippets(B, S, H, W, seed=seed, n_scales=ns, harsh=harsh, dtype=np.float64)


def _rot(a):
    """(Rx . Ry) . Rz of the clipped angles a (N,3) (transform.py:11-40)."""
    a = torch.clamp(a, -np.pi, np.pi)
    c, s = torch.cos(a), torch.sin(a)
    o, z = torch.ones_like(c[:, 0]), torch.zeros_like(c[:, 0])
    rx = torch.stack([o, z, z, z, c[:, 0], -s[:, 0], z, s[:, 0], c[:, 0]], 1).reshape(-1, 3, 3)
    ry = torch.stack([c[:, 1], z, s[:, 1], z, o, z, -s[:, 1], z, c[:, 1]], 1).reshape(-1, 3, 3)
    rz = torch.stack([c[:, 2], -s[:, 2], z, s[:, 2], c[:, 2], z, z, z, o], 1).reshape(-1, 3, 3)
    return (rx @ ry) @ rz


def _torch_total(d, cfg, K):
    """(1 - r) * pixel + r * ssim of base_model.py:64-118 with the intrinsics K (B,ns,3,3) as a torch leaf; the terms
    that do not depend on K (smoothness, explainability regulariser) are left out."""
    B, S, _, H, W = d['src'].shape
    use_exp = bool(cfg.exp_reg)
    use_ssim = not use_exp and bool(cfg.ssim_rate)
    rate = cfg.ssim_rate or 0.0
    pixel = ssim = 0.0
    for ns in range(cfg.n_scales):
        h, w = H >> ns, W >> ns
        ct = torch.from_numpy(O.resize_images(d['tgt'], (h, w)))
        cs = torch.from_numpy(O.resize_images(d['src'].reshape(B, 3 * S, H, W), (h, w)))
        depth = 1.0 / torch.from_numpy(d['disps'][ns]).reshape(B, 1, h * w)
        ys, xs = torch.meshgrid(torch.arange(h, dtype=K.dtype), torch.arange(w, dtype=K.dtype), indexing='ij')
        pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(h * w, dtype=K.dtype)])
        Ks = K[:, ns]
        cam = depth * (torch.linalg.inv(Ks) @ pix)                                   # pixel2cam (transform.py:94-109)
        n3 = B * 3 * h * w
        for i in range(S):
            pose = torch.from_numpy(d['poses'][:, i])
            P = Ks @ torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)           # K4 . [R|t] (transform.py:86-88)
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((w - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((h - 1) / 2.) - 1
            inx = ((xn > -1) & (xn < 1)).detach()
            iny = ((yn > -1) & (yn < 1)).detach()
            xn = torch.where(inx, xn, 2 * xn)
            yn = torch.where(iny, yn, 2 * yn)
            grid = torch.stack([xn, yn], -1).reshape(B, h, w, 2)
            Pw = F.grid_sample(cs[:, 3 * i:3 * i + 3], grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            m = (Pw == 0).all(dim=1, keepdim=True).detach()
            err = torch.where(m, torch.zeros_like(Pw), (Pw - ct).abs())
            if use_exp:
                sg = torch.sigmoid(torch.from_numpy(d['logits'][ns][:, i:i + 1]))
                pixel = pixel + (err * sg).sum() / n3
            else:
                pixel = pixel + err.sum() / n3
            if use_ssim:
                pool = lambda x: F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)
                a, my = pool(Pw), pool(ct)
                sx, sy, sxy = pool(Pw * Pw) - a * a, pool(ct * ct) - my * my, pool(Pw * ct) - a * my
                n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
                dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
                e = torch.clamp((1 - n / dd) / 2, 0, 1) * (~m)
                ssim = ssim + e.sum() / n3
    return (1 - rate) * pixel + rate * ssim


@pytest.mark.parametrize('flags', sorted(FLAGS))
@pytest.mark.parametrize('S', [1, 2, 4])
@pytest.mark.parametrize('ns', [1, 4])
@pytest.mark.parametrize('harsh', [False, True])
def test_oracle_intrinsics_grad_matches_torch_autograd(flags, S, ns, harsh):
    d = _data(2, S, 32, 64, ns, harsh, seed=S + 10 * ns + 100 * harsh)
    cfg = O.LossConfig(n_scales=ns, **FLAGS[flags])
    L, G, _ = KO.sfm_loss_with_intrinsics_grad(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg)
    K = torch.from_numpy(d['intrinsics']).requires_grad_(True)
    tot = _torch_total(d, cfg, K)
    tot.backward()
    # the restatement leaves out only K-independent terms
    np.testing.assert_allclose(tot.item(), L['total_loss'] - L['smooth_loss'] - L['exp_loss'], rtol=1e-9, atol=1e-12)
    ref = K.grad.numpy()
    got = G['gintrinsics']
    assert got.dtype == np.float64 and got.shape == (2, ns, 3, 3)
    np.testing.assert_allclose(got, ref, rtol=1e-6, atol=1e-9 * np.abs(ref).max())
    assert np.abs(ref).max() > 0


@pytest.mark.parametrize('flags', sorted(FLAGS))
def test_oracle_intrinsics_grad_central_differences(flags):
    """fp64 central differences of the reported total on every entry of K, the step scaled per entry.  Floor flips
    of the sampling coordinates and the x2 rule's boundary move with K: a kink or jump inside [-eps, eps] shows as a
    one-sided difference that disagrees with the other side, and that entry is skipped."""
    d = _data(2, 2, 32, 64, 4, True, seed=7)
    cfg = O.LossConfig(n_scales=4, **FLAGS[flags])

    def total(K):
        return O.sfm_loss(d['tgt'], d['src'], K, d['disps'], d['poses'], d['logits'], cfg, want_grads=False)[0]['total_loss']

    _, G, _ = KO.sfm_loss_with_intrinsics_grad(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg)
    ref = G['gintrinsics']
    mid = total(d['intrinsics'])
    checked = 0
    for ix in np.ndindex(*ref.shape):
        eps = 1e-7 * max(1.0, abs(d['intrinsics'][ix]))
        vals = []
        for sgn in (1, -1):
            K = d['intrinsics'].copy()
            K[ix] += sgn * eps
            vals.append(total(K))
        if abs((vals[0] - mid) - (mid - vals[1])) > 1e-3 * abs(vals[0] - vals[1]) + 1e-15:
            continue
        fd = (vals[0] - vals[1]) / (2 * eps)
        # the difference of two totals of order 1 carries ~1e-16 / eps of rounding
        assert abs(fd - ref[ix]) <= 1e-5 * abs(ref[ix]) + 2e-16 / eps, (ix, fd, ref[ix])
        checked += 1
    assert checked >= 60


def test_zero_rotation_closed_forms():
    """R = I, t = 0: the loss does not depend on K and the formula is A - A; R = I, t != 0: exactly sum_i g_i t_i^T."""
    d = _data(2, 3, 32, 64, 4, False, seed=21)
    cfg = O.LossConfig(n_scales=4, **FLAGS['ssim'])
    for t in (np.zeros(3), np.array([0.02, -0.01, 0.03])):
        poses = np.zeros_like(d['poses'])
        poses[..., 3:] = t
        _, G, _ = KO.sfm_loss_with_intrinsics_grad(d['tgt'], d['src'], d['intrinsics'], d['disps'], poses, d['logits'], cfg)
        A = G['dP'][..., :3]
        closed = np.einsum('bisk,j->bskj', G['dP'][..., 3], t)
        np.testing.assert_allclose(G['gintrinsics'], closed, rtol=0, atol=1e-12 * np.abs(A).max())
        if t.any():
            assert np.abs(closed).max() > 1e3 * 1e-12 * np.abs(A).max()


def test_raw_counterpart_uses_the_reduced_poses():
    from sfm_learner_chainer_b200.synthetic import make_raw_seam
    d = _data(2, 2, 32, 64, 4, True, seed=31)
    raw_disps, raw_poses = make_raw_seam(d, (1, 4), seed=32)
    cfg = O.LossConfig(n_scales=4, **FLAGS['l1'])
    L, G, dbg = KO.sfm_loss_raw_with_intrinsics_grad(d['tgt'], d['src'], d['intrinsics'], raw_disps, raw_poses, d['logits'],
                                                     cfg, raw_disp_scales=0xF, raw_pose=True)
    L2, G2, _ = KO.sfm_loss_with_intrinsics_grad(d['tgt'], d['src'], d['intrinsics'], dbg['disps'], dbg['poses'], d['logits'], cfg)
    assert L == L2
    np.testing.assert_array_equal(G['gintrinsics'], G2['gintrinsics'])


# ---- C ABI, without a device ---------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as ge
    ge.build()
    from sfm_learner_chainer_b200 import lib as L
    return L


def test_intrinsics_grad_symbols(lib):
    so = lib.load()
    for name in ('sfm_intrinsics_grad', 'sfm_scale_intrinsics_grad'):
        assert name in lib.SYMBOLS and getattr(so, name) is not None


def test_intrinsics_grad_argument_errors(lib):
    so = lib.load()
    d = lib.SfmDesc(4, 2, 128, 416, 4, 0, 0.1, 0.0, 0.15, 0)
    buf = (C.c_float * 16)()
    inp = lib.SfmInputs()
    inp.intrinsics, inp.poses = C.cast(buf, C.c_void_p), C.cast(buf, C.c_void_p)
    ws, gk = C.c_void_p(256), C.cast(buf, C.c_void_p)
    call = lambda desc, i, w, g: so.sfm_intrinsics_grad(C.byref(desc), i, w, g, None)
    assert call(d, None, ws, gk) == lib.SFM_E_NULL_POINTER
    assert call(d, C.byref(lib.SfmInputs()), ws, gk) == lib.SFM_E_NULL_POINTER     # no intrinsics / poses
    assert call(d, C.byref(inp), None, gk) == lib.SFM_E_NULL_POINTER
    assert call(d, C.byref(inp), ws, None) == lib.SFM_E_NULL_POINTER
    assert call(d, C.byref(inp), C.c_void_p(16), gk) == lib.SFM_E_INVALID_DESC    # misaligned workspace
    assert so.sfm_intrinsics_grad(None, C.byref(inp), ws, gk, None) == lib.SFM_E_NULL_POINTER
    bad = lib.SfmDesc(0, 2, 128, 416, 4, 0, 0.1, 0.0, 0.15, 0)
    assert call(bad, C.byref(inp), ws, gk) == lib.SFM_E_INVALID_DESC
    d.flags = lib.SFM_FLAG_TABLES_PROVIDED
    assert call(d, C.byref(inp), ws, gk) == lib.SFM_E_UNSUPPORTED
    assert b'SFM_FLAG_TABLES_PROVIDED' in so.sfm_last_error()
    d.flags = 0
    assert so.sfm_scale_intrinsics_grad(C.byref(d), None, gk, None) == lib.SFM_E_NULL_POINTER
    assert so.sfm_scale_intrinsics_grad(C.byref(d), C.c_void_p(256), None, None) == lib.SFM_E_NULL_POINTER
    assert so.sfm_scale_intrinsics_grad(C.byref(bad), C.c_void_p(256), gk, None) == lib.SFM_E_INVALID_DESC


def test_operator_refuses_caller_tables(lib):
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    op = ViewSynthesisLoss(0.1, 0.0, 0.15, intrinsics_grad=True)
    d = _data(1, 2, 32, 64, 4, False)
    args = (d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'])
    with pytest.raises(ValueError):
        op.forward_backward(*args, proj=np.zeros(1), kinv=np.zeros(1))
    with pytest.raises(ValueError):
        op.backward(*args, proj=np.zeros(1), kinv=np.zeros(1))
