"""Reference of the full-resolution multi-scale loss (SFM_FLAG_FULL_RES_MULTISCALE), composed from the existing references.

U_s upsamples d_s to (H, W) in the arithmetic of torch's F.interpolate(mode='bilinear', align_corners=False) in the
inputs' dtype.  The photometric terms of scale s are those of a one-scale call of tests/pixel_oracle.sfm_loss_pixel (or
tests/min_reprojection_oracle.sfm_loss_min_reprojection) with intrinsics[:, :1], disps=[U_s(d_s)] and smooth_reg=0; the
smoothness terms come from one call at the native scales with zero photometric weights.  The loss is linear in the
scales' terms, so the losses, gposes and the intrinsics gradients are sums, and gdisp[s] is U_s^T of the one-scale
gradient plus the smoothness gradient."""
import numpy as np

from oracle import sfm_oracle as O
from tests import min_reprojection_oracle as MR
from tests.pixel_oracle import sfm_loss_pixel


def up_axis(n, n_out, dtype):
    """One axis of U for n -> n_out points: (i0, i1, l0, l1) arrays of n_out entries, in `dtype` arithmetic."""
    t = np.dtype(dtype).type
    scale = t(n) / t(n_out)
    src = np.maximum((np.arange(n_out).astype(dtype) + t(0.5)) * scale - t(0.5), t(0))
    i0 = src.astype(np.int64)                            # src >= 0: truncation is the floor
    i1 = i0 + (i0 < n - 1)
    l1 = src - i0.astype(dtype)
    return i0, i1, t(1) - l1, l1


def upsample(d, H, W):
    """U(d): (N,1,h,w) -> (N,1,H,W) as F.interpolate(d, size=(H, W), mode='bilinear', align_corners=False) computes it:
    ly0 * (lx0 * d00 + lx1 * d01) + ly1 * (lx0 * d10 + lx1 * d11), every operation rounded to d's dtype."""
    h, w = d.shape[2:]
    y0, y1, ly0, ly1 = up_axis(h, H, d.dtype)
    x0, x1, lx0, lx1 = up_axis(w, W, d.dtype)
    r0, r1 = d[:, :, y0], d[:, :, y1]
    top = lx0 * r0[..., x0] + lx1 * r0[..., x1]
    bot = lx0 * r1[..., x0] + lx1 * r1[..., x1]
    return ly0[:, None] * top + ly1[:, None] * bot


def up_matrix(n, n_out, dtype):
    """(n_out, n) float64 matrix of one axis of U with the weights of `dtype` arithmetic: U(d) = Ay d Ax^T."""
    i0, i1, l0, l1 = up_axis(n, n_out, dtype)
    A = np.zeros((n_out, n))
    np.add.at(A, (np.arange(n_out), i0), l0.astype(np.float64))
    np.add.at(A, (np.arange(n_out), i1), l1.astype(np.float64))
    return A


def upsample_adjoint(g, h, w, dtype=np.float32):
    """U^T: (N,1,H,W) -> (N,1,h,w) float64, for the U of a (h, w) map in `dtype` arithmetic."""
    H, W = g.shape[2:]
    return np.einsum('Yy,ncYX,Xx->ncyx', up_matrix(h, H, dtype), g.astype(np.float64), up_matrix(w, W, dtype))


def sfm_loss_full_res(tgt, src, intrinsics, disps, poses, cfg, pixel_weights=None, min_reprojection=False, automask=True,
                      selection=None, want_grads=True, want_intrinsics_grad=False, raw_disp_scales=0, raw_pose=False):
    """-> (losses dict with `pixel_losses` (list of (B,S,H,W)) [and `selection` (list of (B,H,W))], grads dict or None).

    pixel_weights: None or a list of n_scales (B,S,H,W) arrays or None entries.  min_reprojection / automask /
    selection: as min_reprojection_oracle.sfm_loss_min_reprojection, per scale at full resolution.  raw_disp_scales /
    raw_pose: inputs as oracle.sfm_loss_raw takes them; the activation is applied at native resolution before U.
    The grads dict holds gdisp (native shapes), gpose and, with want_intrinsics_grad, gintrinsics (B,n_scales,3,3) with the
    whole gradient at [:, 0]."""
    dt = tgt.dtype
    B, S, _, H, W = src.shape
    ns = cfg.n_scales
    dd, dacts = [], []
    for s, d in enumerate(disps):
        a, da = O.disp_activation(d) if (raw_disp_scales >> s) & 1 else (d, None)
        dd.append(a)
        dacts.append(da)
    pp = O.pose_from_raw(poses, S) if raw_pose else poses
    cfg1 = O.LossConfig(ssim_rate=cfg.ssim_rate, n_scales=1, B_global=cfg.B_global)
    K0 = np.ascontiguousarray(intrinsics[:, :1])
    kw = dict(want_grads=want_grads, want_intrinsics_grad=want_intrinsics_grad)
    pixel = ssim = 0.0
    maps, sels = [], []
    gdisp = [np.zeros(d.shape) for d in disps]
    gpose = np.zeros((B, S, 6))
    gK = np.zeros((B, ns, 3, 3))
    for s in range(ns):
        u = dd[0] if s == 0 else upsample(dd[s], H, W)
        if min_reprojection:
            L, G = MR.sfm_loss_min_reprojection(tgt, src, K0, [u], pp, cfg1, automask=automask,
                                                selection=None if selection is None else [selection[s]], **kw)
            sels.append(L['selection'][0])
        else:
            w = None if pixel_weights is None else [pixel_weights[s]]
            L, G = sfm_loss_pixel(tgt, src, K0, [u], pp, None, cfg1, pixel_weights=w, **kw)
        pixel += L['pixel_loss']
        ssim += L['ssim_loss']
        maps.append(L['pixel_losses'][0])
        if want_grads:
            g = G['gdisp'][0].astype(np.float64)
            gdisp[s] += g if s == 0 else upsample_adjoint(g, *disps[s].shape[2:], dtype=dt)
            gpose += G['gpose']
            if want_intrinsics_grad:
                gK[:, 0] += G['gintrinsics'][:, 0]
    smooth = 0.0
    if cfg.smooth_reg:
        zeros = [np.zeros((B, S) + d.shape[2:], dt) for d in disps]
        cfg_s = O.LossConfig(smooth_reg=cfg.smooth_reg, ssim_rate=cfg.ssim_rate, n_scales=ns, B_global=cfg.B_global,
                             edge_aware_smooth=cfg.edge_aware_smooth)
        L, G = sfm_loss_pixel(tgt, src, intrinsics, dd, pp, None, cfg_s, pixel_weights=zeros, want_grads=want_grads)
        smooth = L['smooth_loss']
        if want_grads:
            for s in range(ns):
                gdisp[s] += G['gdisp'][s]
    r = cfg.ssim_rate if cfg.ssim_rate else 0.0
    losses = dict(total_loss=(1 - r) * pixel + r * ssim + smooth, pixel_loss=pixel, smooth_loss=smooth, exp_loss=0.0,
                  ssim_loss=ssim, pixel_losses=maps)
    if min_reprojection:
        losses['selection'] = sels
    if not want_grads:
        return losses, None
    gdisp = [(g if da is None else g * da.astype(np.float64)).astype(dt) for g, da in zip(gdisp, dacts)]
    if raw_pose:
        n = int(np.prod(poses.shape[2:]))
        gp = gpose.reshape(B, 6 * S, *([1] * (poses.ndim - 2)))
        gpose = np.broadcast_to(gp * (0.01 / n), poses.shape)
    grads = dict(gdisp=gdisp, gpose=gpose.astype(dt))
    if want_intrinsics_grad:
        grads['gintrinsics'] = gK
    return losses, grads
