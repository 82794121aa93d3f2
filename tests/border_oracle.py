"""Reference of Monodepth2's image borders (SFM_FLAG_BORDER_PADDING, include/sfmloss.h), in numpy on the oracle's helpers.

The photometric loop of tests/pixel_oracle.sfm_loss_pixel restated with the border-clamped sampler and its gradient (no
x2 rule), no mask except degenerate projections, and reflection-padded SSIM windows with their adjoint; per-pixel
weights and maps as there.  The smoothness term (unchanged by the flag) comes from tests/pixel_oracle.sfm_loss_pixel
with zero photometric weights.  loss_min_reprojection and loss_full_res compose it as the min-reprojection and
full-resolution references compose the weighted one.  No explainability branch, image gradients or debug dumps."""
import numpy as np

from oracle import sfm_oracle as O
from tests import min_reprojection_oracle as MR
from tests.full_res_oracle import upsample, upsample_adjoint
from tests.pixel_oracle import sfm_loss_pixel


def border_sampler(img, gr, h, w):
    """Monodepth2's grid_sample(padding_mode="border", align_corners=True) on the grid of O.cam2pixel without its x2 rule,
    in the image dtype with the sampler's association.  -> (P (N,C,hw), tap record, degenerate (N,hw) bool)."""
    dt = img.dtype
    N = img.shape[0]
    q, z = gr['q'], gr['z']
    with np.errstate(all='ignore'):
        xn = (q[:, 0] / z) / gr['hw'] - dt.type(1)
        yn = (q[:, 1] / z) / gr['hh'] - dt.type(1)
        az = np.abs(z)
        ok = (az >= dt.type(2.0 ** -58)) & (az <= dt.type(2.0 ** 126)) & np.isfinite(xn) & np.isfinite(yn)
        uc = np.where(ok, ((xn + dt.type(1)) * dt.type(w - 1)) / dt.type(2), dt.type(0))
        vc = np.where(ok, ((yn + dt.type(1)) * dt.type(h - 1)) / dt.type(2), dt.type(0))
    u = np.clip(uc, 0, w - 1).astype(dt)
    v = np.clip(vc, 0, h - 1).astype(dt)
    u0f = np.minimum(np.floor(u), w - 2).astype(dt)
    v0f = np.minimum(np.floor(v), h - 2).astype(dt)
    wa, wb = (u0f + dt.type(1)) - u, u - u0f
    wc, wd = (v0f + dt.type(1)) - v, v - v0f
    u0, v0 = u0f.astype(np.int64), v0f.astype(np.int64)
    bi = np.arange(N)[:, None]

    def tap(vi, ui):
        return img[bi, :, vi, ui].transpose(0, 2, 1)

    t = dict(wa=wa, wb=wb, wc=wc, wd=wd, I00=tap(v0, u0), I01=tap(v0, u0 + 1), I10=tap(v0 + 1, u0),
             I11=tap(v0 + 1, u0 + 1), ok=ok, gate_u=ok & (uc > 0) & (uc < w - 1), gate_v=ok & (vc > 0) & (vc < h - 1))
    w1, w2 = (wa * wc)[:, None], (wb * wc)[:, None]
    w3, w4 = (wa * wd)[:, None], (wb * wd)[:, None]
    P = ((w1 * t['I00'] + w2 * t['I01']) + w3 * t['I10']) + w4 * t['I11']
    return np.where(ok[:, None], P, dt.type(0)), t, ~ok


def border_sampler_grad(t, gy, h, w):
    """d/d(xn, yn) of border_sampler (float64 record): the bilinear derivative times (w-1)/2 where the unclamped
    coordinate lies strictly inside (0, w-1), else 0 (torch's clip_coordinates_set_grad)."""
    du = t['wc'][:, None] * (t['I01'] - t['I00']) + t['wd'][:, None] * (t['I11'] - t['I10'])
    dv = t['wa'][:, None] * (t['I10'] - t['I00']) + t['wb'][:, None] * (t['I11'] - t['I01'])
    gu = np.where(t['gate_u'], np.sum(gy * du, axis=1), 0.0)
    gv = np.where(t['gate_v'], np.sum(gy * dv, axis=1), 0.0)
    return gu * ((w - 1) / 2.), gv * ((h - 1) / 2.)


def avg_pool3_reflect(x):
    """nn.ReflectionPad2d(1) + nn.AvgPool2d(3, 1): the running sum of O.avg_pool3 over the reflected image, then /9."""
    h, w = x.shape[-2:]
    xp = np.pad(x, [(0, 0)] * (x.ndim - 2) + [(1, 1), (1, 1)], mode='reflect')
    acc = None
    for dy in range(3):
        for dx in range(3):
            t = xp[..., dy:dy + h, dx:dx + w]
            acc = t if acc is None else acc + t
    return acc / x.dtype.type(9)


def avg_pool3_reflect_adjoint(g):
    """Adjoint of avg_pool3_reflect (float64): every window spreads g/9 over its padded 3x3 taps, then padded row /
    column -1 folds onto 1 and h / w onto h-2 / w-2."""
    h, w = g.shape[-2:]
    G = np.zeros(g.shape[:-2] + (h + 2, w + 2), np.float64)
    for dy in range(3):
        for dx in range(3):
            G[..., dy:dy + h, dx:dx + w] += g
    G[..., 2, :] += G[..., 0, :]
    G[..., h - 1, :] += G[..., h + 1, :]
    G[..., :, 2] += G[..., :, 0]
    G[..., :, w - 1] += G[..., :, w + 1]
    return G[..., 1:h + 1, 1:w + 1] / 9.0


def ssim_terms_reflect(P, T):
    """O.ssim_terms on the reflected windows of avg_pool3_reflect."""
    dt = P.dtype
    c1, c2 = dt.type(O.SSIM_C1), dt.type(O.SSIM_C2)
    a = avg_pool3_reflect(P)
    my = avg_pool3_reflect(T)
    sx = avg_pool3_reflect(P * P) - a * a
    sy = avg_pool3_reflect(T * T) - my * my
    sxy = avg_pool3_reflect(P * T) - a * my
    n1 = dt.type(2) * a * my + c1
    n2 = dt.type(2) * sxy + c2
    d1 = a * a + my * my + c1
    d2 = sx + sy + c2
    n = n1 * n2
    d = d1 * d2
    raw = (dt.type(1) - n / d) / dt.type(2)
    return dict(a=a, my=my, n1=n1, n2=n2, d1=d1, d2=d2, n=n, d=d, raw=raw)


def _smoothness(tgt, src, intrinsics, disps, poses, cfg, want_grads):
    """(smooth loss, list of smoothness gdisp or None) of the reference, through zero photometric weights."""
    if not cfg.smooth_reg:
        return 0.0, None
    B, S = src.shape[:2]
    zeros = [np.zeros((B, S) + d.shape[2:], tgt.dtype) for d in disps]
    cfg_s = O.LossConfig(smooth_reg=cfg.smooth_reg, ssim_rate=cfg.ssim_rate, n_scales=cfg.n_scales, B_global=cfg.B_global,
                         edge_aware_smooth=cfg.edge_aware_smooth)
    L, G = sfm_loss_pixel(tgt, src, intrinsics, disps, poses, None, cfg_s, pixel_weights=zeros, want_grads=want_grads)
    return L['smooth_loss'], (G['gdisp'] if want_grads else None)


def loss_pixel(tgt, src, intrinsics, disps, poses, cfg, pixel_weights=None, want_grads=True, want_intrinsics_grad=False):
    """-> (losses dict with `pixel_losses`, a list of (B,S,h_s,w_s) float64 maps, grads dict or None): the loss of
    tests/pixel_oracle.sfm_loss_pixel (no explainability branch) under SFM_FLAG_BORDER_PADDING."""
    if cfg.exp_reg:
        raise ValueError('border padding: no explainability branch')
    dt = tgt.dtype
    B, S, _, H, W = src.shape
    Bg = cfg.B_global if cfg.B_global else B
    stacked = src.reshape(B, 3 * S, H, W)
    use_ssim = bool(cfg.ssim_rate)
    r = cfg.ssim_rate if cfg.ssim_rate else 0.0
    pixel_loss = ssim_loss = 0.0
    gdisp = [np.zeros(d.shape, np.float64) for d in disps]
    dP_all = [[None] * cfg.n_scales for _ in range(S)]
    maps = []
    for ns in range(cfg.n_scales):
        h, w = O.scale_shape(H, W, ns)
        hw_n = h * w
        cur_tgt = O.resize_images(tgt, (h, w))
        cur_src = O.resize_images(stacked, (h, w))
        maps.append(np.zeros((B, S, h, w), np.float64))
        disp_flat = disps[ns].reshape(B, hw_n)
        depth = dt.type(1) / disp_flat
        K = intrinsics[:, ns]
        ray, cam = O.pixel2cam(depth, O.batch_inv3(K), h, w)
        g_depth = np.zeros((B, hw_n), np.float64)
        for i in range(S):
            img = cur_src[:, 3 * i:3 * i + 3]
            proj = O.proj_tgt_to_src(poses[:, i], K)
            gr = O.cam2pixel(cam, proj, h, w)
            Pf, t, deg = border_sampler(img, gr, h, w)
            P = Pf.reshape(B, 3, h, w)
            diff = P - cur_tgt
            m = deg.reshape(B, 1, h, w)
            err = np.where(m, dt.type(0), np.abs(diff))
            n_pix3 = Bg * 3 * h * w
            sgn = np.where(m, 0.0, np.sign(diff)).astype(np.float64)
            Mw = None
            if pixel_weights is not None and pixel_weights[ns] is not None:
                Mw = pixel_weights[ns][:, i:i + 1]
            M64 = 1.0 if Mw is None else Mw.astype(np.float64)
            e_sum = np.sum(err.astype(np.float64), axis=1, keepdims=True)
            maps[ns][:, i] += (e_sum * ((1 - r) / n_pix3))[:, 0]
            pixel_loss += O._fsum(err if Mw is None else err * Mw) / n_pix3
            gP = sgn * M64 * ((1 - r) / n_pix3)
            if use_ssim:
                st = ssim_terms_reflect(P, cur_tgt)
                e = np.clip(st['raw'], 0, 1) * (1 - m)
                maps[ns][:, i] += np.sum(e.astype(np.float64), axis=1) * (r / n_pix3)
                ssim_loss += O._fsum(e if Mw is None else e * Mw) / n_pix3
                raw = st['raw'].astype(np.float64)
                a, my = st['a'].astype(np.float64), st['my'].astype(np.float64)
                n1, n2 = st['n1'].astype(np.float64), st['n2'].astype(np.float64)
                d1, d2 = st['d1'].astype(np.float64), st['d2'].astype(np.float64)
                n, d = st['n'].astype(np.float64), st['d'].astype(np.float64)
                g_e = (r / n_pix3) * (1 - m) * ((raw >= 0) & (raw <= 1)) * M64
                g_n = -g_e / (2 * d)
                g_d = g_e * n / (2 * d * d)
                g_a = g_n * (2 * my * n2 - 2 * my * n1) + g_d * (2 * a * d2 - 2 * a * d1)
                g_s = g_d * d1
                g_c = 2 * g_n * n1
                Pd, Td = P.astype(np.float64), cur_tgt.astype(np.float64)
                adj = avg_pool3_reflect_adjoint
                gP = gP + adj(g_a) + 2 * Pd * adj(g_s) + Td * adj(g_c)
            if want_grads:                                           # sampler -> grid -> q -> cam / proj
                t64 = {k: (v.astype(np.float64) if v.dtype.kind == 'f' else v) for k, v in t.items()}
                g_xn, g_yn = border_sampler_grad(t64, gP.reshape(B, 3, hw_n), h, w)
                q = gr['q'].astype(np.float64)
                z = gr['z'].astype(np.float64)
                hw_, hh_ = float(gr['hw']), float(gr['hh'])
                with np.errstate(divide='ignore', invalid='ignore'):
                    g_q = np.stack([g_xn / (z * hw_), g_yn / (z * hh_),
                                    -(g_xn * q[:, 0] / hw_ + g_yn * q[:, 1] / hh_) / (z * z)], axis=1)
                g_q = np.where(t['ok'][:, None], g_q, 0.0)
                g_cam = np.einsum('nkp,nkj->njp', g_q, proj.astype(np.float64)[:, :3, :3])
                g_depth += np.sum(g_cam * ray.astype(np.float64), axis=1)
                cam4 = np.concatenate([cam.astype(np.float64), np.ones((B, 1, hw_n))], axis=1)
                dP_all[i][ns] = np.einsum('nkp,njp->nkj', g_q, cam4)
        if want_grads:
            d64 = disp_flat.astype(np.float64)
            gdisp[ns] += (-g_depth / (d64 * d64)).reshape(disps[ns].shape)
    smooth_loss, gsm = _smoothness(tgt, src, intrinsics, disps, poses, cfg, want_grads)
    total = (1 - r) * pixel_loss + r * ssim_loss + smooth_loss
    losses = dict(total_loss=total, pixel_loss=pixel_loss, smooth_loss=smooth_loss, exp_loss=0.0, ssim_loss=ssim_loss,
                  pixel_losses=maps)
    if not want_grads:
        return losses, None
    if gsm is not None:
        gdisp = [g + s.astype(np.float64) for g, s in zip(gdisp, gsm)]
    gpose = np.zeros((B, S, 6), dt)
    K_scales = [intrinsics[:, ns] for ns in range(cfg.n_scales)]
    for i in range(S):
        gpose[:, i] = O._pose_backward(poses[:, i], K_scales, dP_all[i])[0]
    grads = dict(gdisp=[g.astype(dt) for g in gdisp], gpose=gpose)
    if want_intrinsics_grad:
        dP = np.stack([np.stack(dP_all[i], 1) for i in range(S)], 1)
        grads.update(dP=dP, gintrinsics=O.intrinsics_grad(intrinsics, poses, dP))
    return losses, grads


def loss_pixel_raw(tgt, src, intrinsics, disps_in, poses_in, cfg, raw_disp_scales=0, raw_pose=False, **kw):
    """loss_pixel with the seam included, as tests/pixel_oracle.sfm_loss_pixel_raw."""
    S = src.shape[1]
    disps, dacts = [], []
    for s, d in enumerate(disps_in):
        dd, da = O.disp_activation(d) if (raw_disp_scales >> s) & 1 else (d, None)
        disps.append(dd)
        dacts.append(da)
    poses = O.pose_from_raw(poses_in, S) if raw_pose else poses_in
    losses, grads = loss_pixel(tgt, src, intrinsics, disps, poses, cfg, **kw)
    if grads is not None:
        grads = dict(grads)
        grads['gdisp'] = [g if da is None else (g.astype(np.float64) * da).astype(g.dtype) for g, da in zip(grads['gdisp'], dacts)]
        if raw_pose:
            n = int(np.prod(poses_in.shape[2:]))
            gp = grads['gpose'].astype(np.float64).reshape(poses_in.shape[0], 6 * S, *([1] * (poses_in.ndim - 2)))
            grads['gpose'] = np.broadcast_to(gp * (0.01 / n), poses_in.shape).astype(poses_in.dtype)
    return losses, grads


def errors(tgt, src, intrinsics, disps, poses, cfg):
    """tests/min_reprojection_oracle.errors under the flag: (e, masked, e_id) per scale, with the border sampler, its
    degenerate mask and the reflected SSIM windows for both errors."""
    B, S, _, H, W = src.shape
    use_ssim = not cfg.exp_reg and bool(cfg.ssim_rate)
    r = cfg.ssim_rate if cfg.ssim_rate else 0.0
    stacked = src.reshape(B, 3 * S, H, W)
    out_e, out_m, out_id = [], [], []
    for ns in range(cfg.n_scales):
        h, w = O.scale_shape(H, W, ns)
        cur_tgt = O.resize_images(tgt, (h, w))
        cur_src = O.resize_images(stacked, (h, w))
        depth = tgt.dtype.type(1) / disps[ns].reshape(B, h * w)
        K = intrinsics[:, ns]
        _, cam = O.pixel2cam(depth, O.batch_inv3(K), h, w)
        e, msk, e_id = np.zeros((B, S, h, w)), np.zeros((B, S, h, w), bool), np.zeros((B, S, h, w))
        for i in range(S):
            img = cur_src[:, 3 * i:3 * i + 3]
            Pf, _, deg = border_sampler(img, O.cam2pixel(cam, O.proj_tgt_to_src(poses[:, i], K), h, w), h, w)
            P, m = Pf.reshape(B, 3, h, w), deg.reshape(B, 1, h, w)
            for out, X, mm in ((e, P, m), (e_id, img, np.zeros_like(m))):
                v = (1 - r) * np.where(mm, 0.0, np.abs(X - cur_tgt).astype(np.float64)).sum(1)
                if use_ssim:
                    v = v + r * (np.clip(ssim_terms_reflect(X, cur_tgt)['raw'], 0, 1) * (1 - mm)).astype(np.float64).sum(1)
                out[:, i] = v
            msk[:, i] = m[:, 0]
        out_e.append(e)
        out_m.append(msk)
        out_id.append(e_id)
    return out_e, out_m, out_id


def loss_min_reprojection(tgt, src, intrinsics, disps, poses, cfg, automask=True, selection=None, want_grads=True,
                          want_intrinsics_grad=False, raw_disp_scales=0, raw_pose=False):
    """tests/min_reprojection_oracle.sfm_loss_min_reprojection under the flag (the same selection rules)."""
    S = src.shape[1]
    if selection is None:
        dd = [O.disp_activation(d)[0] if (raw_disp_scales >> s) & 1 else d for s, d in enumerate(disps)]
        pp = O.pose_from_raw(poses, S) if raw_pose else poses
        e, m, e_id = errors(tgt, src, intrinsics, dd, pp, cfg)
        selection = [MR.select(e[s], m[s], e_id[s], automask) for s in range(cfg.n_scales)]
    kw = dict(pixel_weights=[MR.one_hot(sel, S, tgt.dtype) for sel in selection], want_grads=want_grads,
              want_intrinsics_grad=want_intrinsics_grad)
    L, G = loss_pixel_raw(tgt, src, intrinsics, disps, poses, cfg, raw_disp_scales=raw_disp_scales, raw_pose=raw_pose, **kw)
    return dict(L, selection=selection), G


def loss_full_res(tgt, src, intrinsics, disps, poses, cfg, pixel_weights=None, min_reprojection=False, automask=True,
                  selection=None, want_grads=True):
    """tests/full_res_oracle.sfm_loss_full_res under the flag (no raw inputs): the photometric terms of scale s are those
    of a one-scale call with intrinsics[:, :1] and U_s(d_s), the smoothness stays at the native scales."""
    dt = tgt.dtype
    B, S, _, H, W = src.shape
    ns = cfg.n_scales
    cfg1 = O.LossConfig(ssim_rate=cfg.ssim_rate, n_scales=1, B_global=cfg.B_global)
    K0 = np.ascontiguousarray(intrinsics[:, :1])
    pixel = ssim = 0.0
    maps, sels = [], []
    gdisp = [np.zeros(d.shape) for d in disps]
    gpose = np.zeros((B, S, 6))
    for s in range(ns):
        u = disps[0] if s == 0 else upsample(disps[s], H, W)
        if min_reprojection:
            L, G = loss_min_reprojection(tgt, src, K0, [u], poses, cfg1, automask=automask, want_grads=want_grads,
                                         selection=None if selection is None else [selection[s]])
            sels.append(L['selection'][0])
        else:
            w = None if pixel_weights is None else [pixel_weights[s]]
            L, G = loss_pixel(tgt, src, K0, [u], poses, cfg1, pixel_weights=w, want_grads=want_grads)
        pixel += L['pixel_loss']
        ssim += L['ssim_loss']
        maps.append(L['pixel_losses'][0])
        if want_grads:
            g = G['gdisp'][0].astype(np.float64)
            gdisp[s] += g if s == 0 else upsample_adjoint(g, *disps[s].shape[2:], dtype=dt)
            gpose += G['gpose']
    smooth, gsm = _smoothness(tgt, src, intrinsics, disps, poses, cfg, want_grads)
    r = cfg.ssim_rate if cfg.ssim_rate else 0.0
    losses = dict(total_loss=(1 - r) * pixel + r * ssim + smooth, pixel_loss=pixel, smooth_loss=smooth, exp_loss=0.0,
                  ssim_loss=ssim, pixel_losses=maps)
    if min_reprojection:
        losses['selection'] = sels
    if not want_grads:
        return losses, None
    if gsm is not None:
        gdisp = [g + sm.astype(np.float64) for g, sm in zip(gdisp, gsm)]
    return losses, dict(gdisp=[g.astype(dt) for g in gdisp], gpose=gpose.astype(dt))
