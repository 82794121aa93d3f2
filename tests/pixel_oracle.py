"""Reference of the loss with per-pixel weights and of the per-pixel loss maps, in numpy on the oracle's helpers.

The loss loop of `oracle.sfm_loss` restated for the photometric terms weighted per (pixel, source): the weights
multiply `err * sigma` (or `err`) and the SSIM term, and with them the factors of dL/dP and of glogits; the smoothness
and explainability regularisers are not weighted.  The map of a (pixel, source) is d total / d M, which does not depend
on M.  With `pixel_weights=None` the arithmetic is that of `oracle.sfm_loss` (checked bit for bit in
tests/test_pixel_terms_cpu.py), so the copy cannot drift unnoticed.  No image gradients and no debug dumps."""
import numpy as np

from oracle import sfm_oracle as O


def sfm_loss_pixel(tgt, src, intrinsics, disps, poses, logits, cfg, pixel_weights=None, want_grads=True,
                   want_intrinsics_grad=False, proj_override=None, kinv_override=None):
    """-> (losses dict with `pixel_losses`, a list of (B,S,h_s,w_s) float64 maps, grads dict or None).

    pixel_weights: None, or a list of n_scales (B,S,h_s,w_s) arrays or None entries (None = 1).  The grads dict has
    the keys of oracle.sfm_loss (gdisp, gpose, glogits, dT; with want_intrinsics_grad also dP and gintrinsics)."""
    if want_intrinsics_grad and not want_grads:
        raise ValueError('the intrinsics gradient needs want_grads')
    dt = tgt.dtype
    B, S, _, H, W = src.shape
    Bg = cfg.B_global if cfg.B_global else B
    ns_total = cfg.n_scales
    stacked = src.reshape(B, 3 * S, H, W)
    pixel_loss = smooth_loss = exp_loss = ssim_loss = 0.0
    use_exp = bool(cfg.exp_reg)
    use_ssim = (not use_exp) and bool(cfg.ssim_rate)
    use_smooth = bool(cfg.smooth_reg)
    r = cfg.ssim_rate if cfg.ssim_rate else 0.0
    gdisp = [np.zeros(d.shape, np.float64) for d in disps]
    glogits = [np.zeros(l.shape, np.float64) for l in logits] if (use_exp and logits is not None) else None
    dP_all = [[None] * ns_total for _ in range(S)]
    maps = []
    for ns in range(ns_total):
        h, w = O.scale_shape(H, W, ns)
        hw_n = h * w
        cur_tgt = O.resize_images(tgt, (h, w))
        cur_src = O.resize_images(stacked, (h, w))
        D = disps[ns]
        maps.append(np.zeros((B, S, h, w), np.float64))
        if use_smooth and cfg.edge_aware_smooth:                     # base_model.py:144-155
            wgt = cfg.smooth_reg / (2 ** ns)
            d_dx, e_x, d_dy, e_y = O.disp_smooth_terms(cur_tgt, D)
            n_x, n_y = Bg * h * (w - 1), Bg * (h - 1) * w
            smooth_loss += wgt * (O._fsum(np.abs(d_dx) * e_x) / n_x + O._fsum(np.abs(d_dy) * e_y) / n_y)
            if want_grads:
                g = gdisp[ns][:, 0]
                sx = np.sign(d_dx[:, 0]).astype(np.float64) * e_x[:, 0] * (wgt / n_x)
                g[:, :, 1:] += sx
                g[:, :, :-1] -= sx
                sy = np.sign(d_dy[:, 0]).astype(np.float64) * e_y[:, 0] * (wgt / n_y)
                g[:, 1:, :] += sy
                g[:, :-1, :] -= sy
        elif use_smooth:                                             # base_model.py:169-185
            wgt = cfg.smooth_reg / (2 ** ns)
            dx2, dxdy, dydx, dy2 = O.smooth_terms(D)
            n_dx2, n_mix, n_dy2 = Bg * h * (w - 2), Bg * (h - 1) * (w - 1), Bg * (h - 2) * w
            smooth_loss += wgt * (O._fsum(np.abs(dx2)) / n_dx2 + O._fsum(np.abs(dxdy)) / n_mix
                                  + O._fsum(np.abs(dydx)) / n_mix + O._fsum(np.abs(dy2)) / n_dy2)
            if want_grads:
                g = gdisp[ns][:, 0]
                s = np.sign(dx2[:, 0]).astype(np.float64) * (wgt / n_dx2)
                g[:, :, :-2] += s
                g[:, :, 1:-1] -= 2 * s
                g[:, :, 2:] += s
                s = np.sign(dy2[:, 0]).astype(np.float64) * (wgt / n_dy2)
                g[:, :-2, :] += s
                g[:, 1:-1, :] -= 2 * s
                g[:, 2:, :] += s
                for m in (dxdy, dydx):
                    s = np.sign(m[:, 0]).astype(np.float64) * (wgt / n_mix)
                    g[:, 1:, 1:] += s
                    g[:, 1:, :-1] -= s
                    g[:, :-1, 1:] -= s
                    g[:, :-1, :-1] += s
        disp_flat = D.reshape(B, hw_n)
        depth = dt.type(1) / disp_flat
        K = intrinsics[:, ns]
        Kinv = kinv_override[:, ns] if kinv_override is not None else O.batch_inv3(K)
        ray, cam = O.pixel2cam(depth, Kinv, h, w)
        g_depth = np.zeros((B, hw_n), np.float64)
        for i in range(S):
            img = cur_src[:, 3 * i:3 * i + 3]
            proj = proj_override[:, i, ns] if proj_override is not None else O.proj_tgt_to_src(poses[:, i], K)
            gr = O.cam2pixel(cam, proj, h, w)
            Pf, t = O.spatial_transformer_sampler(img, gr['xn'], gr['yn'])
            P = Pf.reshape(B, 3, h, w)
            diff = P - cur_tgt
            err = np.abs(diff)
            m = np.all(P == 0, axis=1, keepdims=True)               # base_model.py:96
            err = np.where(m, dt.type(0), err)
            n_pix3 = Bg * 3 * h * w
            gP = np.zeros(P.shape, np.float64)
            sgn = np.where(m, 0.0, np.sign(diff)).astype(np.float64)
            Mw = None                                                # weight (B,1,h,w) of this source, None = 1
            if pixel_weights is not None and pixel_weights[ns] is not None:
                Mw = pixel_weights[ns][:, i:i + 1]
            M64 = 1.0 if Mw is None else Mw.astype(np.float64)
            e_sum = np.sum(err.astype(np.float64), axis=1, keepdims=True)
            if use_exp:
                l = logits[ns][:, i:i + 1]
                sg = O._sigmoid(l)
                sg64 = sg.astype(np.float64)
                maps[ns][:, i] += (e_sum * sg64 * ((1 - r) / n_pix3))[:, 0]
                exp_loss += cfg.exp_reg * O._fsum(O._softplus_neg(l)) / (Bg * h * w)
                pixel_loss += O._fsum(err * sg if Mw is None else err * sg * Mw) / n_pix3
                if want_grads:
                    gP += sgn * sg64 * M64 * ((1 - r) / n_pix3)
                    glogits[ns][:, i:i + 1] += ((1 - r) * (e_sum * M64) * sg64 * (1 - sg64) / n_pix3
                                                - cfg.exp_reg * (1 - sg64) / (Bg * h * w))
            else:
                maps[ns][:, i] += (e_sum * ((1 - r) / n_pix3))[:, 0]
                pixel_loss += O._fsum(err if Mw is None else err * Mw) / n_pix3
                if want_grads:
                    gP += sgn * M64 * ((1 - r) / n_pix3)
            if use_ssim:
                st = O.ssim_terms(P, cur_tgt)
                e = np.clip(st['raw'], 0, 1) * (1 - m)
                maps[ns][:, i] += np.sum(e.astype(np.float64), axis=1) * (r / n_pix3)
                ssim_loss += O._fsum(e if Mw is None else e * Mw) / n_pix3
                if want_grads:
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
                    gP += O.avg_pool3(g_a) + 2 * Pd * O.avg_pool3(g_s) + Td * O.avg_pool3(g_c)
            if want_grads:                                           # sampler -> grid -> q -> cam / proj (A.6)
                gyf = gP.reshape(B, 3, hw_n)
                t64 = {k: (v.astype(np.float64) if v.dtype.kind == 'f' else v) for k, v in t.items()}
                g_xn, g_yn = O.spatial_transformer_sampler_grad(t64, gyf, h, w)
                g_xn = g_xn * np.where(gr['inx'], 1.0, 2.0)
                g_yn = g_yn * np.where(gr['iny'], 1.0, 2.0)
                q = gr['q'].astype(np.float64)
                z = gr['z'].astype(np.float64)
                hw_, hh_ = float(gr['hw']), float(gr['hh'])
                with np.errstate(divide='ignore', invalid='ignore'):
                    g_q0 = g_xn / (z * hw_)
                    g_q1 = g_yn / (z * hh_)
                    g_q2 = -(g_xn * q[:, 0] / hw_ + g_yn * q[:, 1] / hh_) / (z * z)
                g_q = np.stack([g_q0, g_q1, g_q2], axis=1)
                g_q = np.where(t['any_valid'][:, None], g_q, 0.0)
                P64 = proj.astype(np.float64)
                g_cam = np.einsum('nkp,nkj->njp', g_q, P64[:, :3, :3])
                g_depth += np.sum(g_cam * ray.astype(np.float64), axis=1)
                cam4 = np.concatenate([cam.astype(np.float64), np.ones((B, 1, hw_n))], axis=1)
                dP_all[i][ns] = np.einsum('nkp,njp->nkj', g_q, cam4)
        if want_grads:
            d64 = disp_flat.astype(np.float64)
            gdisp[ns] += (-g_depth / (d64 * d64)).reshape(D.shape)
    total = (1 - r) * pixel_loss + r * ssim_loss + smooth_loss + exp_loss
    losses = dict(total_loss=total, pixel_loss=pixel_loss, smooth_loss=smooth_loss, exp_loss=exp_loss,
                  ssim_loss=ssim_loss, pixel_losses=maps)
    if not want_grads:
        return losses, None
    gpose = np.zeros((B, S, 6), dt)
    dT_all = np.zeros((B, S, 3, 4), np.float64)
    K_scales = [intrinsics[:, ns] for ns in range(ns_total)]
    for i in range(S):
        gpose[:, i], dT_all[:, i] = O._pose_backward(poses[:, i], K_scales, dP_all[i])
    grads = dict(gdisp=[g.astype(dt) for g in gdisp], gpose=gpose,
                 glogits=[g.astype(dt) for g in glogits] if glogits is not None else None, dT=dT_all)
    if want_intrinsics_grad:
        dP = np.stack([np.stack(dP_all[i], 1) for i in range(S)], 1)
        grads.update(dP=dP, gintrinsics=O.intrinsics_grad(intrinsics, poses, dP))
    return losses, grads


def sfm_loss_pixel_raw(tgt, src, intrinsics, disps_in, poses_in, logits, cfg, raw_disp_scales=0, raw_pose=False, **kw):
    """sfm_loss_pixel with the seam included, as oracle.sfm_loss_raw: the scales of `raw_disp_scales` take the
    pre-activation disparity map, `raw_pose` the poseout map; the gradients are w.r.t. what was passed in."""
    S = src.shape[1]
    disps, dacts = [], []
    for s, d in enumerate(disps_in):
        if (raw_disp_scales >> s) & 1:
            dd, da = O.disp_activation(d)
            disps.append(dd)
            dacts.append(da)
        else:
            disps.append(d)
            dacts.append(None)
    poses = O.pose_from_raw(poses_in, S) if raw_pose else poses_in
    losses, grads = sfm_loss_pixel(tgt, src, intrinsics, disps, poses, logits, cfg, **kw)
    if grads is not None:
        grads = dict(grads)
        grads['gdisp'] = [g if da is None else (g.astype(np.float64) * da).astype(g.dtype) for g, da in zip(grads['gdisp'], dacts)]
        if raw_pose:
            n = int(np.prod(poses_in.shape[2:]))
            gp = grads['gpose'].astype(np.float64).reshape(poses_in.shape[0], 6 * S, *([1] * (poses_in.ndim - 2)))
            grads['gpose'] = np.broadcast_to(gp * (0.01 / n), poses_in.shape).astype(poses_in.dtype)
    return losses, grads
