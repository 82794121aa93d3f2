"""Reference of sfm_loss_geometry_valid_mean (SC-SfMLearner's means over the valid pixels, its auto-mask and its clamped
L1), in numpy on the oracle's helpers, tests/geometry_oracle.py and the per-pixel reference (tests/pixel_oracle.py).

Per scale s and source i: the projection, D_diff and the in-view flag are those of geometry_oracle.geometry_terms; the
warped source W is the oracle's sampler.  The valid-pixel mask a is the in-view flag (times w_b != 0), and with the
auto-mask also ((E_0 + E_1) + E_2) / 3 < ((|T_0 - S_0| + |T_1 - S_1|) + |T_2 - S_2|) / 3 in fp32, E_c = min(|T_c - W_c|, 1).
n counts a over the snippets of a group.  The photometric loop is that of pixel_oracle.sfm_loss_pixel without the
explainability branch, with the clamped L1 (its gradient passes where |d| <= 1) and the weights a M (B h w) / n, formed in
fp32 as the device does (0 where 3 n <= min_count); the geometry term is geometry_reg sum_a D_diff / n (0 where
n <= min_count).  The upstream of D_diff is a (geometry_reg / n - map (B h w) / n), chained in fp64 as in the geometry
reference.  `masks` (a list of (B,S,h,w)) replaces the computed auto-mask, so that the device's choice at near ties can be
fed back; it is still ANDed with the in-view flag."""
import numpy as np

from oracle import sfm_oracle as O
from tests import axisangle_oracle as AA
from tests import geometry_oracle as GO


def automask_sides(cur_tgt, img, gr):
    """-> (e, e_id) (B,h,w) fp32: the two sides of the auto-mask's comparison for one source at one scale."""
    f = np.float32
    B, _, h, w = cur_tgt.shape
    Pf, _ = O.spatial_transformer_sampler(img, gr['xn'], gr['yn'])
    P = Pf.reshape(B, 3, h, w)
    E = np.minimum(np.abs(P - cur_tgt), f(1))
    Ei = np.abs(cur_tgt - img)
    return ((E[:, 0] + E[:, 1]) + E[:, 2]).astype(f) / f(3), ((Ei[:, 0] + Ei[:, 1]) + Ei[:, 2]).astype(f) / f(3)


def near_ties(tgt, src, intrinsics, disps, poses, src_disps, cfg, rel=1e-4):
    """-> list over scales of (B,S,h,w) bool: pairs whose auto-mask sides agree to `rel`."""
    B, S, _, H, W = src.shape
    terms = GO.geometry_terms(intrinsics, disps, poses, src_disps, cfg)
    out = []
    for T_ in terms:
        h, w = T_['h'], T_['w']
        cur_tgt = O.resize_images(tgt, (h, w))
        cur_src = O.resize_images(src.reshape(B, 3 * S, H, W), (h, w))
        t = np.zeros((B, S, h, w), bool)
        for i in range(S):
            e, ei = automask_sides(cur_tgt, cur_src[:, 3 * i:3 * i + 3], T_['per'][i]['gr'])
            t[:, i] = np.abs(e - ei) <= rel * np.maximum(np.abs(ei), np.abs(e))
        out.append(t)
    return out


def valid_masks(tgt, src, terms, automask, snippet_weights=None, masks=None):
    """-> list over scales of (B,S,h,w) bool: a."""
    B, S, _, H, W = src.shape
    stacked = src.reshape(B, 3 * S, H, W)
    out = []
    for ns, T_ in enumerate(terms):
        h, w = T_['h'], T_['w']
        cur_tgt = O.resize_images(tgt, (h, w))
        cur_src = O.resize_images(stacked, (h, w))
        a = np.zeros((B, S, h, w), bool)
        for i in range(S):
            r = T_['per'][i]
            ok = r['inb'].reshape(B, h, w).copy()
            if snippet_weights is not None:
                ok &= (np.asarray(snippet_weights) != 0)[:, None, None]
            if masks is not None:
                ok &= masks[ns][:, i].astype(bool)
            elif automask:
                e, ei = automask_sides(cur_tgt, cur_src[:, 3 * i:3 * i + 3], r['gr'])
                ok &= e < ei
            a[:, i] = ok
        out.append(a)
    return out


def counts_of(a, groups):
    """-> (n_scales, S, G) int64 counts of a (list of (B,S,h,w) bool)."""
    out = []
    for m in a:
        B, S = m.shape[:2]
        per_b = m.reshape(B, S, -1).sum(-1)                 # (B,S)
        out.append(np.stack([per_b[g::groups].sum(0) for g in range(groups)], -1))
    return np.stack(out, 0)


def photometric_factor(n, min_count, bhw):
    """(B h w) / n rounded to fp32, 0 where 3 n <= min_count (the device's factor)."""
    n = np.asarray(n, np.float64)
    with np.errstate(divide='ignore'):
        return np.where((n > 0) & (3.0 * n > min_count), (bhw / np.maximum(n, 1)).astype(np.float32), np.float32(0))


def loss(tgt, src, intrinsics, disps, poses, src_disps, cfg, geometry_reg=0.5, self_mask=True, automask=True, groups=1,
         min_count=10000.0, snippet_weights=None, masks=None, want_grads=True, want_intrinsics_grad=False,
         proj_override=None, kinv_override=None, invert_sources=None):
    """-> (losses dict with geometry_diff, valid_masks (bool) and valid_counts, grads dict or None).

    grads: gdisp, gpose, gsrc_disp (float64), dT; with want_intrinsics_grad dP and gintrinsics.  snippet_weights: only
    the exclusion of zero-weight snippets (the weights must otherwise be 0 or 1)."""
    if cfg.exp_reg:
        raise ValueError('valid-pixel means: no explainability branch')
    if invert_sources is not None:
        proj_override, kinv_override = AA.tables(poses, intrinsics, invert_sources)
    dt = tgt.dtype
    B, S, _, H, W = src.shape
    terms = GO.geometry_terms(intrinsics, disps, poses, src_disps, cfg, proj_override, kinv_override)
    a_all = valid_masks(tgt, src, terms, automask, snippet_weights, masks)
    cnt = counts_of(a_all, groups)
    stacked = src.reshape(B, 3 * S, H, W)
    pixel_loss = smooth_loss = ssim_loss = geo = 0.0
    use_ssim = bool(cfg.ssim_rate)
    use_smooth = bool(cfg.smooth_reg)
    r = cfg.ssim_rate if cfg.ssim_rate else 0.0
    gdisp = [np.zeros(d.shape, np.float64) for d in disps]
    dP = np.zeros((B, S, cfg.n_scales, 3, 4))
    gsrc = [np.zeros(x.shape, np.float64) for x in src_disps]
    diffs = []
    for ns in range(cfg.n_scales):
        T_ = terms[ns]
        h, w = T_['h'], T_['w']
        hw_n = h * w
        cur_tgt = O.resize_images(tgt, (h, w))
        cur_src = O.resize_images(stacked, (h, w))
        D = disps[ns]
        if use_smooth and cfg.edge_aware_smooth:                     # as pixel_oracle
            wgt = cfg.smooth_reg / (2 ** ns)
            d_dx, e_x, d_dy, e_y = O.disp_smooth_terms(cur_tgt, D)
            n_x, n_y = B * h * (w - 1), B * (h - 1) * w
            smooth_loss += wgt * (O._fsum(np.abs(d_dx) * e_x) / n_x + O._fsum(np.abs(d_dy) * e_y) / n_y)
            if want_grads:
                g = gdisp[ns][:, 0]
                sx = np.sign(d_dx[:, 0]).astype(np.float64) * e_x[:, 0] * (wgt / n_x)
                g[:, :, 1:] += sx
                g[:, :, :-1] -= sx
                sy = np.sign(d_dy[:, 0]).astype(np.float64) * e_y[:, 0] * (wgt / n_y)
                g[:, 1:, :] += sy
                g[:, :-1, :] -= sy
        elif use_smooth:
            wgt = cfg.smooth_reg / (2 ** ns)
            dx2, dxdy, dydx, dy2 = O.smooth_terms(D)
            n_dx2, n_mix, n_dy2 = B * h * (w - 2), B * (h - 1) * (w - 1), B * (h - 2) * w
            smooth_loss += wgt * (O._fsum(np.abs(dx2)) / n_dx2 + O._fsum(np.abs(dxdy)) / n_mix
                                  + O._fsum(np.abs(dydx)) / n_mix + O._fsum(np.abs(dy2)) / n_dy2)
            if want_grads:
                g = gdisp[ns][:, 0]
                s_ = np.sign(dx2[:, 0]).astype(np.float64) * (wgt / n_dx2)
                g[:, :, :-2] += s_
                g[:, :, 1:-1] -= 2 * s_
                g[:, :, 2:] += s_
                s_ = np.sign(dy2[:, 0]).astype(np.float64) * (wgt / n_dy2)
                g[:, :-2, :] += s_
                g[:, 1:-1, :] -= 2 * s_
                g[:, 2:, :] += s_
                for m_ in (dxdy, dydx):
                    s_ = np.sign(m_[:, 0]).astype(np.float64) * (wgt / n_mix)
                    g[:, 1:, 1:] += s_
                    g[:, 1:, :-1] -= s_
                    g[:, :-1, 1:] -= s_
                    g[:, :-1, :-1] += s_
        ray, cam = T_['ray'], T_['cam']
        g_depth = np.zeros((B, hw_n), np.float64)
        n_pix3 = B * 3 * h * w
        diffs.append(np.stack([T_['per'][i]['diff'].reshape(B, h, w) for i in range(S)], 1))
        for i in range(S):
            rr = T_['per'][i]
            gr, t = rr['gr'], rr['t']
            a = a_all[ns][:, i]                                      # (B,h,w)
            grp = np.arange(B) % groups
            n_b = cnt[ns, i][grp].astype(np.float64)                 # (B,) the group's count
            fph = photometric_factor(n_b, min_count, B * h * w)     # (B,) fp32
            diff = diffs[ns][:, i]
            # in the inputs' precision (fp32: the device's rounding; fp64: no rounding steps for central differences)
            M = (dt.type(1) - diff).astype(dt) if self_mask else np.ones_like(diff)
            fd = fph.astype(dt) if dt == np.float32 else np.where(fph != 0, (B * h * w) / np.maximum(n_b, 1), 0.0)
            Wt = np.where(a, (M * fd[:, None, None]).astype(dt), dt.type(0))[:, None]   # (B,1,h,w)
            W64 = Wt.astype(np.float64)
            # geometry term: reg sum_a D_diff / n
            with np.errstate(divide='ignore', invalid='ignore'):
                wgeo = np.where(n_b > min_count, geometry_reg / np.maximum(n_b, 1), 0.0)   # (B,)
            geo += float(np.sum(np.sum(np.where(a, diff, 0).astype(np.float64), axis=(1, 2)) * wgeo))
            img = cur_src[:, 3 * i:3 * i + 3]
            Pf, t_img = O.spatial_transformer_sampler(img, gr['xn'], gr['yn'])
            P = Pf.reshape(B, 3, h, w)
            dff = P - cur_tgt
            m = np.all(P == 0, axis=1, keepdims=True)
            err = np.where(m, dt.type(0), np.minimum(np.abs(dff), dt.type(1)))
            sgn = np.where(m | (np.abs(dff) > 1), 0.0, np.sign(dff)).astype(np.float64)
            e_sum = np.sum(err.astype(np.float64), axis=1, keepdims=True)
            pmap = e_sum * ((1 - r) / n_pix3)
            pixel_loss += O._fsum(err * Wt) / n_pix3
            gP = sgn * W64 * ((1 - r) / n_pix3)
            if use_ssim:
                st = O.ssim_terms(P, cur_tgt)
                e = np.clip(st['raw'], 0, 1) * (1 - m)
                pmap = pmap + np.sum(e.astype(np.float64), axis=1, keepdims=True) * (r / n_pix3)
                ssim_loss += O._fsum(e * Wt) / n_pix3
                if want_grads:
                    raw = st['raw'].astype(np.float64)
                    a_, my = st['a'].astype(np.float64), st['my'].astype(np.float64)
                    n1, n2 = st['n1'].astype(np.float64), st['n2'].astype(np.float64)
                    d1, d2 = st['d1'].astype(np.float64), st['d2'].astype(np.float64)
                    n_, d_ = st['n'].astype(np.float64), st['d'].astype(np.float64)
                    g_e = (r / n_pix3) * (1 - m) * ((raw >= 0) & (raw <= 1)) * W64
                    g_n = -g_e / (2 * d_)
                    g_d = g_e * n_ / (2 * d_ * d_)
                    g_a = g_n * (2 * my * n2 - 2 * my * n1) + g_d * (2 * a_ * d2 - 2 * a_ * d1)
                    g_s = g_d * d1
                    g_c = 2 * g_n * n1
                    Pd, Td = P.astype(np.float64), cur_tgt.astype(np.float64)
                    gP += O.avg_pool3(g_a) + 2 * Pd * O.avg_pool3(g_s) + Td * O.avg_pool3(g_c)
            if not want_grads:
                continue
            P64 = rr['proj'].astype(np.float64)
            cam4 = np.concatenate([cam.astype(np.float64), np.ones((B, 1, hw_n))], axis=1)
            t64 = {k: (v.astype(np.float64) if v.dtype.kind == 'f' else v) for k, v in t.items()}
            q = gr['q'].astype(np.float64)
            z = gr['z'].astype(np.float64)
            hw_, hh_ = float(gr['hw']), float(gr['hh'])
            # photometric chain (pixel_oracle), on the colour image's sampler record
            ti64 = {k: (v.astype(np.float64) if v.dtype.kind == 'f' else v) for k, v in t_img.items()}
            g_xn, g_yn = O.spatial_transformer_sampler_grad(ti64, gP.reshape(B, 3, hw_n), h, w)
            g_xn = g_xn * np.where(gr['inx'], 1.0, 2.0)
            g_yn = g_yn * np.where(gr['iny'], 1.0, 2.0)
            with np.errstate(divide='ignore', invalid='ignore'):
                g_q = np.stack([g_xn / (z * hw_), g_yn / (z * hh_), -(g_xn * q[:, 0] / hw_ + g_yn * q[:, 1] / hh_) / (z * z)], 1)
            g_q = np.where(t_img['any_valid'][:, None], g_q, 0.0)
            g_depth += np.sum(np.einsum('nkp,nkj->njp', g_q, P64[:, :3, :3]) * ray.astype(np.float64), axis=1)
            dP[:, i, ns] += np.einsum('nkp,njp->nkj', g_q, cam4)
            # geometry chain (geometry_oracle) with the upstream a (reg / n - map (B h w) / n)
            up = wgeo[:, None] - (pmap[:, 0].reshape(B, hw_n) * fd[:, None].astype(np.float64) if self_mask else 0.0)
            up = np.where(a.reshape(B, hw_n), up, 0.0)
            ratio = rr['ratio'].astype(np.float64)
            ok = rr['inb'] & a.reshape(B, hw_n) & (ratio >= 0) & (ratio <= 1)
            aa, c = rr['a'].astype(np.float64), rr['c'].astype(np.float64)
            with np.errstate(divide='ignore', invalid='ignore'):
                gz = np.where(ok, up * (np.sign(aa) - ratio) / c, 0.0)
                gD = np.where(ok, up * (-np.sign(aa) - ratio) / c, 0.0)
            g_xn, g_yn = O.spatial_transformer_sampler_grad(t64, gD[:, None, :], h, w)
            with np.errstate(divide='ignore', invalid='ignore'):
                g_q0 = np.where(ok, g_xn / (z * hw_), 0.0)
                g_q1 = np.where(ok, g_yn / (z * hh_), 0.0)
                g_q2 = np.where(ok, gz - (g_xn * q[:, 0] / hw_ + g_yn * q[:, 1] / hh_) / (z * z), 0.0)
            g_q = np.stack([g_q0, g_q1, g_q2], axis=1)
            g_depth += np.sum(np.einsum('nkp,nkj->njp', g_q, P64[:, :3, :3]) * ray.astype(np.float64), axis=1)
            dP[:, i, ns] += np.einsum('nkp,njp->nkj', g_q, cam4)
            bb = np.repeat(np.arange(B), hw_n)
            u0, v0 = t64['u0'].reshape(-1), t64['v0'].reshape(-1)
            okf = ok.reshape(-1)
            wa, wb, wc, wd = (t64[k].reshape(-1) for k in ('wa', 'wb', 'wc', 'wd'))
            gDf = gD.reshape(-1)
            inv_img = 1.0 / src_disps[ns][:, i].astype(np.float64)
            for wk, dv, du in ((wa * wc, 0, 0), (wb * wc, 0, 1), (wa * wd, 1, 0), (wb * wd, 1, 1)):
                vv = np.clip(v0 + dv, 0, h - 1)
                uu = np.clip(u0 + du, 0, w - 1)
                np.add.at(gsrc[ns][:, i], (bb, vv, uu), np.where(okf, -gDf * wk * inv_img[bb, vv, uu] ** 2, 0.0))
        if want_grads:
            d64 = D.reshape(B, hw_n).astype(np.float64)
            gdisp[ns] += (-g_depth / (d64 * d64)).reshape(D.shape)
    total = (1 - r) * pixel_loss + r * ssim_loss + smooth_loss + geo
    L = dict(total_loss=total, pixel_loss=pixel_loss, smooth_loss=smooth_loss, exp_loss=geo, ssim_loss=ssim_loss,
             geometry_diff=diffs, valid_masks=a_all, valid_counts=cnt)
    if not want_grads:
        return L, None
    dT = np.zeros((B, S, 3, 4))
    K_scales = [intrinsics[:, s] for s in range(cfg.n_scales)]
    gpose = np.zeros((B, S, 6))
    for i in range(S):
        gpose[:, i], dT[:, i] = O._pose_backward(poses[:, i], K_scales, [dP[:, i, s] for s in range(cfg.n_scales)])
    if invert_sources is not None:
        gpose = AA.pose_grad(poses, dT, invert_sources)
    grads = dict(gdisp=gdisp, gpose=gpose, gsrc_disp=gsrc, dT=dT)
    if want_intrinsics_grad:
        grads['dP'] = dP
        grads['gintrinsics'] = (AA.intrinsics_grad_rt(intrinsics, poses, dP, invert_sources) if invert_sources is not None
                                else O.intrinsics_grad(intrinsics, poses, dP))
    return L, grads
