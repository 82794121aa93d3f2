"""TEST INFRASTRUCTURE: the numpy oracle's counterpart of the image gradients of the fused loss.

d total / d tgt_img and d total / d src_imgs of SFMLearner.__call__'s loss loop (base_model.py:57-124) with the images
treated as differentiable: the reference's `.data` on the pyramid (:71-72) and on mu_y / sigma_y (:131, :134) are
lifted, so the result is the derivative of the reported total.  The all-zero mask (:96) is piecewise constant
(derivative 0); the smoothness term and the explainability regulariser do not depend on the images.  Built on the
building blocks of oracle/sfm_oracle.py (same forward arithmetic, dtype generic), everything backward in float64:
  * the sampler's adjoint: every pixel scatters dL/dP_c * w_k to its valid taps (np.add.at);
  * the SSIM derivative w.r.t. T: A(g_my) + 2 T A(g_s) + P A(g_c), avg_pool3 being its own adjoint;
  * the pyramid's adjoint: scale 0 is the identity, the other levels pull back through the adjoint of resize_images
    with the forward's tap weights (resize_axis_tables).
"""
import numpy as np

from oracle import sfm_oracle as O


def resize_images_adjoint(gy, in_shape, dtype=np.float32):
    """Adjoint of O.resize_images (float64): gy (B,C,oh,ow) -> (B,C,H,W).  The tap weights are the forward's, float64
    products rounded to `dtype`.  The identity when the sizes agree (scale 0)."""
    B, C, oh, ow = gy.shape
    H, W = in_shape
    if (oh, ow) == (H, W):
        return gy.astype(np.float64)
    u0, ua, ub = O.resize_axis_tables(W, ow)
    v0, va, vb = O.resize_axis_tables(H, oh)
    gx = np.zeros((B, C, H, W), np.float64)
    V0, U0 = np.broadcast_arrays(v0[:, None], u0[None, :])
    for wv, wu, dv, du in ((va, ua, 0, 0), (va, ub, 0, 1), (vb, ua, 1, 0), (vb, ub, 1, 1)):
        wk = (wv[:, None] * wu[None, :]).astype(dtype).astype(np.float64)
        np.add.at(gx.transpose(2, 3, 0, 1), (V0 + dv, U0 + du), (wk * gy).transpose(2, 3, 0, 1))
    return gx


def sampler_image_adjoint(t, gP, h, w):
    """Gradient of O.spatial_transformer_sampler w.r.t. its image (float64): every pixel scatters gP_c * w_k to its
    valid taps; a pixel with no valid tap (out of view by the x2 rule) contributes nothing.  t: the tap record of the
    forward, gP (N,3,hw) -> (N,3,h*w)."""
    N = gP.shape[0]
    u0, v0 = t['u0'].astype(np.int64), t['v0'].astype(np.int64)
    wa, wb = t['wa'].astype(np.float64), t['wb'].astype(np.float64)
    wc, wd = t['wc'].astype(np.float64), t['wd'].astype(np.float64)
    out = np.zeros((N, 3, h * w), np.float64)
    bi = np.broadcast_to(np.arange(N)[:, None], u0.shape)
    for du, dv, wk in ((0, 0, wa * wc), (1, 0, wb * wc), (0, 1, wa * wd), (1, 1, wb * wd)):
        uu, vv = u0 + du, v0 + dv
        ok = t['any_valid'] & (uu >= 0) & (uu <= w - 1) & (vv >= 0) & (vv <= h - 1)
        wk = wk.astype(t['wa'].dtype).astype(np.float64)      # the forward rounds the weight products to the image dtype
        idx = np.where(ok, vv * w + uu, 0)
        for c in range(3):
            np.add.at(out[:, c], (bi, idx), np.where(ok, wk * gP[:, c], 0.0))
    return out


def image_grads(tgt, src, intrinsics, disps, poses, logits, cfg, proj_override=None, kinv_override=None):
    """-> (gtgt (B,3,H,W), gsrc (B,S,3,H,W)) in float64; arguments as O.sfm_loss (disps activated)."""
    if cfg.smooth_reg and cfg.edge_aware_smooth:
        raise ValueError('image gradients through the edge-aware smoothness term are not supported')
    dt = tgt.dtype
    B, S, _, H, W = src.shape
    Bg = cfg.B_global if cfg.B_global else B
    use_exp = bool(cfg.exp_reg)
    use_ssim = (not use_exp) and bool(cfg.ssim_rate)
    rate = cfg.ssim_rate if cfg.ssim_rate else 0.0
    stacked = src.reshape(B, 3 * S, H, W)
    gtgt = np.zeros(tgt.shape, np.float64)
    gsrc = np.zeros(src.shape, np.float64)
    for ns in range(cfg.n_scales):
        h, w = O.scale_shape(H, W, ns)
        cur_tgt = O.resize_images(tgt, (h, w))
        cur_src = O.resize_images(stacked, (h, w))
        T64 = cur_tgt.astype(np.float64)
        depth = dt.type(1) / disps[ns].reshape(B, h * w)
        K = intrinsics[:, ns]
        Kinv = kinv_override[:, ns] if kinv_override is not None else O.batch_inv3(K)
        _, cam = O.pixel2cam(depth, Kinv, h, w)
        n3 = Bg * 3 * h * w
        gT = np.zeros((B, 3, h, w), np.float64)
        gS = np.zeros((B, S, 3, h, w), np.float64)
        for i in range(S):
            proj = proj_override[:, i, ns] if proj_override is not None else O.proj_tgt_to_src(poses[:, i], K)
            gr = O.cam2pixel(cam, proj, h, w)
            Pf, t = O.spatial_transformer_sampler(cur_src[:, 3 * i:3 * i + 3], gr['xn'], gr['yn'])
            P = Pf.reshape(B, 3, h, w)
            m = np.all(P == 0, axis=1, keepdims=True)
            sgn = np.where(m, 0.0, np.sign(P - cur_tgt)).astype(np.float64)
            wl1 = (1 - rate) / n3
            if use_exp:
                wl1 = wl1 * O._sigmoid(logits[ns][:, i:i + 1]).astype(np.float64)
            gP = sgn * wl1
            gT -= sgn * wl1
            if use_ssim:
                st = O.ssim_terms(P, cur_tgt)
                f = {k: st[k].astype(np.float64) for k in ('raw', 'a', 'my', 'n1', 'n2', 'd1', 'd2', 'n', 'd')}
                g_e = (rate / n3) * (1 - m) * ((f['raw'] >= 0) & (f['raw'] <= 1))
                g_n = -g_e / (2 * f['d'])
                g_d = g_e * f['n'] / (2 * f['d'] * f['d'])
                g_a = g_n * (2 * f['my'] * f['n2'] - 2 * f['my'] * f['n1']) + g_d * (2 * f['a'] * f['d2'] - 2 * f['a'] * f['d1'])
                g_my = g_n * (2 * f['a'] * f['n2'] - 2 * f['a'] * f['n1']) + g_d * (2 * f['my'] * f['d2'] - 2 * f['my'] * f['d1'])
                g_s = g_d * f['d1']
                g_c = 2 * g_n * f['n1']
                P64 = P.astype(np.float64)
                As, Ac = O.avg_pool3(g_s), O.avg_pool3(g_c)
                gP = gP + O.avg_pool3(g_a) + 2 * P64 * As + T64 * Ac
                gT += O.avg_pool3(g_my) + 2 * T64 * As + P64 * Ac
            gS[:, i] = sampler_image_adjoint(t, gP.reshape(B, 3, h * w), h, w).reshape(B, 3, h, w)
        gtgt += resize_images_adjoint(gT, (H, W), dt)
        gsrc += resize_images_adjoint(gS.reshape(B, 3 * S, h, w), (H, W), dt).reshape(src.shape)
    return gtgt, gsrc


def sfm_loss_with_image_grads(tgt, src, intrinsics, disps, poses, logits, cfg, proj_override=None, kinv_override=None,
                              **kw):
    """O.sfm_loss, its grads dict completed with gtgt / gsrc."""
    L, G, dbg = O.sfm_loss(tgt, src, intrinsics, disps, poses, logits, cfg, proj_override=proj_override,
                           kinv_override=kinv_override, **kw)
    G = dict(G)
    G['gtgt'], G['gsrc'] = image_grads(tgt, src, intrinsics, disps, poses, logits, cfg, proj_override, kinv_override)
    return L, G, dbg


def sfm_loss_raw_with_image_grads(tgt, src, intrinsics, disps_in, poses_in, logits, cfg, **kw):
    """O.sfm_loss_raw, its grads dict completed with gtgt / gsrc (computed on the activated disparities)."""
    L, G, dbg = O.sfm_loss_raw(tgt, src, intrinsics, disps_in, poses_in, logits, cfg, **kw)
    G = dict(G)
    G['gtgt'], G['gsrc'] = image_grads(tgt, src, intrinsics, dbg['disps'], dbg['poses'], logits, cfg)
    return L, G, dbg
