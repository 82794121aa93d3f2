"""Reference of the mean-normalised smoothness (SFM_FLAG_MEAN_NORM_SMOOTH) and of Monodepth2's edge weight
(SFM_FLAG_EDGE_MEAN_ABS), built on the numpy oracle's helpers.

`smoothness` evaluates either smoothness kind per (snippet, scale) on the native planes, with the oracle's arithmetic
(differences in the disparity's dtype, sums in fp64) and optionally Monodepth2's edge weight exp(-mean_c |dI_c|).  With
mean_norm, the term of (b, s) is evaluated on d / (m_bs + 1e-7), m_bs the mean of the activated disparity, through the
homogeneity identity: loss r L_bs, gradient r G_j - r^2 L_bs / N.  `add_smoothness` adds it to the losses and gradients of
any existing reference (pixel_oracle, min_reprojection_oracle, full_res_oracle) run with smooth_reg = 0."""
import numpy as np

from oracle import sfm_oracle as O


def edge_weights(img, dt, mean_abs):
    """(e_x, e_y) of compute_disp_smooth on img (B,3,h,w): exp(-|mean_c dI|), or exp(-mean_c |dI|) with mean_abs."""
    i_dy = img[:, :, 1:] - img[:, :, :-1]
    i_dx = img[:, :, :, 1:] - img[:, :, :, :-1]
    if mean_abs:
        e_x = np.exp(-np.abs(i_dx).mean(axis=1, keepdims=True, dtype=dt))
        e_y = np.exp(-np.abs(i_dy).mean(axis=1, keepdims=True, dtype=dt))
    else:
        e_x = np.exp(-np.abs(i_dx.mean(axis=1, keepdims=True, dtype=dt)))
        e_y = np.exp(-np.abs(i_dy.mean(axis=1, keepdims=True, dtype=dt)))
    return e_x.astype(dt), e_y.astype(dt)


def smoothness(tgt, disps, cfg, raw_disp_scales=0, mean_norm=True, edge_mean_abs=False, snippet_weights=None,
               want_grads=True):
    """-> (loss, rows, gdisp): loss = sum_b w_b l_b (float), rows (B,) the unweighted per-snippet l_b (with the 1/B_global
    means), gdisp a list of (B,1,h_s,w_s) float64 gradients of `loss` w.r.t. the caller's maps (raw bits: pre-activation),
    or None.  cfg: smooth_reg, n_scales, B_global, edge_aware_smooth."""
    B, _, H, W = tgt.shape
    Bg = cfg.B_global or B
    wb = np.ones(B) if snippet_weights is None else np.asarray(snippet_weights, np.float64)
    rows = np.zeros(B)
    gdisp = []
    for s in range(cfg.n_scales):
        h, w = O.scale_shape(H, W, s)
        x = disps[s]
        D, dact = O.disp_activation(x) if (raw_disp_scales >> s) & 1 else (x, None)
        wgt = cfg.smooth_reg / (2 ** s)
        g = np.zeros((B, h, w))
        if cfg.edge_aware_smooth:
            e_x, e_y = edge_weights(O.resize_images(tgt, (h, w)), D.dtype, edge_mean_abs)
            d_dx = D[:, :, :, 1:] - D[:, :, :, :-1]
            d_dy = D[:, :, 1:] - D[:, :, :-1]
            n_x, n_y = Bg * h * (w - 1), Bg * (h - 1) * w
            L = wgt * (np.sum(np.abs(d_dx) * e_x, axis=(1, 2, 3), dtype=np.float64) / n_x
                       + np.sum(np.abs(d_dy) * e_y, axis=(1, 2, 3), dtype=np.float64) / n_y)
            sx = np.sign(d_dx[:, 0]).astype(np.float64) * e_x[:, 0] * (wgt / n_x)
            g[:, :, 1:] += sx
            g[:, :, :-1] -= sx
            sy = np.sign(d_dy[:, 0]).astype(np.float64) * e_y[:, 0] * (wgt / n_y)
            g[:, 1:, :] += sy
            g[:, :-1, :] -= sy
        else:
            dx2, dxdy, dydx, dy2 = O.smooth_terms(D)
            n_dx2, n_mix, n_dy2 = Bg * h * (w - 2), Bg * (h - 1) * (w - 1), Bg * (h - 2) * w
            ssum = lambda a: np.sum(np.abs(a), axis=(1, 2, 3), dtype=np.float64)
            L = wgt * (ssum(dx2) / n_dx2 + ssum(dxdy) / n_mix + ssum(dydx) / n_mix + ssum(dy2) / n_dy2)
            t = np.sign(dx2[:, 0]).astype(np.float64) * (wgt / n_dx2)
            g[:, :, :-2] += t
            g[:, :, 1:-1] -= 2 * t
            g[:, :, 2:] += t
            t = np.sign(dy2[:, 0]).astype(np.float64) * (wgt / n_dy2)
            g[:, :-2, :] += t
            g[:, 1:-1, :] -= 2 * t
            g[:, 2:, :] += t
            for m in (dxdy, dydx):
                t = np.sign(m[:, 0]).astype(np.float64) * (wgt / n_mix)
                g[:, 1:, 1:] += t
                g[:, :-1, :-1] += t
                g[:, 1:, :-1] -= t
                g[:, :-1, 1:] -= t
        if mean_norm:
            r = 1.0 / (D.astype(np.float64).mean(axis=(1, 2, 3)) + 1e-7)
            g = r[:, None, None] * g - (r * r * L / (h * w))[:, None, None]
            L = r * L
        rows += L
        g = g * wb[:, None, None]
        if dact is not None:
            g = g * dact[:, 0].astype(np.float64)
        gdisp.append(g[:, None])
    loss = float(np.sum(wb * rows))
    return loss, rows, (gdisp if want_grads else None)


def add_smoothness(losses, grads, tgt, disps, cfg, raw_disp_scales=0, mean_norm=True, edge_mean_abs=False):
    """losses / grads of a reference run with smooth_reg = 0 (the oracle's dict layout) -> the same with the smoothness
    term of `cfg` added."""
    loss, _, g = smoothness(tgt, disps, cfg, raw_disp_scales, mean_norm, edge_mean_abs, want_grads=grads is not None)
    losses = dict(losses)
    losses['smooth_loss'] = losses.get('smooth_loss', 0.0) + loss
    losses['total_loss'] = losses['total_loss'] + loss
    if grads is None:
        return losses, None
    grads = dict(grads)
    grads['gdisp'] = [a.astype(np.float64) + b for a, b in zip(grads['gdisp'], g)]
    return losses, grads
