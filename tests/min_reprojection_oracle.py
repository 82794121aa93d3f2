"""Reference of per-pixel minimum reprojection with auto-masking (sfm_loss_min_reprojection), in numpy on the oracle.

The per-(pixel, source) reprojection errors and all-zero masks come from the oracle's warp and SSIM helpers, the
identity errors from the same helpers applied to the unwarped source levels, the selection follows the rules of
include/sfmloss.h, and the loss is tests/pixel_oracle.sfm_loss_pixel with the one-hot weights of that selection."""
import numpy as np

from oracle import sfm_oracle as O
from tests.pixel_oracle import sfm_loss_pixel, sfm_loss_pixel_raw


def errors(tgt, src, intrinsics, disps, poses, cfg):
    """-> (e, masked, e_id): per scale (B,S,h,w) float64 reprojection errors e_i, bool all-zero masks and float64
    identity errors, all without the 1/(B_global*3*h*w) factor:
      e    = (1 - r) * sum_c |P - T| + r * sum_c clip((1 - SSIM) / 2, 0, 1) * (1 - m)   (P the warped source)
      e_id = the same with P the source's own pyramid level and no mask
    (the SSIM parts only when SSIM runs)."""
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
        e = np.zeros((B, S, h, w))
        msk = np.zeros((B, S, h, w), bool)
        e_id = np.zeros((B, S, h, w))
        for i in range(S):
            img = cur_src[:, 3 * i:3 * i + 3]
            gr = O.cam2pixel(cam, O.proj_tgt_to_src(poses[:, i], K), h, w)
            P = O.spatial_transformer_sampler(img, gr['xn'], gr['yn'])[0].reshape(B, 3, h, w)
            m = np.all(P == 0, axis=1, keepdims=True)              # base_model.py:96
            for out, X, mm in ((e, P, m), (e_id, img, np.zeros_like(m))):
                err = np.where(mm, 0.0, np.abs(X - cur_tgt).astype(np.float64))
                v = (1 - r) * err.sum(1)
                if use_ssim:
                    v = v + r * (np.clip(O.ssim_terms(X, cur_tgt)['raw'], 0, 1) * (1 - mm)).astype(np.float64).sum(1)
                out[:, i] = v
            msk[:, i] = m[:, 0]
        out_e.append(e)
        out_m.append(msk)
        out_id.append(e_id)
    return out_e, out_m, out_id


def select(e, masked, e_id, automask):
    """Selection of one scale, (B,S,h,w) inputs -> (B,h,w) int8: -2 without a candidate (every source masked), else
    the argmin over the unmasked sources (ties to the lowest index), -1 when automask and e_i* >= min_i e_id_i."""
    E = np.where(masked, np.inf, e)
    best = E.min(1)
    sel = E.argmin(1).astype(np.int8)                  # np.argmin returns the first of equal minima
    sel = np.where(np.isinf(best), -2, sel)
    if automask:
        sel = np.where((sel >= 0) & (best >= e_id.min(1)), -1, sel)
    return sel.astype(np.int8)


def one_hot(sel, S, dtype):
    """(B,h,w) selection -> (B,S,h,w) weights [sel == i]."""
    return (sel[:, None] == np.arange(S)[None, :, None, None]).astype(dtype)


def sfm_loss_min_reprojection(tgt, src, intrinsics, disps, poses, cfg, automask=True, selection=None, want_grads=True,
                              want_intrinsics_grad=False, raw_disp_scales=0, raw_pose=False):
    """-> (losses dict with `selection` (list of (B,h,w) int8) and `pixel_losses`, grads dict or None).

    selection: None to compute it, or a given list of per-scale selections (the GPU's exported one: the loss and its
    gradients of that selection, free of near-tie decisions).  raw_disp_scales / raw_pose: inputs as
    oracle.sfm_loss_raw takes them."""
    S = src.shape[1]
    if selection is None:
        dd = [O.disp_activation(d)[0] if (raw_disp_scales >> s) & 1 else d for s, d in enumerate(disps)]
        pp = O.pose_from_raw(poses, S) if raw_pose else poses
        e, m, e_id = errors(tgt, src, intrinsics, dd, pp, cfg)
        selection = [select(e[s], m[s], e_id[s], automask) for s in range(cfg.n_scales)]
    W = [one_hot(sel, S, tgt.dtype) for sel in selection]
    kw = dict(pixel_weights=W, want_grads=want_grads, want_intrinsics_grad=want_intrinsics_grad)
    if raw_disp_scales or raw_pose:
        L, G = sfm_loss_pixel_raw(tgt, src, intrinsics, disps, poses, None, cfg, raw_disp_scales=raw_disp_scales,
                                  raw_pose=raw_pose, **kw)
    else:
        L, G = sfm_loss_pixel(tgt, src, intrinsics, disps, poses, None, cfg, **kw)
    L = dict(L, selection=selection)
    return L, G


def ambiguous(e, masked, e_id, automask, rel=1e-4):
    """(B,h,w) bool of one scale: the best candidate and the runner-up (the identity minimum included with automask) lie
    within a relative `rel` of each other, so fp32 rounding may decide the selection."""
    E = np.where(masked, np.inf, e)
    if automask:
        E = np.concatenate([E, e_id.min(1, keepdims=True)], 1)
    Es = np.sort(E, 1)
    v0, v1 = Es[:, 0], Es[:, 1] if Es.shape[1] > 1 else np.full_like(Es[:, 0], np.inf)
    with np.errstate(invalid='ignore'):
        return np.isfinite(v1) & (v1 - v0 <= rel * np.maximum(np.abs(v1), 1e-30))
