"""TEST INFRASTRUCTURE: the numpy oracle's counterpart of the intrinsics gradient of the fused loss.

d total / d intrinsics of SFMLearner.__call__'s loss loop (base_model.py:57-124), K_s = intrinsics[:, s] treated as
differentiable in both places the reference uses it: the projection P = K4 . [R|t] (transform.py:86-88) and pixel2cam's
batch_inv(K) (:105).  Per pixel q = K (R c + t) with c = depth K^-1 pix, so with the per-(source, scale) cells
dL/dP = [A_i | g_i] (A_i = sum gq (x) c, g_i = sum gq):

    dL/dK_s = sum_i [ A_i R_i^T + g_i t_i^T - K_s^-T R_i^T K_s^T A_i ]

The cells are the ones oracle/sfm_oracle.py itself computes (`dP_all`): they are taken where sfm_loss hands them to its
pose chain (`_pose_backward`), so the numpy oracle runs unchanged.  R_i = (Rx . Ry) . Rz of the clipped angles with
sin / cos rounded to the working dtype and t_i unclipped, as `_pose_backward` has them; K^-1 and the sum in float64.
"""
import numpy as np

from oracle import sfm_oracle as O


def _with_cells(fn, *args, **kw):
    """fn(*args, **kw) (O.sfm_loss or O.sfm_loss_raw) -> (losses, grads with 'dP' (B,S,n_scales,3,4) float64, debug)."""
    cells = []
    pose_backward = O._pose_backward

    def record(vec, K_scales, dP_scales):
        cells.append(np.stack(dP_scales, 1))
        return pose_backward(vec, K_scales, dP_scales)

    O._pose_backward = record
    try:
        L, G, dbg = fn(*args, **kw)
    finally:
        O._pose_backward = pose_backward
    G = dict(G)
    G['dP'] = np.stack(cells, 1)                # sfm_loss chains the sources in order 0 .. S-1
    return L, G, dbg


def intrinsics_grad(intrinsics, poses, dP):
    """-> gintrinsics (B,n_scales,3,3) float64.  intrinsics (B,n_scales,3,3), poses (B,S,6) as the loss used them (the
    reduced vectors under raw_pose), dP (B,S,n_scales,3,4)."""
    B, S, ns = dP.shape[:3]
    K = intrinsics.astype(np.float64)
    Ki = np.linalg.inv(K)
    out = np.zeros((B, ns, 3, 3), np.float64)
    for i in range(S):
        _, c, s = O.euler_sincos(poses[:, i, :3])
        xm, ym, zm = [m.astype(np.float64) for m in O._rot_mats(c, s)]
        R = ((xm @ ym) @ zm)[:, None]                                    # (B,1,3,3)
        t = poses[:, i, 3:].astype(np.float64)[:, None]                  # (B,1,3)
        A, g = dP[:, i, :, :, :3], dP[:, i, :, :, 3]
        RT = np.swapaxes(R, -1, -2)
        out += A @ RT + g[..., :, None] * t[..., None, :]
        out -= np.swapaxes(Ki, -1, -2) @ RT @ np.swapaxes(K, -1, -2) @ A
    return out


def sfm_loss_with_intrinsics_grad(tgt, src, intrinsics, disps, poses, logits, cfg, **kw):
    """O.sfm_loss, its grads dict completed with 'dP' and 'gintrinsics'."""
    L, G, dbg = _with_cells(O.sfm_loss, tgt, src, intrinsics, disps, poses, logits, cfg, **kw)
    G['gintrinsics'] = intrinsics_grad(intrinsics, poses, G['dP'])
    return L, G, dbg


def sfm_loss_raw_with_intrinsics_grad(tgt, src, intrinsics, disps_in, poses_in, logits, cfg, **kw):
    """O.sfm_loss_raw, its grads dict completed with 'dP' and 'gintrinsics' (R, t from the reduced poses)."""
    L, G, dbg = _with_cells(O.sfm_loss_raw, tgt, src, intrinsics, disps_in, poses_in, logits, cfg, **kw)
    G['gintrinsics'] = intrinsics_grad(intrinsics, dbg['poses'], G['dP'])
    return L, G, dbg
