"""Reference of Monodepth2's axis-angle pose (SFM_FLAG_AXISANGLE_POSE, ViewSynthesisLoss(axisangle_pose=True)) in numpy.

The tables are built bit for bit as the prologue builds them: theta, the axis, sin / cos, R and the inverted -R^T t in
fp64 in the device's order (numpy rounds every operation and never contracts), R and t rounded to fp32 once, then
P = K . [R | t] in the oracle's canonical fp32 order.  The existing references take the tables through `proj_override`
and return dL/dT; `pose_grad` applies the axis-angle chain to it in fp64, and `intrinsics_grad_rt` forms the intrinsics
gradient with the transform's R and t."""
import numpy as np

from oracle import sfm_oracle as O
from tests.pixel_oracle import sfm_loss_pixel

EPS = 1e-7      # Monodepth2's layers.py rot_from_axisangle: axis = vec / (angle + 1e-7)


def invert_mask(invert_sources):
    m = 0
    for i in invert_sources:
        m |= 1 << i
    return m


def rot(v):
    """rot_from_axisangle in fp64, the device's order.  v (N,3) -> dict(th, a, c, s, R (N,3,3))."""
    v = v.astype(np.float64)
    v0, v1, v2 = v[:, 0], v[:, 1], v[:, 2]
    th = np.sqrt((v0 * v0 + v1 * v1) + v2 * v2)
    den = th + EPS
    x, y, z = v0 / den, v1 / den, v2 / den
    s, c = np.sin(th), np.cos(th)
    C = 1.0 - c
    xs, ys, zs = x * s, y * s, z * s
    xC, yC, zC = x * C, y * C, z * C
    xyC, yzC, zxC = x * yC, y * zC, z * xC
    R = np.stack([x * xC + c, xyC - zs, zxC + ys,
                  xyC + zs, y * yC + c, yzC - xs,
                  zxC - ys, yzC + xs, z * zC + c], 1).reshape(-1, 3, 3)
    return dict(th=th, a=np.stack([x, y, z], 1), c=c, s=s, R=R)


def transform(pose, inv):
    """-> (R, t) of the transform rounded to the pose's dtype (fp32: the device's tables): [R | t], or inverted
    [R^T | -R^T t].  pose (N,6), inv bool."""
    dt = pose.dtype
    q = rot(pose[:, :3])
    R = q['R']
    t = pose[:, 3:].astype(np.float64)
    if not inv:
        return R.astype(dt), pose[:, 3:].copy()
    m = (R[:, 0, :] * t[:, 0:1] + R[:, 1, :] * t[:, 1:2]) + R[:, 2, :] * t[:, 2:3]
    return np.swapaxes(R, 1, 2).astype(dt), (-m).astype(dt)


def tables(poses, intrinsics, invert_sources=()):
    """-> (proj (B,S,ns,3,4), kinv (B,ns,3,3)) in the poses' dtype; for fp32 as sfm_build_tables builds them with the
    flag.  The non-finite guard of the prologue is not restated (the tests use finite poses)."""
    B, S = poses.shape[:2]
    ns = intrinsics.shape[1]
    proj = np.zeros((B, S, ns, 3, 4), poses.dtype)
    for i in range(S):
        R, t = transform(poses[:, i], i in invert_sources)
        T = np.concatenate([R, t[:, :, None]], 2)
        for s in range(ns):
            proj[:, i, s] = O._mm(intrinsics[:, s].astype(poses.dtype), T)
    kinv = np.stack([O.batch_inv3(intrinsics[:, s]) for s in range(ns)], 1)
    return proj, kinv


def chain(pose, dT, inv):
    """dL/dpose (N,6) float64 from dL/dT (N,3,4) float64 through transformation_from_parameters (fp64, from the unrounded
    quantities), with torch's d theta / d v = 0 at theta = 0."""
    q = rot(pose[:, :3])
    R, a, c, s, th = q['R'], q['a'], q['c'][:, None, None], q['s'][:, None, None], q['th']
    t = pose[:, 3:].astype(np.float64)
    G3, g = dT[:, :, :3], dT[:, :, 3]
    if inv:
        GR = np.swapaxes(G3, 1, 2) - t[:, :, None] * g[:, None, :]
        gt = -np.einsum('nij,nj->ni', R, g)
    else:
        GR, gt = G3, g
    C = 1.0 - c[:, 0, 0]
    ga = C[:, None] * np.einsum('nkj,nj->nk', GR + np.swapaxes(GR, 1, 2), a)
    ga = ga + s[:, 0] * np.stack([GR[:, 2, 1] - GR[:, 1, 2], GR[:, 0, 2] - GR[:, 2, 0], GR[:, 1, 0] - GR[:, 0, 1]], 1)
    z = np.zeros_like(th)
    skew = np.stack([z, -a[:, 2], a[:, 1], a[:, 2], z, -a[:, 0], -a[:, 1], a[:, 0], z], 1).reshape(-1, 3, 3)
    dR = s * a[:, :, None] * a[:, None, :] + c * skew - s * np.eye(3)
    gth = np.sum(GR * dR, axis=(1, 2))
    v = pose[:, :3].astype(np.float64)
    den = th + EPS
    with np.errstate(divide='ignore', invalid='ignore'):
        k = np.where(th > 0, (gth - np.sum(ga * v, 1) / (den * den)) / th, 0.0)
    return np.concatenate([ga / den[:, None] + k[:, None] * v, gt], 1)


def pose_grad(poses, dT, invert_sources=()):
    """gposes (B,S,6) float64 from the references' dT (B,S,3,4)."""
    return np.stack([chain(poses[:, i], dT[:, i], i in invert_sources) for i in range(poses.shape[1])], 1)


def intrinsics_grad_rt(intrinsics, poses, dP, invert_sources=()):
    """oracle.intrinsics_grad with the R and t of the axis-angle transform (fp32-rounded, inverted per source)."""
    B, S, ns = dP.shape[:3]
    K = intrinsics.astype(np.float64)
    Ki = np.linalg.inv(K)
    out = np.zeros((B, ns, 3, 3), np.float64)
    for i in range(S):
        R, t = transform(poses[:, i], i in invert_sources)
        R = R.astype(np.float64)[:, None]
        t = t.astype(np.float64)[:, None]
        A, g = dP[:, i, :, :, :3], dP[:, i, :, :, 3]
        RT = np.swapaxes(R, -1, -2)
        out += A @ RT + g[..., :, None] * t[..., None, :]
        out -= np.swapaxes(Ki, -1, -2) @ RT @ np.swapaxes(K, -1, -2) @ A
    return out


def loss(tgt, src, intrinsics, disps, poses, cfg, invert_sources=(), pixel_weights=None, want_grads=True,
         want_intrinsics_grad=False, logits=None):
    """The per-pixel (weighted) reference with the axis-angle tables -> (losses, grads); grads hold gdisp, gpose (the
    axis-angle chain, float64) and with want_intrinsics_grad gintrinsics."""
    proj, kinv = tables(poses, intrinsics, invert_sources)
    L, G = sfm_loss_pixel(tgt, src, intrinsics, disps, poses, logits, cfg, pixel_weights=pixel_weights, want_grads=want_grads,
                          want_intrinsics_grad=want_intrinsics_grad, proj_override=proj, kinv_override=kinv)
    if G is not None:
        G = dict(G, gpose=pose_grad(poses, G['dT'], invert_sources))
        if want_intrinsics_grad:
            G['gintrinsics'] = intrinsics_grad_rt(intrinsics, poses, G['dP'], invert_sources)
    return L, G
