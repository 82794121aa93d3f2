"""Reference of sfm_loss_geometry (SC-SfMLearner's geometry consistency term and self-discovered mask), in numpy on the
oracle's helpers and the per-pixel reference (tests/pixel_oracle.py).

Per scale s and source i: the target pixel is projected with the oracle's cam2pixel (the fp32 chain the device repeats
bit for bit), z' = q2 (before the 1e-10), D' is the oracle's bilinear sampler applied to 1 / src_disp (fp32, the same
blend order), D_diff = clip(|z' - D'| / (z' + D'), 0, 1) on the strictly in-view pairs and 0 elsewhere.  The photometric
terms are those of sfm_loss_pixel with the weights M = 1 - D_diff (self-mask) or none; the upstream of D_diff is
geometry_reg / (B_global h w) - map (the map only under the self-mask), chained in fp64 through z' and D' into the
target's disparity, the dL/dP cells (hence the pose and intrinsics gradients) and the source disparity."""
import numpy as np

from oracle import sfm_oracle as O
from tests import axisangle_oracle as AA
from tests.pixel_oracle import sfm_loss_pixel


def geometry_terms(intrinsics, disps, poses, src_disps, cfg, proj_override=None, kinv_override=None):
    """-> list over scales of dicts (per source lists): diff (B,h,w) fp32 and the records of the chain."""
    B, S = poses.shape[:2]
    dt = disps[0].dtype
    out = []
    for ns in range(cfg.n_scales):
        B_, _, h, w = disps[ns].shape
        hw_n = h * w
        depth = dt.type(1) / disps[ns].reshape(B, hw_n)
        K = intrinsics[:, ns]
        Kinv = kinv_override[:, ns] if kinv_override is not None else O.batch_inv3(K)
        ray, cam = O.pixel2cam(depth, Kinv, h, w)
        per = []
        for i in range(S):
            proj = proj_override[:, i, ns] if proj_override is not None else O.proj_tgt_to_src(poses[:, i], K)
            gr = O.cam2pixel(cam, proj, h, w)
            inb = gr['inx'] & gr['iny']
            inv = (dt.type(1) / src_disps[ns][:, i]).reshape(B, 1, h, w)
            Dp, t = O.spatial_transformer_sampler(inv, gr['xn'], gr['yn'])
            Dp = Dp[:, 0]
            zq = gr['q'][:, 2]
            with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
                a = zq - Dp
                c = zq + Dp
                ratio = np.abs(a) / c
            diff = np.where(inb, np.clip(ratio, 0, 1), dt.type(0)).astype(dt)
            per.append(dict(diff=diff, inb=inb, a=a, c=c, ratio=ratio, gr=gr, t=t, proj=proj, inv=inv[:, 0].reshape(B, hw_n)))
        out.append(dict(per=per, ray=ray, cam=cam, depth=depth, h=h, w=w))
    return out


def loss(tgt, src, intrinsics, disps, poses, src_disps, cfg, geometry_reg=0.5, self_mask=True, want_grads=True,
         want_intrinsics_grad=False, proj_override=None, kinv_override=None, invert_sources=None):
    """-> (losses dict (with `geometry_diff`, the D_diff maps (B,S,h,w) per scale), grads dict or None).

    grads: gdisp, gpose (float64 for the axis-angle pose), gsrc_disp (float64), dT; with want_intrinsics_grad dP and
    gintrinsics.  invert_sources not None: the axis-angle pose with those sources inverted (the device's tables)."""
    if invert_sources is not None:
        proj_override, kinv_override = AA.tables(poses, intrinsics, invert_sources)
    B, S = poses.shape[:2]
    Bg = cfg.B_global if cfg.B_global else B
    terms = geometry_terms(intrinsics, disps, poses, src_disps, cfg, proj_override, kinv_override)
    diffs = [np.stack([terms[s]['per'][i]['diff'].reshape(B, terms[s]['h'], terms[s]['w']) for i in range(S)], 1)
             for s in range(cfg.n_scales)]
    W = [(d.dtype.type(1) - d).astype(d.dtype) for d in diffs] if self_mask else None
    L, G = sfm_loss_pixel(tgt, src, intrinsics, disps, poses, None, cfg, pixel_weights=W, want_grads=want_grads,
                          want_intrinsics_grad=want_grads, proj_override=proj_override, kinv_override=kinv_override)
    geo = 0.0
    for s in range(cfg.n_scales):
        geo += geometry_reg * O._fsum(diffs[s]) / (Bg * terms[s]['h'] * terms[s]['w'])
    maps = L['pixel_losses']
    L = dict(L, exp_loss=geo, total_loss=L['total_loss'] + geo, geometry_diff=diffs)
    if not want_grads:
        return L, None
    gdisp = [g.astype(np.float64) for g in G['gdisp']]
    dP = G['dP'].copy()                       # (B,S,ns,3,4)
    gsrc = [np.zeros(x.shape, np.float64) for x in src_disps]
    for s in range(cfg.n_scales):
        T = terms[s]
        h, w = T['h'], T['w']
        hw_n = h * w
        g_depth = np.zeros((B, hw_n))
        for i in range(S):
            r = T['per'][i]
            up = np.full((B, hw_n), geometry_reg / (Bg * h * w))
            if self_mask:
                up = up - maps[s][:, i].reshape(B, hw_n)
            ratio = r['ratio'].astype(np.float64)
            ok = r['inb'] & (ratio >= 0) & (ratio <= 1)
            a, c = r['a'].astype(np.float64), r['c'].astype(np.float64)
            with np.errstate(divide='ignore', invalid='ignore'):
                gz = np.where(ok, up * (np.sign(a) - ratio) / c, 0.0)
                gD = np.where(ok, up * (-np.sign(a) - ratio) / c, 0.0)
            t64 = {k: (v.astype(np.float64) if v.dtype.kind == 'f' else v) for k, v in r['t'].items()}
            g_xn, g_yn = O.spatial_transformer_sampler_grad(t64, gD[:, None, :], h, w)
            gr = r['gr']
            q = gr['q'].astype(np.float64)
            z = gr['z'].astype(np.float64)
            hw_, hh_ = float(gr['hw']), float(gr['hh'])
            with np.errstate(divide='ignore', invalid='ignore'):
                g_q0 = np.where(ok, g_xn / (z * hw_), 0.0)
                g_q1 = np.where(ok, g_yn / (z * hh_), 0.0)
                g_q2 = np.where(ok, gz - (g_xn * q[:, 0] / hw_ + g_yn * q[:, 1] / hh_) / (z * z), 0.0)
            g_q = np.stack([g_q0, g_q1, g_q2], axis=1)
            P64 = r['proj'].astype(np.float64)
            g_cam = np.einsum('nkp,nkj->njp', g_q, P64[:, :3, :3])
            g_depth += np.sum(g_cam * T['ray'].astype(np.float64), axis=1)
            cam4 = np.concatenate([T['cam'].astype(np.float64), np.ones((B, 1, hw_n))], axis=1)
            dP[:, i, s] += np.einsum('nkp,njp->nkj', g_q, cam4)
            # D' = sum_k w_k / d'_k  =>  d / d d'_k = -gD w_k / d'_k^2, scattered to the taps
            inv = r['inv'].astype(np.float64)
            bb = np.repeat(np.arange(B), hw_n)
            u0, v0 = t64['u0'].reshape(-1), t64['v0'].reshape(-1)
            okf = ok.reshape(-1)
            wa, wb, wc, wd = (t64[k].reshape(-1) for k in ('wa', 'wb', 'wc', 'wd'))
            gDf = gD.reshape(-1)
            plane = gsrc[s][:, i]
            inv_img = (1.0 / src_disps[s][:, i].astype(np.float64))
            for wk, dv, du in ((wa * wc, 0, 0), (wb * wc, 0, 1), (wa * wd, 1, 0), (wb * wd, 1, 1)):
                vv = np.clip(v0 + dv, 0, h - 1)
                uu = np.clip(u0 + du, 0, w - 1)
                val = np.where(okf, -gDf * wk * inv_img[bb, vv, uu] ** 2, 0.0)
                np.add.at(plane, (bb, vv, uu), val)
            del inv
        d64 = disps[s].reshape(B, hw_n).astype(np.float64)
        gdisp[s] += (-g_depth / (d64 * d64)).reshape(disps[s].shape)
    dT = np.zeros((B, S, 3, 4))
    K_scales = [intrinsics[:, s] for s in range(cfg.n_scales)]
    gpose = np.zeros((B, S, 6))
    for i in range(S):
        dPi = [dP[:, i, s] for s in range(cfg.n_scales)]
        gpose[:, i], dT[:, i] = O._pose_backward(poses[:, i], K_scales, dPi)
    if invert_sources is not None:
        gpose = AA.pose_grad(poses, dT, invert_sources)
    grads = dict(gdisp=gdisp, gpose=gpose, gsrc_disp=gsrc, dT=dT)
    if want_intrinsics_grad:
        grads['dP'] = dP
        grads['gintrinsics'] = (AA.intrinsics_grad_rt(intrinsics, poses, dP, invert_sources) if invert_sources is not None
                                else O.intrinsics_grad(intrinsics, poses, dP))
    return L, grads


def loss_raw(tgt, src, intrinsics, disps_in, poses_in, src_disps, cfg, raw_disp_scales=0, raw_pose=False, **kw):
    """loss() with the seam included: the scales of raw_disp_scales take DispNet's pre-activation map for the target,
    raw_pose PoseNet's poseout map; the gradients are w.r.t. what was passed in (src_disps stay activated)."""
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
    L, G = loss(tgt, src, intrinsics, disps, poses, src_disps, cfg, **kw)
    if G is not None:
        G = dict(G)
        G['gdisp'] = [g if da is None else g * da.astype(np.float64) for g, da in zip(G['gdisp'], dacts)]
        if raw_pose:
            n = int(np.prod(poses_in.shape[2:]))
            gp = G['gpose'].reshape(poses_in.shape[0], 6 * S, *([1] * (poses_in.ndim - 2)))
            G['gpose'] = np.broadcast_to(gp * (0.01 / n), poses_in.shape).copy()
    return L, G


def make_src_disps(B, S, H, W, n_scales, seed, scale=1.0):
    """Smooth positive disparities (B,S,h_s,w_s) of the source frames, DispNet's range (0.01 .. 10.01)."""
    rs = np.random.RandomState(seed)
    out = []
    for s in range(n_scales):
        h, w = H >> s, W >> s
        lo = rs.standard_normal((B, S, max(h // 8, 2), max(w // 8, 2)))
        yi = np.minimum((np.arange(h) * lo.shape[2]) // h, lo.shape[2] - 1)
        xi = np.minimum((np.arange(w) * lo.shape[3]) // w, lo.shape[3] - 1)
        x = lo[:, :, yi][:, :, :, xi] + 0.05 * rs.standard_normal((B, S, h, w))
        out.append(np.ascontiguousarray(scale * (10.0 / (1.0 + np.exp(-x)) + 0.01), np.float32))
    return out
