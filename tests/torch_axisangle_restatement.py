"""Monodepth2's pose functions (layers.py: rot_from_axisangle, get_translation_matrix, transformation_from_parameters)
copied literally, for torch fp64 autograd checks of tests/axisangle_oracle.py and the device, and the photometric
restatements of tests/torch_restatement.py and tests/torch_border_restatement.py with that transform."""
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from tests.torch_border_restatement import _ssim_err


def rot_from_axisangle(vec):
    """Convert an axisangle rotation into a 4x4 transformation matrix
    (adapted from https://github.com/Wallacoloo/printipi)
    Input 'vec' has to be Bx1x3
    """
    angle = torch.norm(vec, 2, 2, True)
    axis = vec / (angle + 1e-7)

    ca = torch.cos(angle)
    sa = torch.sin(angle)
    C = 1 - ca

    x = axis[..., 0].unsqueeze(1)
    y = axis[..., 1].unsqueeze(1)
    z = axis[..., 2].unsqueeze(1)

    xs = x * sa
    ys = y * sa
    zs = z * sa
    xC = x * C
    yC = y * C
    zC = z * C
    xyC = x * yC
    yzC = y * zC
    zxC = z * xC

    rot = torch.zeros((vec.shape[0], 4, 4), dtype=vec.dtype).to(device=vec.device)

    rot[:, 0, 0] = torch.squeeze(x * xC + ca)
    rot[:, 0, 1] = torch.squeeze(xyC - zs)
    rot[:, 0, 2] = torch.squeeze(zxC + ys)
    rot[:, 1, 0] = torch.squeeze(xyC + zs)
    rot[:, 1, 1] = torch.squeeze(y * yC + ca)
    rot[:, 1, 2] = torch.squeeze(yzC - xs)
    rot[:, 2, 0] = torch.squeeze(zxC - ys)
    rot[:, 2, 1] = torch.squeeze(yzC + xs)
    rot[:, 2, 2] = torch.squeeze(z * zC + ca)
    rot[:, 3, 3] = 1

    return rot


def get_translation_matrix(translation_vector):
    """Convert a translation vector into a 4x4 transformation matrix
    """
    T = torch.zeros(translation_vector.shape[0], 4, 4, dtype=translation_vector.dtype).to(device=translation_vector.device)

    t = translation_vector.contiguous().view(-1, 3, 1)

    T[:, 0, 0] = 1
    T[:, 1, 1] = 1
    T[:, 2, 2] = 1
    T[:, 3, 3] = 1
    T[:, :3, 3, None] = t

    return T


def transformation_from_parameters(axisangle, translation, invert=False):
    """Convert the network's (axisangle, translation) output into a 4x4 matrix
    """
    R = rot_from_axisangle(axisangle)
    t = translation.clone()

    if invert:
        R = R.transpose(1, 2)
        t *= -1

    T = get_translation_matrix(t)

    if invert:
        M = torch.matmul(R, T)
    else:
        M = torch.matmul(T, R)

    return M


def transform_rows(pose, invert=False):
    """(N,6) pose rows (v, t) -> the (N,3,4) transform [R | t] Monodepth2 builds from them (its axisangle / translation
    tensors are (N,1,1,3); dtype kept)."""
    M = transformation_from_parameters(pose[:, None, :3], pose[:, None, 3:], invert)
    return M[:, :3, :]


# ---- whole-loss restatements with Monodepth2's transform in place of the Euler [R | t].  They repeat the photometric
# loops of tests/torch_restatement.torch_total and tests/torch_border_restatement.torch_border line for line; only the
# transform of source i, transform_rows(pose, i in invert_sources), differs.

def torch_total_axisangle(d, cfg, tgt, src, K, invert_sources=()):
    """torch_total (the reference's photometric terms, any of tgt / src / K a leaf) with the axis-angle transform."""
    B, S, _, H, W = src.shape
    use_exp = bool(cfg.exp_reg)
    use_ssim = not use_exp and bool(cfg.ssim_rate)
    rate = cfg.ssim_rate or 0.0
    pixel = ssim = 0.0
    for ns in range(cfg.n_scales):
        h, w = H >> ns, W >> ns
        ct = F.interpolate(tgt, size=(h, w), mode='bilinear', align_corners=True)
        cs = F.interpolate(src.reshape(B, 3 * S, H, W), size=(h, w), mode='bilinear', align_corners=True)
        depth = 1.0 / torch.from_numpy(d['disps'][ns]).reshape(B, 1, h * w)
        ys, xs = torch.meshgrid(torch.arange(h, dtype=K.dtype), torch.arange(w, dtype=K.dtype), indexing='ij')
        pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(h * w, dtype=K.dtype)])
        Ks = K[:, ns]
        cam = depth * (torch.linalg.inv(Ks) @ pix)
        n3 = B * 3 * h * w
        for i in range(S):
            P = Ks @ transform_rows(torch.from_numpy(d['poses'][:, i]), i in invert_sources)
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((w - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((h - 1) / 2.) - 1
            inx = ((xn > -1) & (xn < 1)).detach()
            iny = ((yn > -1) & (yn < 1)).detach()
            xn = torch.where(inx, xn, 2 * xn)
            yn = torch.where(iny, yn, 2 * yn)
            grid = torch.stack([xn, yn], -1).reshape(B, h, w, 2)
            Pw = F.grid_sample(cs[:, 3 * i:3 * i + 3], grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            m = (Pw == 0).all(dim=1, keepdim=True).detach()
            err = torch.where(m, torch.zeros_like(Pw), (Pw - ct).abs())
            if use_exp:
                sg = torch.sigmoid(torch.from_numpy(d['logits'][ns][:, i:i + 1]))
                pixel = pixel + (err * sg).sum() / n3
            else:
                pixel = pixel + err.sum() / n3
            if use_ssim:
                pool = lambda x: F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)
                a, my = pool(Pw), pool(ct)
                sx, sy, sxy = pool(Pw * Pw) - a * a, pool(ct * ct) - my * my, pool(Pw * ct) - a * my
                n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
                dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
                e = torch.clamp((1 - n / dd) / 2, 0, 1) * (~m)
                ssim = ssim + e.sum() / n3
    return (1 - rate) * pixel + rate * ssim


def torch_border_axisangle(d, cfg, disps, poses, invert_sources=(), min_reprojection=False, automask=True, full_res=False):
    """torch_border (Monodepth2's photometric loss at the image borders, poses a leaf or not) with the axis-angle
    transform -> (photometric, pixel, ssim, selections)."""
    tgt, src, K = (torch.from_numpy(d[k]) for k in ('tgt', 'src', 'intrinsics'))
    B, S, _, H, W = src.shape
    use_ssim = bool(cfg.ssim_rate)
    r = cfg.ssim_rate or 0.0
    pixel = ssim = 0.0
    sels = []
    for ns in range(cfg.n_scales):
        if full_res:
            h, w, Ks = H, W, K[:, 0]
            ct, cs = tgt, src.reshape(B, 3 * S, H, W)
            D = disps[ns] if ns == 0 else F.interpolate(disps[ns], size=(H, W), mode='bilinear', align_corners=False)
        else:
            h, w, Ks = H >> ns, W >> ns, K[:, ns]
            ct = F.interpolate(tgt, size=(h, w), mode='bilinear', align_corners=True)
            cs = F.interpolate(src.reshape(B, 3 * S, H, W), size=(h, w), mode='bilinear', align_corners=True)
            D = disps[ns]
        ys, xs = torch.meshgrid(torch.arange(h, dtype=K.dtype), torch.arange(w, dtype=K.dtype), indexing='ij')
        pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(h * w, dtype=K.dtype)])
        cam = (1.0 / D.reshape(B, 1, h * w)) * (torch.linalg.inv(Ks) @ pix)
        l1s, sss, ids = [], [], []
        for i in range(S):
            P = Ks @ transform_rows(poses[:, i], i in invert_sources)
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((w - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((h - 1) / 2.) - 1
            grid = torch.stack([xn, yn], -1).reshape(B, h, w, 2)
            img = cs[:, 3 * i:3 * i + 3]
            Pw = F.grid_sample(img, grid, mode='bilinear', padding_mode='border', align_corners=True)
            l1s.append((Pw - ct).abs().sum(1))
            sss.append(_ssim_err(Pw, ct).sum(1) if use_ssim else torch.zeros_like(l1s[-1]))
            if min_reprojection and automask:
                ids.append((1 - r) * (img - ct).abs().sum(1) + (r * _ssim_err(img, ct).sum(1) if use_ssim else 0.0))
        n3 = B * 3 * h * w
        if min_reprojection:
            best, idx = torch.min(torch.stack([(1 - r) * a + r * b for a, b in zip(l1s, sss)], 1), 1)
            keep = torch.ones_like(best, dtype=torch.bool)
            sel = idx
            if automask:
                am = best >= torch.stack(ids, 1).min(1).values
                sel = torch.where(am, -1, sel)
                keep = ~am
            pick = lambda terms: torch.gather(torch.stack(terms, 1), 1, idx[:, None])[:, 0]
            pixel = pixel + torch.where(keep, pick(l1s), 0.0).sum() / n3
            ssim = ssim + torch.where(keep, pick(sss), 0.0).sum() / n3
            sels.append(sel)
        else:
            pixel = pixel + sum(a.sum() for a in l1s) / n3
            ssim = ssim + sum(b.sum() for b in sss) / n3
    return (1 - r) * pixel + r * ssim, pixel, ssim, sels
