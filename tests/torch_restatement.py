"""An independent torch fp64 restatement of the image- and K-dependent part of the loss, for autograd checks of the
oracle's opt-in gradients (image gradients, intrinsics gradient)."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O


def _rot(a):
    """(Rx . Ry) . Rz of the clipped angles a (N,3) (transform.py:11-40)."""
    a = torch.clamp(a, -np.pi, np.pi)
    c, s = torch.cos(a), torch.sin(a)
    o, z = torch.ones_like(c[:, 0]), torch.zeros_like(c[:, 0])
    rx = torch.stack([o, z, z, z, c[:, 0], -s[:, 0], z, s[:, 0], c[:, 0]], 1).reshape(-1, 3, 3)
    ry = torch.stack([c[:, 1], z, s[:, 1], z, o, z, -s[:, 1], z, c[:, 1]], 1).reshape(-1, 3, 3)
    rz = torch.stack([c[:, 2], -s[:, 2], z, s[:, 2], c[:, 2], z, z, z, o], 1).reshape(-1, 3, 3)
    return (rx @ ry) @ rz


def torch_total(d, cfg, tgt, src, K):
    """(1 - r) * pixel + r * ssim of base_model.py:64-118 for the snippets d (float64) with tgt (B,3,H,W),
    src (B,S,3,H,W) and K (B,ns,3,3) as torch tensors, any of them a leaf: the pyramid through F.interpolate, the grid
    through torch.linalg.inv(K) and K @ [R|t] with the x2 rule, grid_sample.  The terms that depend on none of them
    (smoothness, explainability regulariser) are left out."""
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
        cam = depth * (torch.linalg.inv(Ks) @ pix)                                   # pixel2cam (transform.py:94-109)
        n3 = B * 3 * h * w
        for i in range(S):
            pose = torch.from_numpy(d['poses'][:, i])
            P = Ks @ torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)           # K4 . [R|t] (transform.py:86-88)
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
