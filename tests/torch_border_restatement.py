"""An independent torch fp64 restatement of Monodepth2's photometric loss at the image borders (SFM_FLAG_BORDER_PADDING),
for autograd checks of tests/pixel_oracle.py with border=True: the warp is Monodepth2's
F.grid_sample(padding_mode="border", align_corners=True) on the grid without the x2 rule (the 1e-10 of the library's
projection kept), its SSIM module (reflection padding + 3x3 average pool), and compute_reprojection_loss with torch.min
over the sources and the identity errors.  There is no mask: the inputs have no degenerate projection."""
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from tests.torch_restatement import _rot


def _ssim_err(x, y):
    """Monodepth2's SSIM module: clamp((1 - SSIM_n / SSIM_d) / 2, 0, 1) on ReflectionPad2d(1) + AvgPool2d(3, 1)."""
    x, y = F.pad(x, (1, 1, 1, 1), mode='reflect'), F.pad(y, (1, 1, 1, 1), mode='reflect')
    mu_x, mu_y = F.avg_pool2d(x, 3, 1), F.avg_pool2d(y, 3, 1)
    sigma_x = F.avg_pool2d(x ** 2, 3, 1) - mu_x ** 2
    sigma_y = F.avg_pool2d(y ** 2, 3, 1) - mu_y ** 2
    sigma_xy = F.avg_pool2d(x * y, 3, 1) - mu_x * mu_y
    n = (2 * mu_x * mu_y + O.SSIM_C1) * (2 * sigma_xy + O.SSIM_C2)
    d = (mu_x ** 2 + mu_y ** 2 + O.SSIM_C1) * (sigma_x + sigma_y + O.SSIM_C2)
    return torch.clamp((1 - n / d) / 2, 0, 1)


def torch_border(d, cfg, disps, poses, min_reprojection=False, automask=True, full_res=False):
    """-> (photometric, pixel, ssim, selections) for the float64 snippets d with disps (list of (B,1,h_s,w_s)) and poses
    (B,S,6) torch tensors (leaves or not).  photometric = (1 - r) pixel + r ssim summed over the scales, each a mean over
    B*3*h*w; with min_reprojection the per-pixel minimum of Monodepth2's compute_reprojection_loss (0 where auto-masked),
    and the selections (B,h,w) as include/sfmloss.h defines them.  full_res: Monodepth2's upsampled multi-scale (every
    disparity upsampled with align_corners=False, warped with K_0 against the full-resolution images)."""
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
            pose = poses[:, i]
            P = Ks @ torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)
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
