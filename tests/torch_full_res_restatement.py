"""An independent torch fp64 restatement of the full-resolution multi-scale loss (SFM_FLAG_FULL_RES_MULTISCALE), for
autograd checks of tests/full_res_oracle.py: the coarse disparities go through F.interpolate(align_corners=False), every
scale warps the full-resolution images with K_0 through torch.linalg.inv(K_0) and K_0 @ [R|t] with the x2 rule and
grid_sample, the minimum reprojection is torch.min over the stacked errors, and the smoothness terms stay at the native
resolution (the target pyramid through F.interpolate(align_corners=True))."""
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from tests.torch_restatement import _rot


def _pool(x):
    return F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)


def _ssim_err(x, t):
    a, my = _pool(x), _pool(t)
    sx, sy, sxy = _pool(x * x) - a * a, _pool(t * t) - my * my, _pool(x * t) - a * my
    n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
    dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
    return torch.clamp((1 - n / dd) / 2, 0, 1)


def _smooth(tgt, D, edge):
    """compute_smooth_loss / compute_disp_smooth (base_model.py:169-185 / 144-155) of one scale, unweighted."""
    if edge:
        img = tgt if tgt.shape[2:] == D.shape[2:] else F.interpolate(tgt, size=D.shape[2:], mode='bilinear',
                                                                     align_corners=True)
        d_dx, d_dy = D[..., 1:] - D[..., :-1], D[:, :, 1:] - D[:, :, :-1]
        i_dx = (img[..., 1:] - img[..., :-1]).mean(1, keepdim=True)
        i_dy = (img[:, :, 1:] - img[:, :, :-1]).mean(1, keepdim=True)
        return (d_dx.abs() * torch.exp(-i_dx.abs())).mean() + (d_dy.abs() * torch.exp(-i_dy.abs())).mean()
    dx, dy = D[..., 1:] - D[..., :-1], D[:, :, 1:] - D[:, :, :-1]
    terms = (dx[..., 1:] - dx[..., :-1], dx[:, :, 1:] - dx[:, :, :-1], dy[..., 1:] - dy[..., :-1], dy[:, :, 1:] - dy[:, :, :-1])
    return sum(t.abs().mean() for t in terms)


def torch_full_res(d, cfg, disps, poses, K, pixel_weights=None, min_reprojection=False, automask=True):
    """-> (total, pixel, ssim, smooth, selections) for the float64 snippets d with disps (list of (B,1,h_s,w_s)), poses
    (B,S,6) and K (B,n_scales,3,3) torch tensors (leaves or not).  pixel_weights: None or a list of (B,S,H,W) tensors or
    None entries.  selections: per scale (B,H,W) as include/sfmloss.h defines them (min_reprojection only)."""
    tgt, src = torch.from_numpy(d['tgt']), torch.from_numpy(d['src'])
    B, S, _, H, W = src.shape
    use_ssim = bool(cfg.ssim_rate)
    r = cfg.ssim_rate or 0.0
    K0 = K[:, 0]
    ys, xs = torch.meshgrid(torch.arange(H, dtype=K.dtype), torch.arange(W, dtype=K.dtype), indexing='ij')
    pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(H * W, dtype=K.dtype)])
    n3 = B * 3 * H * W
    pixel = ssim = 0.0
    sels = []
    for ns in range(cfg.n_scales):
        D = disps[ns] if ns == 0 else F.interpolate(disps[ns], size=(H, W), mode='bilinear', align_corners=False)
        cam = (1.0 / D.reshape(B, 1, H * W)) * (torch.linalg.inv(K0) @ pix)
        l1s, sss, errs, ids = [], [], [], []
        for i in range(S):
            pose = poses[:, i]
            P = K0 @ torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((W - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((H - 1) / 2.) - 1
            xn = torch.where((xn > -1) & (xn < 1), xn, 2 * xn)
            yn = torch.where((yn > -1) & (yn < 1), yn, 2 * yn)
            grid = torch.stack([xn, yn], -1).reshape(B, H, W, 2)
            img = src[:, i]
            Pw = F.grid_sample(img, grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            m = (Pw == 0).all(dim=1)
            l1 = torch.where(m, 0.0, (Pw - tgt).abs().sum(1))
            sm = torch.where(m, 0.0, _ssim_err(Pw, tgt).sum(1)) if use_ssim else torch.zeros_like(l1)
            if min_reprojection:
                errs.append(torch.where(m, float('inf'), (1 - r) * l1 + r * sm))
                l1s.append(l1)
                sss.append(sm)
                ids.append((1 - r) * (img - tgt).abs().sum(1) + (r * _ssim_err(img, tgt).sum(1) if use_ssim else 0.0))
            else:
                Mw = pixel_weights[ns][:, i] if pixel_weights is not None and pixel_weights[ns] is not None else 1.0
                pixel = pixel + (l1 * Mw).sum() / n3
                ssim = ssim + (sm * Mw).sum() / n3
        if min_reprojection:
            best, idx = torch.min(torch.stack(errs, 1), 1)          # the first of equal minima
            keep = torch.isfinite(best)
            sel = torch.where(keep, idx, -2)
            if automask:
                am = keep & (best >= torch.stack(ids, 1).min(1).values)
                sel = torch.where(am, -1, sel)
                keep = keep & ~am
            pick = lambda terms: torch.gather(torch.stack(terms, 1), 1, idx[:, None])[:, 0]
            pixel = pixel + torch.where(keep, pick(l1s), 0.0).sum() / n3
            ssim = ssim + torch.where(keep, pick(sss), 0.0).sum() / n3
            sels.append(sel)
    smooth = 0.0
    if cfg.smooth_reg:
        for ns in range(cfg.n_scales):
            smooth = smooth + cfg.smooth_reg / 2 ** ns * _smooth(tgt, disps[ns], cfg.edge_aware_smooth)
    total = (1 - r) * pixel + r * ssim + smooth
    return total, pixel, ssim, smooth, sels
