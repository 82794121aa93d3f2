"""An independent torch fp64 restatement of the photometric loss with per-pixel minimum reprojection and auto-masking,
for autograd checks of tests/min_reprojection_oracle.py: the per-source errors are stacked with +inf where the source is
masked, compared with the identity errors and reduced with torch.min, whose gradient is autograd's one-hot."""
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from tests.torch_restatement import _rot


def _pool(x):
    return F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)


def _ssim_err(x, t):
    """clip((1 - SSIM) / 2, 0, 1) per channel (base_model.py:126-142)."""
    a, my = _pool(x), _pool(t)
    sx, sy, sxy = _pool(x * x) - a * a, _pool(t * t) - my * my, _pool(x * t) - a * my
    n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
    dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
    return torch.clamp((1 - n / dd) / 2, 0, 1)


def torch_min_reprojection(d, cfg, disps, poses, automask=True):
    """-> (photometric, pixel, ssim, selections) for the float64 snippets d with disps (list of (B,1,h,w)) and poses
    (B,S,6) torch tensors (leaves or not).  photometric = sum over the scales of the mean over B*3*h*w of the per-pixel
    minimum (0 where auto-masked or without a candidate), differentiable through torch.min; pixel and ssim are the L1
    and SSIM parts of the chosen terms (as losses_out[1] and [4]); the per-scale selections (B,h,w) are as
    include/sfmloss.h defines them.  The pyramid goes through F.interpolate, the grid through torch.linalg.inv(K) and
    K @ [R|t] with the x2 rule, grid_sample."""
    tgt, src, K = (torch.from_numpy(d[k]) for k in ('tgt', 'src', 'intrinsics'))
    B, S, _, H, W = src.shape
    use_ssim = bool(cfg.ssim_rate)
    r = cfg.ssim_rate or 0.0
    phot = pixel = ssim = 0.0
    sels = []
    for ns in range(cfg.n_scales):
        h, w = H >> ns, W >> ns
        ct = F.interpolate(tgt, size=(h, w), mode='bilinear', align_corners=True)
        cs = F.interpolate(src.reshape(B, 3 * S, H, W), size=(h, w), mode='bilinear', align_corners=True)
        depth = 1.0 / disps[ns].reshape(B, 1, h * w)
        ys, xs = torch.meshgrid(torch.arange(h, dtype=K.dtype), torch.arange(w, dtype=K.dtype), indexing='ij')
        pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(h * w, dtype=K.dtype)])
        Ks = K[:, ns]
        cam = depth * (torch.linalg.inv(Ks) @ pix)
        l1s, sss, errs, ids = [], [], [], []
        for i in range(S):
            pose = poses[:, i]
            P = Ks @ torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((w - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((h - 1) / 2.) - 1
            xn = torch.where((xn > -1) & (xn < 1), xn, 2 * xn)
            yn = torch.where((yn > -1) & (yn < 1), yn, 2 * yn)
            grid = torch.stack([xn, yn], -1).reshape(B, h, w, 2)
            img = cs[:, 3 * i:3 * i + 3]
            Pw = F.grid_sample(img, grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            m = (Pw == 0).all(dim=1)
            l1 = (Pw - ct).abs().sum(1)
            sm = _ssim_err(Pw, ct).sum(1) if use_ssim else torch.zeros_like(l1)
            e = (1 - r) * l1 + r * sm
            errs.append(torch.where(m, torch.full_like(e, float('inf')), e))
            l1s.append(l1)
            sss.append(sm)
            if automask:
                ids.append((1 - r) * (img - ct).abs().sum(1) + (r * _ssim_err(img, ct).sum(1) if use_ssim else 0.0))
        E = torch.stack(errs, 1)
        best, idx = torch.min(E, 1)                     # the first of equal minima
        keep = torch.isfinite(best)
        sel = torch.where(keep, idx, torch.full_like(idx, -2))
        if automask:
            idmin = torch.stack(ids, 1).min(1).values
            am = keep & (best >= idmin)
            sel = torch.where(am, torch.full_like(idx, -1), sel)
            keep = keep & ~am
        n3 = B * 3 * h * w
        pick = lambda terms: torch.gather(torch.stack(terms, 1), 1, idx[:, None])[:, 0]
        phot = phot + torch.where(keep, best, torch.zeros_like(best)).sum() / n3
        pixel = pixel + torch.where(keep, pick(l1s), torch.zeros_like(best)).sum() / n3
        ssim = ssim + torch.where(keep, pick(sss), torch.zeros_like(best)).sum() / n3
        sels.append(sel)
    return phot, pixel, ssim, sels
