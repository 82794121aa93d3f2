"""SC-SfMLearner's compute_pairwise_loss and mean_on_mask (Bian et al., NeurIPS 2019, released code) written literally in
torch fp64, on the library's warp (the x2 rule, zero padding, align-corners; validity = the strict in-view flag), as
sfm_loss_geometry_valid_mean defines them:
    diff_img   = (tgt - warped).abs().clamp(0, 1)
    diff_depth = ((z' - D').abs() / (z' + D')).clamp(0, 1)
    auto_mask  = (diff_img.mean(1) < (tgt - ref).abs().mean(1)) * valid           (with_auto_mask)
    loss       = mean_on_mask(((1 - r) diff_img + r ssim) * (1 - diff_depth), auto_mask)
               + geometry_reg * mean_on_mask(diff_depth, auto_mask)
    mean_on_mask(diff, mask) = (diff * mask).sum() / mask.sum() over the channels of diff, 0 unless mask.sum() > min_count
The counts are taken per (scale, source, group of snippets b mod G).  The mask is a step function of the inputs, so it
carries no gradient; autograd gives the reference gradients of everything else.  The smoothness term is left out."""
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from tests.torch_restatement import _rot


def mean_on_mask(diff, mask, min_count):
    m = mask.expand_as(diff)
    n = m.sum()
    return (diff * m).sum() / n if float(n) > min_count else diff.sum() * 0.0


def torch_total_valid_mean(tgt, src, K, disps, poses, src_disps, cfg, geometry_reg, self_mask, automask, groups=1,
                           min_count=0.0):
    """-> (total, geometry part) torch fp64 scalars; the inputs as torch_geometry_restatement.torch_total_geometry."""
    B, S, _, H, W = src.shape
    r = cfg.ssim_rate or 0.0
    total = geo = 0.0
    for ns in range(cfg.n_scales):
        h, w = H >> ns, W >> ns
        ct = F.interpolate(tgt, size=(h, w), mode='bilinear', align_corners=True)
        cs = F.interpolate(src.reshape(B, 3 * S, H, W), size=(h, w), mode='bilinear', align_corners=True)
        depth = 1.0 / disps[ns].reshape(B, 1, h * w)
        ys, xs = torch.meshgrid(torch.arange(h, dtype=K.dtype), torch.arange(w, dtype=K.dtype), indexing='ij')
        pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(h * w, dtype=K.dtype)])
        Ks = K[:, ns]
        cam = depth * (torch.linalg.inv(Ks) @ pix)
        for i in range(S):
            pose = poses[:, i]
            P = Ks @ torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((w - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((h - 1) / 2.) - 1
            inx = ((xn > -1) & (xn < 1)).detach()
            iny = ((yn > -1) & (yn < 1)).detach()
            valid = (inx & iny).reshape(B, 1, h, w)
            grid = torch.stack([torch.where(inx, xn, 2 * xn), torch.where(iny, yn, 2 * yn)], -1).reshape(B, h, w, 2)
            ref = cs[:, 3 * i:3 * i + 3]
            warped = F.grid_sample(ref, grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            zp = q[:, 2].reshape(B, 1, h, w)
            Dp = F.grid_sample(1.0 / src_disps[ns][:, i:i + 1], grid, mode='bilinear', padding_mode='zeros',
                               align_corners=True)
            c = torch.where(valid, zp + Dp, torch.ones_like(zp))
            diff_depth = torch.where(valid, ((zp - Dp).abs() / c).clamp(0, 1), torch.zeros_like(zp))
            m = (warped == 0).all(dim=1, keepdim=True).detach()     # the library's all-zero mask of the warped value
            diff_img = torch.where(m, torch.zeros_like(warped), (ct - warped).abs().clamp(0, 1))
            mask = valid.to(tgt.dtype)
            if automask:
                e = (ct - warped).abs().clamp(0, 1)
                auto = (e.mean(1, keepdim=True) < (ct - ref).abs().mean(1, keepdim=True)).to(tgt.dtype)
                mask = (auto * mask).detach()
            if r:
                pool = lambda x: F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)
                a, my = pool(warped), pool(ct)
                sx, sy, sxy = pool(warped * warped) - a * a, pool(ct * ct) - my * my, pool(warped * ct) - a * my
                n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
                dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
                ssim_map = torch.clamp((1 - n / dd) / 2, 0, 1) * (~m)
                diff_img = (1 - r) * diff_img + r * ssim_map
            if self_mask:
                diff_img = diff_img * (1 - diff_depth)
            for g in range(groups):
                total = total + mean_on_mask(diff_img[g::groups], mask[g::groups], min_count)
                gc = geometry_reg * mean_on_mask(diff_depth[g::groups], mask[g::groups], min_count)
                total = total + gc
                geo = geo + gc
    return total, geo
