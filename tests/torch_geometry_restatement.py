"""An independent torch fp64 restatement of SC-SfMLearner's loss terms as sfm_loss_geometry defines them (Bian et al.,
NeurIPS 2019, eqs. 5-7): the computed depth z' is the third row of P . [X, Y, Z, 1], the projected depth D' is the source
frame's depth 1 / d' sampled bilinearly (align-corners, zero padding) at the warped location, D_diff =
clamp(|z' - D'| / (z' + D'), 0, 1) on the strictly in-view pixels, the geometry term is its mean over the target pixels,
and the self-discovered mask M = 1 - D_diff weights the photometric terms.  Every input that carries a gradient may be a
leaf; autograd gives the reference gradients.  The smoothness term is left out (it is the oracle's, unchanged)."""
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from tests.torch_restatement import _rot


def torch_total_geometry(tgt, src, K, disps, poses, src_disps, cfg, geometry_reg, self_mask, rot=None):
    """-> (total, geometry term L_geo * geometry_reg) as torch fp64 scalars.  tgt (B,3,H,W), src (B,S,3,H,W), K (B,ns,3,3),
    disps list of (B,1,h,w), poses (B,S,6), src_disps list of (B,S,h,w) -- torch fp64 tensors, any of them a leaf.
    rot: pose rows -> [R | t] (B,3,4), default the reference's Euler transform."""
    B, S, _, H, W = src.shape
    use_ssim = bool(cfg.ssim_rate)
    rate = cfg.ssim_rate or 0.0
    pixel = ssim = geo = 0.0
    for ns in range(cfg.n_scales):
        h, w = H >> ns, W >> ns
        ct = F.interpolate(tgt, size=(h, w), mode='bilinear', align_corners=True)
        cs = F.interpolate(src.reshape(B, 3 * S, H, W), size=(h, w), mode='bilinear', align_corners=True)
        depth = 1.0 / disps[ns].reshape(B, 1, h * w)
        ys, xs = torch.meshgrid(torch.arange(h, dtype=K.dtype), torch.arange(w, dtype=K.dtype), indexing='ij')
        pix = torch.stack([xs.reshape(-1), ys.reshape(-1), torch.ones(h * w, dtype=K.dtype)])
        Ks = K[:, ns]
        cam = depth * (torch.linalg.inv(Ks) @ pix)
        n3, n1 = B * 3 * h * w, B * h * w
        for i in range(S):
            pose = poses[:, i]
            T = rot(pose, i) if rot is not None else torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)
            P = Ks @ T
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((w - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((h - 1) / 2.) - 1
            inx = ((xn > -1) & (xn < 1)).detach()
            iny = ((yn > -1) & (yn < 1)).detach()
            inb = (inx & iny).reshape(B, 1, h, w)
            xn = torch.where(inx, xn, 2 * xn)
            yn = torch.where(iny, yn, 2 * yn)
            grid = torch.stack([xn, yn], -1).reshape(B, h, w, 2)
            # geometry consistency: z' = q2 (the P-row product), D' = 1 / d' sampled where the pixel lands
            zp = q[:, 2].reshape(B, 1, h, w)
            Dp = F.grid_sample(1.0 / src_disps[ns][:, i:i + 1], grid, mode='bilinear', padding_mode='zeros',
                               align_corners=True)
            c = torch.where(inb, zp + Dp, torch.ones_like(zp))
            ratio = (zp - Dp).abs() / c
            diff = torch.where(inb, torch.clamp(ratio, 0, 1), torch.zeros_like(ratio))
            geo = geo + diff.sum() / n1
            Mw = (1 - diff) if self_mask else 1.0
            Pw = F.grid_sample(cs[:, 3 * i:3 * i + 3], grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            m = (Pw == 0).all(dim=1, keepdim=True).detach()
            err = torch.where(m, torch.zeros_like(Pw), (Pw - ct).abs()) * Mw
            pixel = pixel + err.sum() / n3
            if use_ssim:
                pool = lambda x: F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)
                a, my = pool(Pw), pool(ct)
                sx, sy, sxy = pool(Pw * Pw) - a * a, pool(ct * ct) - my * my, pool(Pw * ct) - a * my
                n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
                dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
                ssim = ssim + (torch.clamp((1 - n / dd) / 2, 0, 1) * (~m) * Mw).sum() / n3
    return (1 - rate) * pixel + rate * ssim + geometry_reg * geo, geometry_reg * geo
