"""An independent torch fp64 restatement of the photometric part of the loss with per-pixel weights, for autograd checks
of the per-pixel loss maps of tests/pixel_oracle.py (the map is d total / d M with M a leaf)."""
import torch
import torch.nn.functional as F

from oracle import sfm_oracle as O
from tests.torch_restatement import _rot


def torch_total_weighted(d, cfg, weights):
    """(1 - r) * pixel + r * ssim of base_model.py:64-118 for the float64 snippets d, with weights[s] (B,S,h,w) torch
    tensors (leaves, or None = 1) multiplying the photometric terms of every (pixel, source): the pyramid through
    F.interpolate, the grid through torch.linalg.inv(K) and K @ [R|t] with the x2 rule, grid_sample.  The smoothness and
    explainability-regulariser terms are left out (they are not weighted)."""
    tgt, src, K = (torch.from_numpy(d[k]) for k in ('tgt', 'src', 'intrinsics'))
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
            pose = torch.from_numpy(d['poses'][:, i])
            P = Ks @ torch.cat([_rot(pose[:, :3]), pose[:, 3:, None]], 2)
            q = P[:, :, :3] @ cam + P[:, :, 3:]
            z = q[:, 2] + 1e-10
            xn = (q[:, 0] / z) / ((w - 1) / 2.) - 1
            yn = (q[:, 1] / z) / ((h - 1) / 2.) - 1
            xn = torch.where((xn > -1) & (xn < 1), xn, 2 * xn)
            yn = torch.where((yn > -1) & (yn < 1), yn, 2 * yn)
            grid = torch.stack([xn, yn], -1).reshape(B, h, w, 2)
            Pw = F.grid_sample(cs[:, 3 * i:3 * i + 3], grid, mode='bilinear', padding_mode='zeros', align_corners=True)
            m = (Pw == 0).all(dim=1, keepdim=True)
            Mw = weights[ns][:, i:i + 1] if weights[ns] is not None else 1.0
            err = torch.where(m, torch.zeros_like(Pw), (Pw - ct).abs()) * Mw
            if use_exp:
                err = err * torch.sigmoid(torch.from_numpy(d['logits'][ns][:, i:i + 1]))
            pixel = pixel + err.sum() / n3
            if use_ssim:
                pool = lambda x: F.avg_pool2d(x, 3, 1, 1, count_include_pad=True)
                a, my = pool(Pw), pool(ct)
                sx, sy, sxy = pool(Pw * Pw) - a * a, pool(ct * ct) - my * my, pool(Pw * ct) - a * my
                n = (2 * a * my + O.SSIM_C1) * (2 * sxy + O.SSIM_C2)
                dd = (a * a + my * my + O.SSIM_C1) * (sx + sy + O.SSIM_C2)
                ssim = ssim + (torch.clamp((1 - n / dd) / 2, 0, 1) * (~m) * Mw).sum() / n3
    return (1 - rate) * pixel + rate * ssim
