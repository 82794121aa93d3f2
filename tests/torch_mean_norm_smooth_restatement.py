"""An independent torch fp64 restatement of the mean-normalised smoothness (SFM_FLAG_MEAN_NORM_SMOOTH) and Monodepth2's
edge weight (SFM_FLAG_EDGE_MEAN_ABS), for autograd checks of tests/mean_norm_smooth_oracle.py.  It follows Monodepth2's
training code literally -- mean_disp = disp.mean(2, True).mean(3, True); norm_disp = disp / (mean_disp + 1e-7);
get_smooth_loss(norm_disp, color) -- and differentiates through the division, with no use of the homogeneity identity.
The target pyramid goes through F.interpolate(align_corners=True), the reference's F.resize_images."""
import torch
import torch.nn.functional as F


def _act(x):
    return 10.0 * torch.sigmoid(x) + 0.01            # DISP_SCALING * sigmoid + MIN_DISP (disp_net.py:7-8, 104)


def torch_smoothness(tgt, disps, smooth_reg, B_global=None, edge=False, edge_mean_abs=False, mean_norm=True,
                     raw_disp_scales=0, snippet_weights=None):
    """-> (loss, rows): loss = sum_b w_b l_b and rows (B,) the per-snippet l_b, for tgt (B,3,H,W) and disps (list of
    (B,1,h_s,w_s)) torch tensors (leaves or not)."""
    B = tgt.shape[0]
    Bg = B_global or B
    rows = torch.zeros(B, dtype=tgt.dtype)
    for s, x in enumerate(disps):
        d = _act(x) if (raw_disp_scales >> s) & 1 else x
        if mean_norm:
            d = d / (d.mean(2, True).mean(3, True) + 1e-7)
        h, w = d.shape[2:]
        wgt = smooth_reg / 2 ** s
        per = lambda t: t.sum((1, 2, 3))
        if edge:
            img = tgt if tgt.shape[2:] == (h, w) else F.interpolate(tgt, size=(h, w), mode='bilinear', align_corners=True)
            i_dx, i_dy = img[..., :-1] - img[..., 1:], img[:, :, :-1] - img[:, :, 1:]
            if edge_mean_abs:
                e_x, e_y = torch.exp(-i_dx.abs().mean(1, True)), torch.exp(-i_dy.abs().mean(1, True))
            else:
                e_x, e_y = torch.exp(-i_dx.mean(1, True).abs()), torch.exp(-i_dy.mean(1, True).abs())
            gdx = (d[..., :-1] - d[..., 1:]).abs() * e_x
            gdy = (d[:, :, :-1] - d[:, :, 1:]).abs() * e_y
            l = per(gdx) / (Bg * h * (w - 1)) + per(gdy) / (Bg * (h - 1) * w)
        else:
            dx, dy = d[..., 1:] - d[..., :-1], d[:, :, 1:] - d[:, :, :-1]
            l = (per((dx[..., 1:] - dx[..., :-1]).abs()) / (Bg * h * (w - 2))
                 + per((dx[:, :, 1:] - dx[:, :, :-1]).abs()) / (Bg * (h - 1) * (w - 1))
                 + per((dy[..., 1:] - dy[..., :-1]).abs()) / (Bg * (h - 1) * (w - 1))
                 + per((dy[:, :, 1:] - dy[:, :, :-1]).abs()) / (Bg * (h - 2) * w))
        rows = rows + wgt * l
    wb = torch.ones(B, dtype=tgt.dtype) if snippet_weights is None else torch.as_tensor(snippet_weights, dtype=tgt.dtype)
    return (wb * rows).sum(), rows
