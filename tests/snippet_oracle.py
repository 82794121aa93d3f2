"""Reference of the per-snippet weighted loss, built on linearity from the numpy oracle.

Every term of the loss is a sum over the snippets with the 1/B_global means inside each snippet's term, so the oracle
run on the one-snippet slice b with B_global = the batch's global size gives snippet b's losses l_b and gradients.  The
weighted losses are sum_b w_b * l_b and every gradient is snippet b's gradient times w_b.  This is independent of how
the kernels fold the weight in."""
import copy

import numpy as np

from oracle import sfm_oracle as O

_PER_SNIPPET_KW = ('proj_override', 'kinv_override')


def sfm_loss_snippets(tgt, src, intrinsics, disps, poses, logits, cfg, snippet_weights=None, raw=None, **kw):
    """-> (weighted losses (5,) fp64, rows (B,5) fp64 of the unweighted l_b, weighted grads dict or None).

    raw: None for O.sfm_loss, or dict(raw_disp_scales=..., raw_pose=...) for O.sfm_loss_raw.  kw: passed through
    (want_grads, want_image_grads, want_intrinsics_grad, proj_override, kinv_override)."""
    B = src.shape[0]
    w = np.ones(B) if snippet_weights is None else np.asarray(snippet_weights, np.float64)
    cfg_b = copy.copy(cfg)
    cfg_b.B_global = cfg.B_global or B
    rows = np.zeros((B, 5))
    per = []
    for b in range(B):
        sl = slice(b, b + 1)
        kwb = {k: (v[sl] if k in _PER_SNIPPET_KW and v is not None else v) for k, v in kw.items()}
        args = (tgt[sl], src[sl], intrinsics[sl], [d[sl] for d in disps], poses[sl],
                [l[sl] for l in logits] if logits is not None else None, cfg_b)
        if raw is None:
            L, G, _ = O.sfm_loss(*args, **kwb)
        else:
            L, G, _ = O.sfm_loss_raw(*args, **raw, **kwb)
        rows[b] = O.losses_vec(L)
        per.append(G)
    losses = (w[:, None] * rows).sum(0)
    if per[0] is None:
        return losses, rows, None
    grads = {}
    for k, v in per[0].items():
        if v is None:
            grads[k] = None
        elif isinstance(v, list):
            grads[k] = [np.concatenate([w[b] * per[b][k][s].astype(np.float64) for b in range(B)]) for s in range(len(v))]
        else:
            grads[k] = np.concatenate([w[b] * per[b][k].astype(np.float64) for b in range(B)])
    return losses, rows, grads
