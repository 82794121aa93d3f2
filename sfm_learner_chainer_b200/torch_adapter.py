"""torch.autograd bridge for the fused loss (plumbing only: device memory + graph hook).

Used where the CNNs are torch modules (this image has no Chainer): DispNet/PoseNet stand-ins produce
pred_disps / pred_poses / pred_maskes, the fused kernels produce the loss and -- in the same pass --
its gradients, and backward() hands them to autograd after rescaling by the upstream gradient."""
import torch

from .functions import ViewSynthesisLoss


class _ViewSynthesisLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, op, tgt, src, intrinsics, weights, n_scales, use_exp, n_pred, *rest):
        preds, extra = rest[:n_pred], rest[n_pred:]
        # extra: n_scales per-pixel weights (or None) with op.pixel_terms, n_scales source disparities with
        # op.geometry_consistency
        pix_w = extra if op.pixel_terms else ()
        src_d = extra if op.geometry_consistency else ()
        disps = [p.contiguous() for p in preds[:n_scales]]
        poses = preds[n_scales].contiguous()
        logits = [p.contiguous() for p in preds[n_scales + 1:]] if use_exp else None
        # image gradients (op.image_grads) only for the images autograd asks for; the others are not computed
        ctx.want_tgt = op.image_grads and ctx.needs_input_grad[1]
        ctx.want_src = op.image_grads and ctx.needs_input_grad[2]
        want = tuple(n for n, w in (('tgt', ctx.want_tgt), ('src', ctx.want_src)) if w)
        # likewise the intrinsics gradient (op.intrinsics_grad) only when autograd asks for it
        ctx.want_k = op.intrinsics_grad and ctx.needs_input_grad[3]
        losses, grads = op.forward_backward(tgt.detach().contiguous(), src.detach().contiguous(),
                                            intrinsics.detach().contiguous(), [d.detach() for d in disps], poses.detach(),
                                            [l.detach() for l in logits] if logits else None, image_grads=want,
                                            intrinsics_grad=ctx.want_k,
                                            snippet_weights=weights.detach().contiguous() if weights is not None else None,
                                            **(dict(pixel_weights=[w.detach().contiguous() if w is not None else None
                                                                   for w in pix_w]) if op.pixel_terms else {}),
                                            **(dict(src_disps=[d.detach().contiguous() for d in src_d])
                                               if op.geometry_consistency else {}))
        ctx.op, ctx.grads, ctx.shape = op, grads, tuple(src.shape)
        ctx.n_scales, ctx.use_exp = n_scales, use_exp
        ctx.consumed = False
        outs = [losses]
        ctx.want_w = False
        if op.snippet_terms:
            # d total / d w_b = l_b[0]: the weights' gradient needs the rows alone
            ctx.want_w = weights is not None and ctx.needs_input_grad[4]
            ctx.rows = grads['snippet_losses']
            outs.append(ctx.rows)
        # likewise d total / d M_s = the per-pixel loss map of scale s
        ctx.maps = grads.get('pixel_losses') or []
        ctx.want_pw = [w is not None and ctx.needs_input_grad[8 + n_pred + s] for s, w in enumerate(pix_w)]
        outs += ctx.maps
        outs += grads.get('selection') or []      # min_reprojection: the selection maps, non-differentiable
        outs += grads.get('geometry_diff') or []  # geometry_consistency: the D_diff maps
        if 'valid_counts' in grads:               # valid_mean: the masks and the counts, non-differentiable
            outs += grads['valid_masks']
            outs.append(grads['valid_counts'])
        ctx.gsrc_d = grads.get('gsrc_disps') or []
        ctx.want_sd = [ctx.needs_input_grad[8 + n_pred + s] for s in range(len(src_d))]
        ctx.mark_non_differentiable(*outs)
        return (losses[0].clone(),) + tuple(outs)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gy, *_g_rest):
        # The gradients were produced by the forward's fused pass and are rescaled IN PLACE by the upstream gradient;
        # a second backward through the same node (retain_graph=True) would rescale them again, so it is refused.
        if ctx.consumed:
            raise RuntimeError('view_synthesis_loss: backward through the same loss node twice is not supported '
                               '(its gradients are computed in the forward pass and rescaled in place); call the loss again')
        ctx.consumed = True
        B, S, _, H, W = ctx.shape
        g = ctx.grads
        gy = gy.to(torch.float32).reshape(1).contiguous()
        gw = gy * ctx.rows[:, 0] if ctx.want_w else None
        ctx.op.scale_grads(g, gy, B, S, H, W)            # no-op on the device when gy == 1
        out = list(g['gdisps']) + [g['gposes']]
        if ctx.use_exp:
            out += list(g['glogits'])
        gtgt = g.get('gtgt') if ctx.want_tgt else None
        gsrc = g.get('gsrc') if ctx.want_src else None
        gk = g.get('gintrinsics') if ctx.want_k else None
        gpw = tuple(gy * m if want else None for m, want in zip(ctx.maps, ctx.want_pw))
        gsd = tuple(gy * m if want else None for m, want in zip(ctx.gsrc_d, ctx.want_sd))
        return (None, gtgt, gsrc, gk, gw, None, None, None) + tuple(out) + gpw + gsd


def view_synthesis_loss(op, tgt, src, intrinsics, pred_disps, pred_poses, pred_maskes=None, snippet_weights=None,
                        pixel_weights=None, src_disps=None):
    """-> (total_loss scalar tensor with grad_fn, losses (5,) tensor [total, pixel, smooth, exp, ssim]).

    pred_poses: (B,S,6) tensor or a tuple of S (B,6) tensors as PoseNet returns them (pose_net.py:52-54).
    With op.snippet_terms: -> (total, losses, snippet_losses (B,5)); snippet_weights (B,) (None = all 1) weight the
    snippets, total = sum_b w_b * snippet_losses[b, 0], the other inputs' gradients are the weighted ones, and weights
    that require grad receive gy * snippet_losses[:, 0].  See ViewSynthesisLoss for padding a captured batch.
    With op.pixel_terms: pixel_weights (list of n_scales (B,S,h,w) tensors or None entries; None = all 1) weight the
    photometric terms per (pixel, source), and pixel_losses (list of n_scales maps d total / d weights) is appended to
    the returned tuple; weights that require grad receive gy * pixel_losses[s].
    With op.min_reprojection: the selection maps (list of n_scales (B,h,w) int8 tensors: the chosen source, -1
    auto-masked, -2 no candidate) are appended to the returned tuple; they are not differentiable.
    With op.geometry_consistency: src_disps (list of n_scales (B,S,h,w) tensors, the activated disparity of every source
    frame, e.g. DispNet run on the source frames) is required and receives its gradient through autograd; the D_diff maps
    (list of n_scales (B,S,h,w) tensors, not differentiable) are appended to the returned tuple.
    With op.valid_mean the valid-pixel masks (list of n_scales (B,S,h,w) uint8 tensors) and the counts ((n_scales,S,G)
    int32 tensor) follow the D_diff maps; neither is differentiable.
    """
    assert isinstance(op, ViewSynthesisLoss)
    if snippet_weights is not None and not op.snippet_terms:
        raise ValueError('snippet_weights needs ViewSynthesisLoss(snippet_terms=True)')
    if pixel_weights is not None and not op.pixel_terms:
        raise ValueError('pixel_weights needs ViewSynthesisLoss(pixel_terms=True)')
    pix_w = []
    if op.pixel_terms:
        pix_w = list(pixel_weights) if pixel_weights is not None else [None] * op.n_scales
        if len(pix_w) != op.n_scales:
            raise ValueError('pixel_weights must hold %d entries (one per scale, None = 1)' % op.n_scales)
    if isinstance(pred_poses, (tuple, list)):
        pred_poses = torch.stack(list(pred_poses), dim=1)
    src_d = []
    if op.geometry_consistency:
        if src_disps is None or len(src_disps) != op.n_scales:
            raise ValueError('geometry_consistency needs src_disps, a list of %d (B,S,h,w) tensors' % op.n_scales)
        src_d = list(src_disps)
    elif src_disps is not None:
        raise ValueError('src_disps needs ViewSynthesisLoss(geometry_consistency=True)')
    use_exp = op.use_exp
    preds = list(pred_disps) + [pred_poses] + (list(pred_maskes) if use_exp else [])
    res = _ViewSynthesisLossFn.apply(op, tgt, src, intrinsics, snippet_weights, op.n_scales, use_exp, len(preds), *preds,
                                     *pix_w, *src_d)
    if not (op.pixel_terms or op.min_reprojection or op.geometry_consistency):
        return res
    if op.valid_mean:
        k = len(res) - 2 * op.n_scales - 1
        return tuple(res[:k]) + (list(res[k:k + op.n_scales]), list(res[k + op.n_scales:-1]), res[-1])
    k = len(res) - op.n_scales
    return tuple(res[:k]) + (list(res[k:]),)
