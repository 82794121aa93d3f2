"""Host-side operators of the view-synthesis loss path (thin: argument checks, output allocation and
one C-ABI call each).  Names and argument meaning follow the reference."""
import ctypes as C
import math

from . import device as D
from . import lib as L

N_SCALES = 4


def _vp(a):
    p = D.ptr(a)
    return C.c_void_p(p) if p is not None else C.c_void_p(0)


class ViewSynthesisLoss(object):
    """The loss loop of SFMLearner.__call__ (models/base_model.py:64-118) as one fused operator.

    smooth_reg, exp_reg, ssim_rate: the reference's `architecture:` flags (base_model.py:37-39).
    B_global: batch size every F.mean divides by when the batch is sharded by snippet across
    processes (default: the local batch).
    raw_disp_scales: bit mask of scales whose `pred_disps[s]` is the PRE-activation `dispout` map; the
    kernels then apply disp = 10 * sigmoid(x) + 0.01 (models/disp_net.py:104) and return the gradient
    w.r.t. that map.  raw_pose: `poses` is PoseNet's `poseout` map (B, 6*S, h', w') and the kernels apply
    0.01 * mean over (h', w') (models/pose_net.py:52-53); `gposes` then has the map's shape.
    image_grads: forward_backward also returns gtgt (B,3,H,W) and gsrc (B,S,3,H,W), the gradients of the reported
    total w.r.t. the two images (for images that come out of a differentiable module); not with edge_aware_smooth.
    intrinsics_grad: forward_backward and backward also return gintrinsics (B,n_scales,3,3), the gradient of the
    reported total w.r.t. `intrinsics` (for a camera that is learned); not with caller-supplied proj / kinv.
    snippet_terms: forward and forward_backward take `snippet_weights` (B,) float32 device array w (None = all 1) and
    also return the per-snippet losses (B,5) l_b = total, pixel, smooth, exp, ssim of snippet b (unweighted, with the
    1/B_global means); the five losses are then sum_b w_b * l_b and every gradient is that of their total.  The
    weights are device data, so a CUDA graph captured for B snippets can run a batch of B_real < B: fill the padding
    with copies of a real snippet (a zero disparity gives NaN, and NaN * 0 is NaN), keep B_global = B and pass
    w_b = B / B_real for the real snippets and 0 for the padding; that gives the loss and gradients of the B_real batch
    up to rounding.  d total / d w_b = l_b[0] (the torch adapter returns it as the weights' gradient).
    pixel_terms: forward and forward_backward take `pixel_weights`, a list of n_scales float32 device arrays
    (B,S,h_s,w_s) laid out like the logits, or None entries (None = all 1), and also return the per-pixel loss maps
    (a list of n_scales (B,S,h_s,w_s) arrays).  M_s multiplies the photometric terms of every (pixel, source) at scale s
    (the means keep their denominators; the smoothness and explainability regularisers are not weighted), every gradient
    is that of the weighted total, and the map is d total / d M: each pixel's share of the photometric loss
    (sum M * map = (1 - ssim_rate) * pixel + ssim_rate * ssim).  Masks of moving objects, the ego-vehicle or sky, and
    learned weight maps (whose gradient is the map) go in here; a forward call with maps is the validation use.  Not
    with image_grads.
    min_reprojection: Monodepth2's per-pixel minimum reprojection (each target pixel is scored on the source view with
    the smallest error, masked sources excluded) and, with automask, its auto-masking (a pixel is dropped when an
    unwarped source matches the target at least as well); see sfm_loss_min_reprojection in include/sfmloss.h for the
    exact rules.  forward and forward_backward also return the selection maps (a list of n_scales (B,h_s,w_s) int8
    arrays: the chosen source, -1 auto-masked, -2 no candidate), appended like the pixel maps / as `selection`.  Not
    with exp_reg, image_grads or pixel_terms; ssim_rate must lie in [0, 1].
    full_res_multiscale: Monodepth2's full-resolution multi-scale loss: every coarse disparity is upsampled bilinearly
    to (H, W) (align_corners=False) and the photometric terms of every scale are computed there with intrinsics[:, 0],
    while the smoothness term stays at the scale's own resolution; see SFM_FLAG_FULL_RES_MULTISCALE in include/sfmloss.h.
    The scales are summed (Monodepth2's 1 / num_scales is the caller's).  The gradients keep the native shapes; the
    per-pixel weights and maps, the selection maps and the debug dumps are (.., H, W) at every scale, and gintrinsics
    holds the whole gradient at [:, 0].  Not with exp_reg or image_grads.
    mean_norm_smooth: Monodepth2's mean-normalised smoothness: the smoothness term of every scale (either kind) is
    evaluated on disp / (mean(disp) + 1e-7), the mean per snippet and scale over the native plane of the activated
    disparity; see SFM_FLAG_MEAN_NORM_SMOOTH in include/sfmloss.h.  The photometric terms are untouched.
    edge_mean_abs: with edge_aware_smooth, Monodepth2's edge weight exp(-mean_c |dI_c|) instead of the reference's
    exp(-|mean_c dI_c|).
    border_padding: Monodepth2's image borders: the warp samples with border clamping (grid_sample's
    padding_mode="border", align-corners mapping, no x2 rule) and masks only pixels whose projection is degenerate, and
    the SSIM windows use reflection padding by one pixel; see SFM_FLAG_BORDER_PADDING in include/sfmloss.h.  Not with
    exp_reg, image_grads or debug dumps.
    axisangle_pose: Monodepth2's pose parametrisation: every `poses` row is (v0, v1, v2, tx, ty, tz), an axis-angle
    vector and a translation, turned into [R | t] as Monodepth2's transformation_from_parameters does (no angle
    clipping); gposes is the gradient w.r.t. those rows.  invert_sources: tuple of source indices whose transform is
    inverted, [R^T | -R^T t] (Monodepth2 inverts the pose of every source that precedes the target: frame ids
    [0, -1, 1] give invert_sources=(0,)); needs axisangle_pose and is checked against S at call time.  See
    SFM_FLAG_AXISANGLE_POSE in include/sfmloss.h.
    geometry_consistency: SC-SfMLearner's geometry consistency term (Bian et al., NeurIPS 2019): every target pixel is
    projected into each source frame and its computed depth z' is compared with the source frame's own predicted depth
    D' sampled there, D_diff = clip(|z' - D'| / (z' + D'), 0, 1) on the in-view pairs; geometry_reg times its mean over
    the target pixels (summed over the sources and scales) is added to the total and reported in the exp_loss slot.
    forward and forward_backward then take `src_disps`, a list of n_scales (B,S,h_s,w_s) arrays with the activated
    disparity of every source frame, and return `geometry_diff` (the D_diff maps, like src_disps) appended to the
    forward's tuple / in the grads dict, where forward_backward also puts `gsrc_disps`, the gradient w.r.t. src_disps.
    self_mask: the photometric terms of every (pixel, source) are weighted by M = 1 - D_diff, with the gradient through
    M (SC-SfMLearner's self-discovered mask).  See sfm_loss_geometry in include/sfmloss.h.  Not with exp_reg,
    image_grads, pixel_terms, min_reprojection, full_res_multiscale, border_padding or debug dumps.
    valid_mean: SC-SfMLearner's means over the valid pixels (its released compute_pairwise_loss / mean_on_mask; needs
    geometry_consistency): each (scale, source) term is a mean over the pairs that count instead of over B_global h w,
    and the L1 difference is clamped to 1.  valid_automask: a pair counts only where the clamped L1 of the warped source
    is below the L1 of the unwarped source (--with-auto-mask); else every in-view pair counts.  valid_min_count: a term
    whose count (3 n for the photometric terms, n for the geometry term) is <= it contributes 0 (released value 10000).
    count_groups: G, snippet b counts in group b mod G (1: one batch-wide count per source and scale; S for the reverse
    direction of INTEGRATION.md §6).  forward and forward_backward then also return `valid_masks` (list of n_scales
    (B,S,h,w) uint8, 1 where the pair counts) and `valid_counts` ((n_scales,S,G) int32), appended to the forward's tuple
    after the D_diff maps / in the grads dict.  Not with a peer or B_global != B.  See sfm_loss_geometry_valid_mean in
    include/sfmloss.h.
    """

    def __init__(self, smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0, n_scales=N_SCALES, B_global=None,
                 raw_disp_scales=0, raw_pose=False, edge_aware_smooth=False, image_grads=False,
                 intrinsics_grad=False, snippet_terms=False, pixel_terms=False, min_reprojection=False, automask=True,
                 full_res_multiscale=False, mean_norm_smooth=False, edge_mean_abs=False, border_padding=False,
                 axisangle_pose=False, invert_sources=(), geometry_consistency=False, geometry_reg=0.5, self_mask=False,
                 valid_mean=False, valid_automask=True, valid_min_count=10000.0, count_groups=1):
        if self_mask and not geometry_consistency:
            raise ValueError('self_mask needs geometry_consistency')
        if valid_mean:
            if not geometry_consistency:
                raise ValueError('valid_mean needs geometry_consistency')
            if B_global is not None:
                raise ValueError('valid_mean is not supported with B_global (the counts are batch-global)')
            if not math.isfinite(float(valid_min_count)) or float(valid_min_count) < 0.0:
                raise ValueError('valid_min_count must be finite and >= 0, got %r' % (valid_min_count,))
            if int(count_groups) < 1:
                raise ValueError('count_groups must be >= 1, got %r' % (count_groups,))
        self.valid_mean = bool(valid_mean)
        self.valid_automask = bool(valid_automask)
        self.valid_min_count = float(valid_min_count)
        self.count_groups = int(count_groups)
        if geometry_consistency:
            for name, on in (('image_grads', image_grads), ('pixel_terms', pixel_terms),
                             ('min_reprojection', min_reprojection), ('full_res_multiscale', full_res_multiscale),
                             ('border_padding', border_padding)):
                if on:
                    raise ValueError('geometry_consistency is not supported together with %s' % name)
            if float(exp_reg or 0.0) != 0.0:
                raise ValueError('geometry_consistency is not supported together with the explainability branch (exp_reg)')
        self.geometry_consistency = bool(geometry_consistency)
        self.geometry_reg = float(geometry_reg)
        self.self_mask = bool(self_mask)
        invert_sources = tuple(int(i) for i in (invert_sources or ()))
        if invert_sources and not axisangle_pose:
            raise ValueError('invert_sources needs axisangle_pose')
        if any(i < 0 for i in invert_sources):
            raise ValueError('invert_sources must hold source indices >= 0, got %r' % (invert_sources,))
        self.axisangle_pose = bool(axisangle_pose)
        self.invert_sources = invert_sources
        if edge_mean_abs and not edge_aware_smooth:
            raise ValueError('edge_mean_abs needs edge_aware_smooth')
        if border_padding:
            if image_grads:
                raise ValueError('border_padding is not supported together with image_grads')
            if float(exp_reg or 0.0) != 0.0:
                raise ValueError('border_padding is not supported together with the explainability branch (exp_reg)')
        self.border_padding = bool(border_padding)
        self.mean_norm_smooth = bool(mean_norm_smooth)
        self.edge_mean_abs = bool(edge_mean_abs)
        if full_res_multiscale:
            if image_grads:
                raise ValueError('full_res_multiscale is not supported together with image_grads')
            if float(exp_reg or 0.0) != 0.0:
                raise ValueError('full_res_multiscale is not supported together with the explainability branch (exp_reg)')
        self.full_res_multiscale = bool(full_res_multiscale)
        if image_grads and edge_aware_smooth:
            raise ValueError('image_grads is not supported together with edge_aware_smooth')
        if image_grads and pixel_terms:
            raise ValueError('image_grads is not supported together with pixel_terms')
        if min_reprojection:
            if image_grads or pixel_terms:
                raise ValueError('min_reprojection is not supported together with image_grads or pixel_terms')
            if float(exp_reg or 0.0) != 0.0:
                raise ValueError('min_reprojection is not supported together with the explainability branch (exp_reg)')
            if not 0.0 <= float(ssim_rate or 0.0) <= 1.0:
                raise ValueError('min_reprojection needs ssim_rate in [0, 1]')
        self.min_reprojection = bool(min_reprojection)
        self.automask = bool(automask)
        self.pixel_terms = bool(pixel_terms)
        self.image_grads = bool(image_grads)
        self.intrinsics_grad = bool(intrinsics_grad)
        self.snippet_terms = bool(snippet_terms)
        # edge_aware_smooth: smoothness term = compute_disp_smooth (base_model.py:144-155, commented out at :78-80)
        self.edge_aware_smooth = bool(edge_aware_smooth)
        self.raw_disp_scales = int(raw_disp_scales)
        self.raw_pose = bool(raw_pose)
        self.smooth_reg = float(smooth_reg or 0.0)
        self.exp_reg = float(exp_reg or 0.0)
        self.ssim_rate = float(ssim_rate or 0.0)
        self.n_scales = int(n_scales)
        self.B_global = B_global
        self._lib = L.load()
        self._ws = {}
        self._ev_pyramid = None      # build_pyramid done (the loss call waits for it when it reuses the pyramid)
        self._ev_loss = None         # last loss call done with the workspace (the next build_pyramid waits for it)

    # ---- helpers
    @property
    def use_exp(self):
        return self.exp_reg != 0.0

    def _desc(self, B, S, H, W, flags=0, raw_pose_hw=0):
        if self.edge_aware_smooth:
            flags |= L.SFM_FLAG_EDGE_AWARE_SMOOTH
        if self.image_grads:
            flags |= L.SFM_FLAG_IMAGE_GRADS
        if self.snippet_terms:
            flags |= L.SFM_FLAG_SNIPPET_TERMS
        if self.min_reprojection:
            flags |= L.SFM_FLAG_MIN_REPROJECTION
        if self.full_res_multiscale:
            flags |= L.SFM_FLAG_FULL_RES_MULTISCALE
        if self.mean_norm_smooth:
            flags |= L.SFM_FLAG_MEAN_NORM_SMOOTH
        if self.edge_mean_abs:
            flags |= L.SFM_FLAG_EDGE_MEAN_ABS
        if self.border_padding:
            flags |= L.SFM_FLAG_BORDER_PADDING
        if self.geometry_consistency:
            flags |= L.SFM_FLAG_GEOMETRY_CONSISTENCY
        if self.valid_mean:
            flags |= L.SFM_FLAG_VALID_MEAN
        if self.axisangle_pose:
            flags |= L.SFM_FLAG_AXISANGLE_POSE
            for i in self.invert_sources:
                if i >= S:
                    raise ValueError('invert_sources names source %d, but there are S=%d sources' % (i, S))
                flags |= 1 << (L.SFM_FLAG_POSE_INVERT_SHIFT + i)
        return L.SfmDesc(B, S, H, W, self.n_scales, int(self.B_global or 0), self.smooth_reg, self.exp_reg,
                         self.ssim_rate, flags, self.raw_disp_scales, raw_pose_hw)

    def _workspace(self, desc, like):
        # the image-gradient, snippet-terms, min-reprojection, full-resolution and mean-normalisation flags size the
        # workspace; the per-call flags (tables, reused pyramid) do not
        sizing = (L.SFM_FLAG_IMAGE_GRADS | L.SFM_FLAG_SNIPPET_TERMS | L.SFM_FLAG_MIN_REPROJECTION
                  | L.SFM_FLAG_FULL_RES_MULTISCALE | L.SFM_FLAG_MEAN_NORM_SMOOTH | L.SFM_FLAG_GEOMETRY_CONSISTENCY
                  | L.SFM_FLAG_VALID_MEAN)
        key = (desc.B, desc.S, desc.H, desc.W, desc.n_scales, desc.flags & sizing,
               str(getattr(like, 'device', '')))
        ws = self._ws.get(key)
        if ws is None:
            n = self._lib.sfm_workspace_bytes(C.byref(desc))
            if n == 0:
                L.check(L.SFM_E_INVALID_DESC)
            ws = D.empty(like, (n + 256,), 'uint8')
            self._ws = {key: ws}
        p = D.ptr(ws)
        return C.c_void_p((p + 255) // 256 * 256)

    def _pack(self, tgt, src, intrinsics, disps, poses, logits, proj=None, kinv=None):
        if getattr(src, 'ndim', len(src.shape)) != 5:
            raise ValueError('src_imgs must be (B, S, 3, H, W) (base_model.py:57)')
        B, S, _, H, W = src.shape
        ns = self.n_scales
        D.check_array(tgt, 'tgt_img', (B, 3, H, W))
        D.check_array(src, 'src_imgs', (B, S, 3, H, W))
        D.check_array(intrinsics, 'intrinsics', (B, ns, 3, 3))
        raw_pose_hw = 0
        if self.raw_pose:
            if len(poses.shape) not in (3, 4) or poses.shape[0] != B or poses.shape[1] != 6 * S:
                raise ValueError('raw poses must be the poseout map (B, 6*S, h\', w\') (pose_net.py:51)')
            D.check_array(poses, 'poses')
            raw_pose_hw = 1
            for n in poses.shape[2:]:
                raw_pose_hw *= int(n)
            self._pose_shape = tuple(poses.shape)
        else:
            D.check_array(poses, 'poses', (B, S, 6))
            self._pose_shape = (B, S, 6)
        if len(disps) != ns:
            raise ValueError('expected %d disparity maps, got %d' % (ns, len(disps)))
        flags = 0
        inp = L.SfmInputs()
        inp.tgt, inp.src, inp.intrinsics, inp.poses = _vp(tgt), _vp(src), _vp(intrinsics), _vp(poses)
        for s in range(ns):
            D.check_array(disps[s], 'pred_disps[%d]' % s, (B, 1, H >> s, W >> s))
            inp.disps[s] = D.ptr(disps[s])
        if self.use_exp:
            if logits is None or len(logits) != ns:
                raise ValueError('exp_reg > 0 needs %d explainability logit maps (pose_net do_exp=True)' % ns)
            for s in range(ns):
                D.check_array(logits[s], 'pred_maskes[%d]' % s, (B, S, H >> s, W >> s))
                inp.logits[s] = D.ptr(logits[s])
        if proj is not None or kinv is not None:
            D.check_array(proj, 'proj', (B, S, ns, 3, 4))
            D.check_array(kinv, 'kinv', (B, ns, 3, 3))
            inp.proj, inp.kinv = _vp(proj), _vp(kinv)
            flags |= L.SFM_FLAG_TABLES_PROVIDED
        return self._desc(B, S, H, W, flags, raw_pose_hw), inp

    def _step_hw(self, desc, s):
        """(h, w) of the photometric terms of scale s: the scale's own size, or (H, W) with full_res_multiscale."""
        if self.full_res_multiscale:
            return desc.H, desc.W
        return desc.H >> s, desc.W >> s

    def _alloc_grads(self, desc, tgt):
        B, S, H, W = desc.B, desc.S, desc.H, desc.W
        g = L.SfmGrads()
        gd = [D.empty(tgt, (B, 1, H >> s, W >> s)) for s in range(self.n_scales)]
        gp = D.empty(tgt, self._pose_shape)
        gl = [D.empty(tgt, (B, S, H >> s, W >> s)) for s in range(self.n_scales)] if self.use_exp else None
        for s in range(self.n_scales):
            g.gdisps[s] = D.ptr(gd[s])
            if gl is not None:
                g.glogits[s] = D.ptr(gl[s])
        g.gposes = D.ptr(gp)
        return g, dict(gdisps=gd, gposes=gp, glogits=gl)

    def _want_intrinsics_grad(self, want, proj, kinv):
        if not (self.intrinsics_grad and want):
            return False
        if proj is not None or kinv is not None:
            raise ValueError('intrinsics_grad needs the projection tables built from the intrinsics (no proj / kinv)')
        return True

    def _intrinsics_grad(self, desc, inp, tgt, out, want):
        """Adds gintrinsics to `out` (None when not requested) from the cells the gradient call just left in the
        workspace."""
        if not self.intrinsics_grad:
            return
        out['gintrinsics'] = None
        if want:
            out['gintrinsics'] = D.empty(tgt, (desc.B, self.n_scales, 3, 3))
            L.check(self._lib.sfm_intrinsics_grad(C.byref(desc), C.byref(inp), self._workspace(desc, tgt),
                                                  _vp(out['gintrinsics']), C.c_void_p(D.current_stream(tgt))))

    def _snippet_terms(self, desc, tgt, snippet_weights):
        """-> (SfmSnippetTerms or None, snippet losses (B,5) or None)."""
        if not self.snippet_terms:
            if snippet_weights is not None:
                raise ValueError('snippet_weights needs ViewSynthesisLoss(snippet_terms=True)')
            return None, None
        if snippet_weights is not None:
            D.check_array(snippet_weights, 'snippet_weights', (desc.B,))
        rows = D.empty(tgt, (desc.B, 5))
        return L.SfmSnippetTerms(_vp(snippet_weights), _vp(rows)), rows

    def _pixel_terms(self, desc, tgt, pixel_weights):
        """-> (SfmPixelTerms or None, per-pixel loss maps (list of n_scales (B,S,h,w)) or None)."""
        if not self.pixel_terms:
            if pixel_weights is not None:
                raise ValueError('pixel_weights needs ViewSynthesisLoss(pixel_terms=True)')
            return None, None
        ns = self.n_scales
        if pixel_weights is None:
            pixel_weights = [None] * ns
        if len(pixel_weights) != ns:
            raise ValueError('pixel_weights must hold %d entries (one per scale, None = 1), got %d' % (ns, len(pixel_weights)))
        pt = L.SfmPixelTerms()
        maps = []
        for s in range(ns):
            shape = (desc.B, desc.S) + self._step_hw(desc, s)
            if pixel_weights[s] is not None:
                D.check_array(pixel_weights[s], 'pixel_weights[%d]' % s, shape)
                pt.weights[s] = D.ptr(pixel_weights[s])
            maps.append(D.empty(tgt, shape))
            pt.losses[s] = D.ptr(maps[s])
        return pt, maps

    def _min_reprojection(self, desc, tgt):
        """-> (SfmMinReprojection or None, selection maps (list of n_scales (B,h,w) int8) or None)."""
        if not self.min_reprojection:
            return None, None
        mr = L.SfmMinReprojection()
        mr.automask = 1 if self.automask else 0
        sel = []
        for s in range(self.n_scales):
            sel.append(D.empty(tgt, (desc.B,) + self._step_hw(desc, s), 'int8'))
            mr.selection[s] = D.ptr(sel[s])
        return mr, sel

    def _geometry(self, desc, tgt, src_disps, want_grads):
        """-> (SfmGeometry, D_diff maps, gsrc_disps or None), each a list of n_scales (B,S,h_s,w_s) arrays."""
        if src_disps is None or len(src_disps) != self.n_scales:
            raise ValueError('geometry_consistency needs src_disps, a list of %d (B,S,h,w) source disparity maps'
                             % self.n_scales)
        ge = L.SfmGeometry()
        ge.geometry_reg = self.geometry_reg
        ge.self_mask = 1 if self.self_mask else 0
        diff, gsd = [], [] if want_grads else None
        for s in range(self.n_scales):
            shape = (desc.B, desc.S, desc.H >> s, desc.W >> s)
            D.check_array(src_disps[s], 'src_disps[%d]' % s, shape)
            ge.src_disps[s] = D.ptr(src_disps[s])
            diff.append(D.empty(tgt, shape))
            ge.diff_maps[s] = D.ptr(diff[s])
            if want_grads:
                gsd.append(D.empty(tgt, shape))
                ge.gsrc_disps[s] = D.ptr(gsd[s])
        return ge, diff, gsd

    def _valid_mean(self, desc, tgt):
        """-> (SfmValidMean or None, masks (list of n_scales (B,S,h_s,w_s) uint8), counts (n_scales,S,G) int32)."""
        if not self.valid_mean:
            return None, None, None
        if not 1 <= self.count_groups <= desc.B:
            raise ValueError('count_groups = %d must lie in [1, B = %d]' % (self.count_groups, desc.B))
        vm = L.SfmValidMean()
        vm.automask = 1 if self.valid_automask else 0
        vm.groups = self.count_groups
        vm.min_count = self.valid_min_count
        masks = []
        for s in range(self.n_scales):
            masks.append(D.empty(tgt, (desc.B, desc.S, desc.H >> s, desc.W >> s), 'uint8'))
            vm.masks[s] = D.ptr(masks[s])
        counts = D.empty(tgt, (self.n_scales, desc.S, self.count_groups), 'int32')
        vm.counts = D.ptr(counts)
        return vm, masks, counts

    def _run_geometry(self, desc, inp, terms, ge, vm, losses, grads, tgt, peer):
        args = (C.byref(desc), C.byref(inp), C.byref(terms) if terms else None, C.byref(ge))
        tail = (_vp(losses), C.byref(grads) if grads is not None else None, self._workspace(desc, tgt), peer,
                C.c_void_p(D.current_stream(tgt)))
        if vm is None:
            L.check(self._lib.sfm_loss_geometry(*args, *tail))
        else:
            L.check(self._lib.sfm_loss_geometry_valid_mean(*args, C.byref(vm), *tail))

    # ---- operators
    def forward(self, tgt, src, intrinsics, disps, poses, logits=None, proj=None, kinv=None, debug=False,
                snippet_weights=None, pixel_weights=None, src_disps=None):
        """-> losses (5,) device array in the order of lib.LOSS_KEYS [, debug dict].
        With the operator's snippet_terms: -> (losses, snippet losses (B,5)), losses = sum_b w_b * l_b.
        With the operator's pixel_terms the per-pixel loss maps (list of n_scales (B,S,h,w)) are appended as the last
        element: (losses, maps) or (losses, snippet losses, maps).
        With the operator's min_reprojection the selection maps (list of n_scales (B,h,w) int8) are appended likewise.
        With the operator's geometry_consistency: src_disps (list of n_scales (B,S,h,w)) is required and the D_diff maps
        (list of n_scales (B,S,h,w)) are appended likewise; with valid_mean then also the masks and the counts."""
        if debug and (self.snippet_terms or self.pixel_terms or self.min_reprojection or self.border_padding
                      or self.geometry_consistency):
            raise ValueError('debug dumps are not available on an operator with snippet_terms, pixel_terms, min_reprojection, '
                             'border_padding or geometry_consistency')
        if src_disps is not None and not self.geometry_consistency:
            raise ValueError('src_disps needs ViewSynthesisLoss(geometry_consistency=True)')
        desc, inp = self._pack(tgt, src, intrinsics, disps, poses, logits, proj, kinv)
        losses = D.empty(tgt, (5,))
        if self.geometry_consistency:
            terms, rows = self._snippet_terms(desc, tgt, snippet_weights)
            if pixel_weights is not None:
                raise ValueError('pixel_weights needs ViewSynthesisLoss(pixel_terms=True)')
            ge, diff, _ = self._geometry(desc, tgt, src_disps, False)
            vm, masks, counts = self._valid_mean(desc, tgt)
            self._run_geometry(desc, inp, terms, ge, vm, losses, None, tgt, None)
            return (losses,) + ((rows,) if self.snippet_terms else ()) + (diff,) + ((masks, counts) if vm else ())
        if self.min_reprojection:
            terms, rows = self._snippet_terms(desc, tgt, snippet_weights)
            if pixel_weights is not None:
                raise ValueError('pixel_weights needs ViewSynthesisLoss(pixel_terms=True)')
            mr, sel = self._min_reprojection(desc, tgt)
            L.check(self._lib.sfm_loss_min_reprojection(C.byref(desc), C.byref(inp), C.byref(terms) if terms else None,
                                                        C.byref(mr), _vp(losses), None, self._workspace(desc, tgt), None,
                                                        C.c_void_p(D.current_stream(tgt))))
            return (losses,) + ((rows,) if self.snippet_terms else ()) + (sel,)
        if self.snippet_terms or self.pixel_terms:
            terms, rows = self._snippet_terms(desc, tgt, snippet_weights)
            pt, maps = self._pixel_terms(desc, tgt, pixel_weights)
            L.check(self._lib.sfm_loss_weighted(C.byref(desc), C.byref(inp), C.byref(terms) if terms else None,
                                                C.byref(pt) if pt else None, _vp(losses), None, None,
                                                self._workspace(desc, tgt), None, C.c_void_p(D.current_stream(tgt))))
            out = (losses,) + ((rows,) if self.snippet_terms else ()) + ((maps,) if self.pixel_terms else ())
            return out
        if snippet_weights is not None:
            raise ValueError('snippet_weights needs ViewSynthesisLoss(snippet_terms=True)')
        if pixel_weights is not None:
            raise ValueError('pixel_weights needs ViewSynthesisLoss(pixel_terms=True)')
        dbg_struct, dbg = None, None
        if debug:
            B, S, H, W = desc.B, desc.S, desc.H, desc.W
            dbg_struct = L.SfmDebug()
            dbg = dict(P=[], u0=[], v0=[], inb=[])
            for s in range(self.n_scales):
                h, w = self._step_hw(desc, s)
                dbg['P'].append(D.empty(tgt, (B, S, 3, h, w)))
                dbg['u0'].append(D.empty(tgt, (B, S, h, w), 'int32'))
                dbg['v0'].append(D.empty(tgt, (B, S, h, w), 'int32'))
                dbg['inb'].append(D.empty(tgt, (B, S, h, w), 'uint8'))
                dbg_struct.P[s], dbg_struct.u0[s] = D.ptr(dbg['P'][s]), D.ptr(dbg['u0'][s])
                dbg_struct.v0[s], dbg_struct.inb[s] = D.ptr(dbg['v0'][s]), D.ptr(dbg['inb'][s])
        L.check(self._lib.sfm_loss_forward(C.byref(desc), C.byref(inp), _vp(losses),
                                           C.byref(dbg_struct) if debug else None,
                                           self._workspace(desc, tgt), C.c_void_p(D.current_stream(tgt))))
        return (losses, dbg) if debug else losses

    def backward(self, tgt, src, intrinsics, disps, poses, logits=None, gy=None, proj=None, kinv=None,
                 intrinsics_grad=True):
        """Recomputing backward: -> dict(gdisps, gposes, glogits).  gy: device scalar or None (= 1).
        With the operator's intrinsics_grad the dict also holds gintrinsics (None when `intrinsics_grad` is False)."""
        want_k = self._want_intrinsics_grad(intrinsics_grad, proj, kinv)
        desc, inp = self._pack(tgt, src, intrinsics, disps, poses, logits, proj, kinv)
        g, out = self._alloc_grads(desc, tgt)
        L.check(self._lib.sfm_loss_backward(C.byref(desc), C.byref(inp), _vp(gy), C.byref(g),
                                            self._workspace(desc, tgt), C.c_void_p(D.current_stream(tgt))))
        self._intrinsics_grad(desc, inp, tgt, out, want_k)
        return out

    def build_pyramid(self, tgt, src):
        """F.resize_images pyramid of this batch (base_model.py:70-72; scales >= 1, scale 0 is the input itself) into
        the operator's workspace.  It depends on the input images alone, so it can be issued as soon as the batch is
        on the device; the following forward_backward(..., reuse_pyramid=True) -- with the SAME tgt / src tensors,
        which it still reads at scale 0 -- then only builds the projection tables.
        May be issued on a side stream: the operator records an event here that the reusing loss call waits for,
        and the loss call records one that the next build_pyramid waits for.  The workspace is a single buffer, so
        one batch is in flight per operator; use one operator per in-flight batch to overlap more."""
        B, S, _, H, W = src.shape
        D.check_array(tgt, 'tgt_img', (B, 3, H, W))
        D.check_array(src, 'src_imgs', (B, S, 3, H, W))
        desc = self._desc(B, S, H, W)
        D.wait_event(tgt, self._ev_loss)           # a loss call on another stream may still be reading the workspace
        L.check(self._lib.sfm_pyramid(C.byref(desc), _vp(tgt), _vp(src), self._workspace(desc, tgt),
                                      C.c_void_p(D.current_stream(tgt))))
        self._ev_pyramid = D.record_event(tgt)

    def forward_backward(self, tgt, src, intrinsics, disps, poses, logits=None, proj=None, kinv=None, reuse_pyramid=False,
                         peer=None, image_grads=('tgt', 'src'), intrinsics_grad=True, snippet_weights=None,
                         pixel_weights=None, src_disps=None):
        """Single fused pass: -> (losses (5,), dict(gdisps, gposes, glogits)) for upstream gradient 1.
        reuse_pyramid: the workspace already holds this batch's pyramid (build_pyramid).
        peer: a distributed.PeerLossSum -- the batch is sharded by snippet over several GPUs (B_global set) and the
        epilogue kernel completes the five losses across the ranks over NVLink peer memory.
        With the operator's image_grads the dict also holds gtgt and gsrc (None for an image left out of
        `image_grads`, a subset of ('tgt', 'src'); an empty one runs the plain pass).
        With the operator's intrinsics_grad the dict also holds gintrinsics (None when `intrinsics_grad` is False).
        With the operator's snippet_terms: snippet_weights (B,) (None = all 1; under peer the local shard's) weight the
        snippets, the losses are sum_b w_b * l_b, every gradient is that of their total, and the dict also holds
        snippet_losses (B,5), this shard's rows l_b.
        With the operator's pixel_terms: pixel_weights (list of n_scales (B,S,h,w) or None entries) weight the
        photometric terms per (pixel, source), and the dict also holds pixel_losses, the maps d total / d weights
        (this shard's, under peer).
        With the operator's min_reprojection the dict also holds selection (list of n_scales (B,h,w) int8; this
        shard's, under peer).
        With the operator's geometry_consistency: src_disps (list of n_scales (B,S,h,w) activated source disparities) is
        required, and the dict also holds geometry_diff (the D_diff maps, this shard's under peer) and gsrc_disps (the
        gradient w.r.t. src_disps); with valid_mean also valid_masks and valid_counts."""
        if src_disps is not None and not self.geometry_consistency:
            raise ValueError('src_disps needs ViewSynthesisLoss(geometry_consistency=True)')
        want_k = self._want_intrinsics_grad(intrinsics_grad, proj, kinv)
        desc, inp = self._pack(tgt, src, intrinsics, disps, poses, logits, proj, kinv)
        if reuse_pyramid:
            desc.flags |= L.SFM_FLAG_REUSE_PYRAMID
            D.wait_event(tgt, self._ev_pyramid)     # build_pyramid may have run on another stream
        g, out = self._alloc_grads(desc, tgt)
        losses = D.empty(tgt, (5,))
        terms, rows = self._snippet_terms(desc, tgt, snippet_weights)
        if rows is not None:
            out['snippet_losses'] = rows
        pt, maps = self._pixel_terms(desc, tgt, pixel_weights)
        if maps is not None:
            out['pixel_losses'] = maps
        if self.geometry_consistency:
            ge, out['geometry_diff'], out['gsrc_disps'] = self._geometry(desc, tgt, src_disps, True)
            vm, masks, counts = self._valid_mean(desc, tgt)
            if vm is not None:
                if peer is not None:
                    raise ValueError('valid_mean is not supported with a peer (the counts are batch-global)')
                out['valid_masks'], out['valid_counts'] = masks, counts
            self._run_geometry(desc, inp, terms, ge, vm, losses, g, tgt, peer.handle if peer is not None else None)
            self._intrinsics_grad(desc, inp, tgt, out, want_k)
            if self._ev_pyramid is not None:
                self._ev_loss = D.record_event(tgt)
            return losses, out
        if self.min_reprojection:
            mr, out['selection'] = self._min_reprojection(desc, tgt)
            L.check(self._lib.sfm_loss_min_reprojection(C.byref(desc), C.byref(inp), C.byref(terms) if terms else None,
                                                        C.byref(mr), _vp(losses), C.byref(g), self._workspace(desc, tgt),
                                                        peer.handle if peer is not None else None,
                                                        C.c_void_p(D.current_stream(tgt))))
            self._intrinsics_grad(desc, inp, tgt, out, want_k)
            if self._ev_pyramid is not None:
                self._ev_loss = D.record_event(tgt)
            return losses, out
        ig = None
        want = set(image_grads) if self.image_grads else set()
        if want:
            if not want <= {'tgt', 'src'}:
                raise ValueError("image_grads must be a subset of ('tgt', 'src')")
            out['gtgt'] = D.empty(tgt, (desc.B, 3, desc.H, desc.W)) if 'tgt' in want else None
            out['gsrc'] = D.empty(tgt, (desc.B, desc.S, 3, desc.H, desc.W)) if 'src' in want else None
            ig = L.SfmImageGrads(_vp(out['gtgt']), _vp(out['gsrc']))
        # one entry point for every combination of image gradients, peer sum, snippet and per-pixel terms
        L.check(self._lib.sfm_loss_weighted(C.byref(desc), C.byref(inp), C.byref(terms) if terms else None,
                                            C.byref(pt) if pt else None, _vp(losses), C.byref(g), C.byref(ig) if ig else None,
                                            self._workspace(desc, tgt), peer.handle if peer is not None else None,
                                            C.c_void_p(D.current_stream(tgt))))
        self._intrinsics_grad(desc, inp, tgt, out, want_k)
        if self._ev_pyramid is not None:
            self._ev_loss = D.record_event(tgt)
        return losses, out

    def scale_grads(self, grads, gy, B, S, H, W):
        """grads *= gy (device scalar); a no-op on the device when gy == 1.  gsrc_disps (geometry_consistency) is not
        touched: it has the shape of a per-pixel map and is scaled by the caller as the maps are."""
        gp_shape = tuple(grads['gposes'].shape)
        desc = self._desc(B, S, H, W, 0, int(gp_shape[2] * (gp_shape[3] if len(gp_shape) > 3 else 1)) if self.raw_pose else 0)
        g = L.SfmGrads()
        for s in range(self.n_scales):
            g.gdisps[s] = D.ptr(grads['gdisps'][s])
            if self.use_exp:
                g.glogits[s] = D.ptr(grads['glogits'][s])
        g.gposes = D.ptr(grads['gposes'])
        L.check(self._lib.sfm_scale_grads(C.byref(desc), _vp(gy), C.byref(g),
                                          C.c_void_p(D.current_stream(grads['gposes']))))
        if grads.get('gtgt') is not None or grads.get('gsrc') is not None:
            ig = L.SfmImageGrads(_vp(grads.get('gtgt')), _vp(grads.get('gsrc')))
            L.check(self._lib.sfm_scale_image_grads(C.byref(desc), _vp(gy), C.byref(ig),
                                                    C.c_void_p(D.current_stream(grads['gposes']))))
        if grads.get('gintrinsics') is not None:
            L.check(self._lib.sfm_scale_intrinsics_grad(C.byref(desc), _vp(gy), _vp(grads['gintrinsics']),
                                                        C.c_void_p(D.current_stream(grads['gposes']))))
        return grads

    def pyramid(self, tgt, src):
        """F.resize_images pyramid (base_model.py:70-72) -> lists of (B,3,h,w) and (B,S,3,h,w)."""
        B, S, _, H, W = src.shape
        D.check_array(tgt, 'tgt_img', (B, 3, H, W))
        D.check_array(src, 'src_imgs', (B, S, 3, H, W))
        desc = self._desc(B, S, H, W)
        ws = self._workspace(desc, tgt)
        st = C.c_void_p(D.current_stream(tgt))
        L.check(self._lib.sfm_pyramid(C.byref(desc), _vp(tgt), _vp(src), ws, st))
        tp, sp = [tgt], [src]                     # scale 0 is the identity of resize_images: the inputs themselves
        for s in range(1, self.n_scales):
            t = D.empty(tgt, (B, 3, H >> s, W >> s))
            r = D.empty(tgt, (B, S, 3, H >> s, W >> s))
            L.check(self._lib.sfm_pyramid_export(C.byref(desc), ws, s, _vp(t), _vp(r), st))
            tp.append(t)
            sp.append(r)
        return tp, sp

    def build_tables(self, poses, intrinsics, H, W):
        """proj_tgt_to_src (transform.py:64-91) + batch_inv(K) (:105) on the device."""
        B, S = poses.shape[:2]
        desc = self._desc(B, S, H, W)
        proj = D.empty(poses, (B, S, self.n_scales, 3, 4))
        kinv = D.empty(poses, (B, self.n_scales, 3, 3))
        L.check(self._lib.sfm_build_tables(C.byref(desc), _vp(poses), _vp(intrinsics), _vp(proj), _vp(kinv),
                                           C.c_void_p(D.current_stream(poses))))
        return proj, kinv


def draw_augmentation(H, W, rng=None):
    """The random numbers of data_augmentation (datasets/kitti/kitti_raw_transformed.py:23-74), drawn in the
    reference's order from `rng` (default: the global numpy RNG the reference uses): scaling pair (:34),
    crop offsets (:49-50), flip (:64).  -> dict for ingest_u8."""
    import numpy as np
    rng = rng or np.random
    scaling = rng.uniform(1, 1.15, 2)
    x_scaling, y_scaling = scaling[0], scaling[1]
    out_h, out_w = int(H * y_scaling), int(W * x_scaling)
    off_y = int(rng.randint(0, out_h - H + 1))
    off_x = int(rng.randint(0, out_w - W + 1))
    flip = bool(rng.rand() < 0.5)
    return dict(out_h=out_h, out_w=out_w, off_y=off_y, off_x=off_x, flip=flip, x_scaling=float(x_scaling),
                y_scaling=float(y_scaling))


def ingest_u8(frames, K, aug=None, n_scales=N_SCALES):
    """Decoded uint8 frames -> what SFMLearner.__call__ receives, in one device gather:
    load_as_float_norm (datasets/kitti/kitti_raw_dataset.py:12-14), data_augmentation and
    get_multi_scale_intrinsics (datasets/kitti/kitti_raw_transformed.py:23-93).

    frames (B, 1+S, H, W, 3) uint8 device array (frame 0 = target); K (B,3,3); aug: list of B dicts from
    draw_augmentation, or None (no augmentation).  -> tgt (B,3,H,W), src (B,S,3,H,W), intrinsics (B,n_scales,3,3)."""
    if len(frames.shape) != 5 or frames.shape[4] != 3:
        raise ValueError('frames must be (B, 1+S, H, W, 3) uint8')
    B, n, H, W, _ = [int(v) for v in frames.shape]
    S = n - 1
    D.check_array(frames, 'frames', (B, n, H, W, 3), 'uint8')
    D.check_array(K, 'K', (B, 3, 3))
    aug_dev = None
    if aug is not None:
        if len(aug) != B:
            raise ValueError('aug must hold one entry per snippet')
        arr = (L.SfmAugment * B)()
        for b, a in enumerate(aug):
            if not (H <= a['out_h'] and W <= a['out_w'] and 0 <= a['off_y'] <= a['out_h'] - H and 0 <= a['off_x'] <= a['out_w'] - W):
                raise ValueError('aug[%d]: crop window outside the rescaled image' % b)
            arr[b] = L.SfmAugment(a['out_h'], a['out_w'], a['off_y'], a['off_x'], 1 if a['flip'] else 0, 0,
                                  a['x_scaling'], a['y_scaling'])
        aug_dev = D.from_host_bytes(frames, arr)
    tgt = D.empty(K, (B, 3, H, W))
    src = D.empty(K, (B, S, 3, H, W))
    Ks = D.empty(K, (B, n_scales, 3, 3))
    L.check(L.load().sfm_ingest_u8(B, S, H, W, n_scales, _vp(frames), _vp(K), _vp(aug_dev), _vp(tgt), _vp(src), _vp(Ks),
                                   C.c_void_p(D.current_stream(K))))
    return tgt, src, Ks


def evaluate_depth_batch(pred_depth, gt_depth, mask, min_depth, max_depth):
    """One iteration of evaluate_depth's loop (evaluate.py:94-103) + compute_depth_errors
    (kitti_eval/depth_util.py:6-22) on the device: pred_depth (B,1,h,w), gt_depth (B,Hg,Wg), mask (B,Hg,Wg) uint8.
    -> device float array (8,): abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, scale_factor."""
    B, _, h, w = [int(v) for v in pred_depth.shape]
    Hg, Wg = int(gt_depth.shape[1]), int(gt_depth.shape[2])
    D.check_array(pred_depth, 'pred_depth', (B, 1, h, w))
    D.check_array(gt_depth, 'gt_depth', (B, Hg, Wg))
    D.check_array(mask, 'mask', (B, Hg, Wg), 'uint8')
    lib = L.load()
    scratch = D.empty(pred_depth, (lib.sfm_eval_depth_scratch_bytes(B, Hg, Wg) + 256,), 'uint8')
    sp = C.c_void_p((D.ptr(scratch) + 255) // 256 * 256)
    out = D.empty(pred_depth, (8,))
    L.check(lib.sfm_eval_depth(B, h, w, Hg, Wg, _vp(pred_depth), _vp(gt_depth), _vp(mask), float(min_depth), float(max_depth),
                               _vp(out), sp, C.c_void_p(D.current_stream(pred_depth))))
    return out


def disp_activation(x, want_dact=False):
    """DISP_SCALING * F.sigmoid(x) + MIN_DISP (models/disp_net.py:7-8,104) as a stage, with the device code
    the fused kernels inline under `raw_disp_scales`.  -> disp [, d disp / d x]."""
    D.check_array(x, 'x')
    n = 1
    for k in x.shape:
        n *= int(k)
    disp = D.empty(x, tuple(x.shape))
    dact = D.empty(x, tuple(x.shape)) if want_dact else None
    L.check(L.load().sfm_disp_activation(n, _vp(x), _vp(disp), _vp(dact), C.c_void_p(D.current_stream(x))))
    return (disp, dact) if want_dact else disp


def upsample_disparity(x, H, W):
    """F.interpolate(x, size=(H, W), mode='bilinear', align_corners=False) of disparity maps x (N,1,h,w) in the fp32
    arithmetic the full-resolution multi-scale step uses (the same device code).  -> (N,1,H,W)."""
    D.check_array(x, 'x')
    if len(x.shape) != 4 or x.shape[1] != 1:
        raise ValueError('x must be (N, 1, h, w)')
    N, _, h, w = [int(v) for v in x.shape]
    y = D.empty(x, (N, 1, int(H), int(W)))
    L.check(L.load().sfm_upsample_disparity(N, h, w, int(H), int(W), _vp(x), _vp(y), C.c_void_p(D.current_stream(x))))
    return y


def pose_reduce(x, n_sources):
    """0.01 * F.mean(poseout, (2, 3)) split into n_sources 6-DoF vectors (models/pose_net.py:52-54):
    x (B, 6*S, h', w') -> (B, S, 6)."""
    D.check_array(x, 'x')
    B = int(x.shape[0])
    if x.shape[1] != 6 * n_sources:
        raise ValueError('x.shape[1] must be 6 * n_sources')
    hw = 1
    for k in x.shape[2:]:
        hw *= int(k)
    out = D.empty(x, (B, n_sources, 6))
    L.check(L.load().sfm_pose_reduce(B, n_sources, hw, _vp(x), _vp(out), C.c_void_p(D.current_stream(x))))
    return out


def projective_inverse_warp(imgs, depthes, poses, K, proj=None, kinv=None, return_indices=False):
    """models/transform.py:156-165.

    imgs (N,3,H,W); depthes (N,H*W) -- or (N,3,H*W) as the reference passes it, of which row 0 is used
    (the three rows are a broadcast, base_model.py:81-84); poses (N,6); K (N,3,3).
    Returns the warped images (N,3,H,W) [, u0, v0 (int32) and the in-bounds mask (uint8)].
    """
    lib = L.load()
    N, _, H, W = imgs.shape
    D.check_array(imgs, 'imgs', (N, 3, H, W))
    if len(depthes.shape) == 3:
        if tuple(depthes.shape) != (N, 3, H * W):
            raise ValueError('depthes: expected (N,3,H*W) or (N,H*W), got %s' % (tuple(depthes.shape),))
        depthes = depthes[:, 0]
        if not (depthes.is_contiguous() if D.is_torch(depthes) else depthes.flags.c_contiguous):
            depthes = depthes.contiguous() if D.is_torch(depthes) else depthes.copy()
    D.check_array(depthes, 'depthes', (N, H * W))
    D.check_array(poses, 'poses', (N, 6))
    D.check_array(K, 'K', (N, 3, 3))
    out = D.empty(imgs, (N, 3, H, W))
    u0 = v0 = inb = None
    if return_indices:
        u0, v0 = D.empty(imgs, (N, H, W), 'int32'), D.empty(imgs, (N, H, W), 'int32')
        inb = D.empty(imgs, (N, H, W), 'uint8')
    L.check(lib.sfm_warp_forward(N, H, W, _vp(imgs), _vp(depthes), _vp(poses), _vp(K), _vp(proj), _vp(kinv),
                                 _vp(out), _vp(u0), _vp(v0), _vp(inb), C.c_void_p(D.current_stream(imgs))))
    return (out, u0, v0, inb) if return_indices else out


def projective_inverse_warp_backward(imgs, depthes, poses, K, gy, want_gimgs=False):
    """Backward of projective_inverse_warp: -> (gdepth (N,H*W), gposes (N,6)[, gimgs])."""
    lib = L.load()
    N, _, H, W = imgs.shape
    D.check_array(imgs, 'imgs', (N, 3, H, W))
    D.check_array(depthes, 'depthes', (N, H * W))
    D.check_array(poses, 'poses', (N, 6))
    D.check_array(K, 'K', (N, 3, 3))
    D.check_array(gy, 'gy', (N, 3, H, W))
    gdepth, gposes = D.empty(imgs, (N, H * W)), D.empty(imgs, (N, 6))
    gimgs = D.empty(imgs, (N, 3, H, W)) if want_gimgs else None
    scratch = D.empty(imgs, (lib.sfm_warp_backward_scratch_bytes(N) + 8,), 'uint8')
    L.check(lib.sfm_warp_backward(N, H, W, _vp(imgs), _vp(depthes), _vp(poses), _vp(K), _vp(gy), _vp(gdepth),
                                  _vp(gposes), _vp(gimgs), _vp(scratch), C.c_void_p(D.current_stream(imgs))))
    return (gdepth, gposes, gimgs) if want_gimgs else (gdepth, gposes)


class SpatialTransformerSamplerInterp(object):
    """models/spational_transformer_sampler_interp.py:9-149 with the old-style chainer.Function method
    names (forward_gpu / backward_gpu on tuples of device arrays)."""

    def check_type_forward(self, x, grid):
        # spational_transformer_sampler_interp.py:11-24
        if len(x.shape) != 4 or len(grid.shape) != 4:
            raise TypeError('x and grid must be 4-dimensional')
        if grid.shape[1] != 2:
            raise TypeError('grid.shape[1] must be 2')
        if x.shape[0] != grid.shape[0]:
            raise TypeError('x and grid must have the same batch size')
        D.check_array(x, 'x')
        D.check_array(grid, 'grid')

    def forward_gpu(self, inputs):
        x, grid = inputs
        self.check_type_forward(x, grid)
        B, Cc, H, W = x.shape
        oH, oW = grid.shape[2:]
        y = D.empty(x, (B, Cc, oH, oW))
        L.check(L.load().sfm_sampler_interp_forward(B, Cc, H, W, oH, oW, _vp(x), _vp(grid), _vp(y),
                                                    C.c_void_p(D.current_stream(x))))
        return y,

    def backward_gpu(self, inputs, grad_outputs):
        x, grid = inputs
        gy, = grad_outputs
        self.check_type_forward(x, grid)
        B, Cc, H, W = x.shape
        oH, oW = grid.shape[2:]
        D.check_array(gy, 'gy', (B, Cc, oH, oW))
        gx = D.empty(x, (B, Cc, H, W))
        ggrid = D.empty(x, (B, 2, oH, oW))
        L.check(L.load().sfm_sampler_interp_backward(B, Cc, H, W, oH, oW, _vp(x), _vp(grid), _vp(gy), _vp(gx),
                                                     _vp(ggrid), C.c_void_p(D.current_stream(x))))
        return gx, ggrid

    def forward_cpu(self, inputs):
        raise RuntimeError('SpatialTransformerSamplerInterp: no CPU path in the B200 build')

    backward_cpu = forward_cpu

    def __call__(self, x, grid):
        return self.forward_gpu((x, grid))[0]


def spatial_transformer_sampler_interp(x, grid, **kwargs):
    """spational_transformer_sampler_interp.py:152-159 (forward only; see the class for backward)."""
    if kwargs:
        raise TypeError('unexpected keyword arguments: %s' % sorted(kwargs))
    return SpatialTransformerSamplerInterp()(x, grid)
