// api.cu -- extern "C" entry points of libsfmloss.so (see include/sfmloss.h for the contract and the
// reference interfaces each one replaces).
#include <stdarg.h>
#include <string.h>

#include <new>
#include <vector>

#include "common.cuh"
#include "kernels.h"

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void sfm_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* sfm_last_error(void) { return g_err; }

thread_local cudaEvent_t sfm_ev_start = nullptr, sfm_ev_stop = nullptr;   // recorded around the fused kernel (fused_loss.cu)
extern "C" int sfm_set_kernel_events(void* start_event, void* stop_event) {
  sfm_ev_start = (cudaEvent_t)start_event;
  sfm_ev_stop = (cudaEvent_t)stop_event;
  return 0;
}
extern "C" int sfm_version(void) { return SFM_VERSION; }

int sfm_validate_desc(const SfmDesc* d) {
  if (!d) { sfm_set_error("SfmDesc is NULL"); return SFM_E_NULL_POINTER; }
  if (d->B < 1 || d->S < 1 || d->S > SFM_MAX_SOURCES || d->n_scales < 1 || d->n_scales > SFM_MAX_SCALES) {
    sfm_set_error("invalid SfmDesc: B=%d S=%d (1..%d) n_scales=%d (1..%d)", d->B, d->S, SFM_MAX_SOURCES, d->n_scales, SFM_MAX_SCALES);
    return SFM_E_INVALID_DESC;
  }
  if (d->B_global != 0 && d->B_global < d->B) {
    sfm_set_error("invalid SfmDesc: B_global=%d < B=%d", d->B_global, d->B);
    return SFM_E_INVALID_DESC;
  }
  const int hs = d->H >> (d->n_scales - 1), ws = d->W >> (d->n_scales - 1);
  if (d->H < 2 || d->W < 2 || hs < 4 || ws < 4) {
    // resize_images needs >= 2 input rows/cols; the smoothness means need (h-2)*(w-2) > 0 at every scale; and
    // with >= 4 rows/cols every tap of an out-of-view pixel (x2 rule) lies in the sampler's zero padding
    sfm_set_error("invalid shape: H=%d W=%d give %dx%d at the coarsest of %d scales (need >= 4x4)", d->H, d->W, hs, ws, d->n_scales);
    return SFM_E_INVALID_SHAPE;
  }
  if ((long long)d->B * (1 + d->S) * d->H * d->W >= (1ll << 31)) {
    sfm_set_error("invalid shape: B*(1+S)*H*W exceeds 2^31 pixels");
    return SFM_E_INVALID_SHAPE;
  }
  if (d->raw_disp_scales >> d->n_scales) {
    sfm_set_error("invalid SfmDesc: raw_disp_scales=0x%x names a scale >= n_scales=%d", d->raw_disp_scales, d->n_scales);
    return SFM_E_INVALID_DESC;
  }
  if (d->raw_pose_hw < 0 || d->raw_pose_hw > 128) {
    sfm_set_error("unsupported SfmDesc: raw_pose_hw=%d (0 = 6-DoF vectors, 1..128 = positions of the poseout map)", d->raw_pose_hw);
    return SFM_E_UNSUPPORTED;
  }
  if (d->raw_pose_hw > 0 && (d->flags & SFM_FLAG_TABLES_PROVIDED)) {
    sfm_set_error("unsupported SfmDesc: raw_pose_hw > 0 together with SFM_FLAG_TABLES_PROVIDED (the tables are built from the reduced poses)");
    return SFM_E_UNSUPPORTED;
  }
  if ((d->flags & SFM_FLAG_EDGE_MEAN_ABS) && !(d->flags & SFM_FLAG_EDGE_AWARE_SMOOTH)) {
    sfm_set_error("invalid SfmDesc: SFM_FLAG_EDGE_MEAN_ABS needs SFM_FLAG_EDGE_AWARE_SMOOTH");
    return SFM_E_INVALID_DESC;
  }
  const unsigned inv = (d->flags & SFM_FLAG_POSE_INVERT_MASK) >> SFM_FLAG_POSE_INVERT_SHIFT;
  if (inv && !(d->flags & SFM_FLAG_AXISANGLE_POSE)) {
    sfm_set_error("invalid SfmDesc: pose inversion bits 0x%x need SFM_FLAG_AXISANGLE_POSE", inv);
    return SFM_E_INVALID_DESC;
  }
  if (inv >> d->S) {
    sfm_set_error("invalid SfmDesc: pose inversion bits 0x%x name a source >= S=%d", inv, d->S);
    return SFM_E_INVALID_DESC;
  }
  if (!(d->smooth_reg == d->smooth_reg) || !(d->exp_reg == d->exp_reg) || !(d->ssim_rate == d->ssim_rate)) {
    sfm_set_error("invalid SfmDesc: NaN loss weight");
    return SFM_E_INVALID_DESC;
  }
  return 0;
}

extern "C" size_t sfm_workspace_bytes(const SfmDesc* desc) {
  if (sfm_validate_desc(desc) != 0) return 0;
  SfmWsLayout L;
  sfm_ws_layout(desc, &L);
  return L.total;
}

// ------------------------------------------------------------------------------------------------
// common driver
// ------------------------------------------------------------------------------------------------
namespace {

struct Modes {
  bool use_exp, use_ssim, use_smooth;
};

// Python truthiness of the reference's flags (base_model.py:75,86,103,112): 0 / 0.0 disable a term;
// SSIM sits in the else-branch of the explainability test (:103-115).
Modes modes_of(const SfmDesc* d) {
  Modes m;
  m.use_exp = d->exp_reg != 0.f;
  m.use_ssim = !m.use_exp && d->ssim_rate != 0.f;
  m.use_smooth = d->smooth_reg != 0.f;
  return m;
}

int check_inputs(const SfmDesc* d, const SfmInputs* in, bool need_images) {
  if (!in) { sfm_set_error("SfmInputs is NULL"); return SFM_E_NULL_POINTER; }
  const Modes m = modes_of(d);
  if (need_images && (!in->tgt || !in->src)) { sfm_set_error("tgt/src image pointer is NULL"); return SFM_E_NULL_POINTER; }
  if (!in->intrinsics || !in->poses) { sfm_set_error("intrinsics/poses pointer is NULL"); return SFM_E_NULL_POINTER; }
  for (int s = 0; s < d->n_scales; ++s) {
    if (!in->disps[s]) { sfm_set_error("disps[%d] is NULL", s); return SFM_E_NULL_POINTER; }
    if (m.use_exp && !in->logits[s]) { sfm_set_error("exp_reg > 0 but logits[%d] is NULL", s); return SFM_E_NULL_POINTER; }
  }
  if ((d->flags & SFM_FLAG_TABLES_PROVIDED) && (!in->proj || !in->kinv)) {
    sfm_set_error("SFM_FLAG_TABLES_PROVIDED set but proj/kinv is NULL");
    return SFM_E_NULL_POINTER;
  }
  return 0;
}

int check_grads(const SfmDesc* d, const SfmGrads* g) {
  if (!g) { sfm_set_error("SfmGrads is NULL"); return SFM_E_NULL_POINTER; }
  const Modes m = modes_of(d);
  if (!g->gposes) { sfm_set_error("gposes is NULL"); return SFM_E_NULL_POINTER; }
  for (int s = 0; s < d->n_scales; ++s) {
    if (!g->gdisps[s]) { sfm_set_error("gdisps[%d] is NULL", s); return SFM_E_NULL_POINTER; }
    if (m.use_exp && !g->glogits[s]) { sfm_set_error("exp_reg > 0 but glogits[%d] is NULL", s); return SFM_E_NULL_POINTER; }
  }
  return 0;
}

// Parameters of the prologue kernel.  It builds the pyramid of (tgt, src) into the workspace when tgt is given, the
// projection tables of (poses, intrinsics) when proj_out is given, and with `step` (a loss call) also resets the
// workspace's fp64 cells and stores the reduced pose vectors there.
SfmPrepParams prep_params(const SfmDesc* d, int band, char* ws, const float* tgt, const float* src, const float* intrinsics,
                          const float* poses, float* proj_out, float* kinv_out, bool step) {
  SfmWsLayout L;
  sfm_ws_layout(d, &L);
  SfmPrepParams p{};
  p.B = d->B; p.S = d->S; p.H = d->H; p.W = d->W; p.ns = d->n_scales;
  p.band = band;
  p.do_pyramid = tgt ? 1 : 0;
  p.build_tables = proj_out ? 1 : 0;
  p.tgt = tgt; p.src = src; p.intrinsics = intrinsics; p.poses = poses;
  if (tgt)
    for (int s = 0; s < d->n_scales; ++s) {
      p.tgt_pyr[s] = (float*)(ws + L.off_tgt[s]);
      p.src_pyr[s] = (float*)(ws + L.off_src[s]);
    }
  p.proj_out = proj_out;
  p.kinv_out = kinv_out;
  p.raw_pose_hw = d->raw_pose_hw;
  if (step) {
    p.acc = (double*)(ws + L.off_acc);
    p.n_acc = (int)L.acc_doubles;
    p.posevec_out = (float*)(ws + L.off_posevec);
  }
  return p;
}

// SM count of the device, queried once
int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = SFM_REF_SMS;
  }
  return n;
}

int run_loss(const SfmDesc* d, const SfmInputs* in, float* losses_out, const SfmGrads* grads, const float* gy,
             const SfmDebug* dbg, void* workspace, cudaStream_t st, const SfmPeerDev* peer = nullptr,
             const SfmImageGrads* ig = nullptr, const SfmSnippetTerms* snip = nullptr, const SfmPixelTerms* pix = nullptr,
             const SfmMinReprojection* mr = nullptr, const SfmGeometry* geo = nullptr, const SfmValidMean* vm = nullptr) {
  int rc = sfm_validate_desc(d);
  if (rc) return rc;
  // SFM_FLAG_BORDER_PADDING runs the per-pixel instances (weights and maps NULL unless the caller passed them)
  const bool border = (d->flags & SFM_FLAG_BORDER_PADDING) != 0;
  if (border && (modes_of(d).use_exp || ig || dbg)) {
    sfm_set_error("unsupported: SFM_FLAG_BORDER_PADDING together with %s", modes_of(d).use_exp ? "the explainability branch (exp_reg != 0)"
                  : ig ? "image gradients" : "debug dumps");
    return SFM_E_UNSUPPORTED;
  }
  const bool reuse = (d->flags & SFM_FLAG_REUSE_PYRAMID) != 0;
  rc = check_inputs(d, in, true);      // the images are always needed: scale 0 is read from the caller's tensors
  if (rc) return rc;
  if (grads && (rc = check_grads(d, grads))) return rc;
  if (!workspace) { sfm_set_error("workspace is NULL"); return SFM_E_NULL_POINTER; }
  if (((uintptr_t)workspace & 255) != 0) { sfm_set_error("workspace must be 256-byte aligned"); return SFM_E_INVALID_DESC; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    sfm_set_error("no CUDA device: libsfmloss has no CPU fallback");
    return SFM_E_NO_DEVICE;
  }
  const Modes m = modes_of(d);
  const bool fr = sfm_full_res(d);
  if (fr && m.use_exp) {
    sfm_set_error("unsupported: SFM_FLAG_FULL_RES_MULTISCALE together with the explainability branch (exp_reg != 0): the logits "
                  "live at scale resolution");
    return SFM_E_UNSUPPORTED;
  }
  if (fr && ig) {
    sfm_set_error("unsupported: image gradients together with SFM_FLAG_FULL_RES_MULTISCALE");
    return SFM_E_UNSUPPORTED;
  }
  int mode = 0;
  if (m.use_exp) mode |= SFM_MODE_EXP;
  if (m.use_ssim) mode |= SFM_MODE_SSIM;
  if (m.use_smooth) mode |= SFM_MODE_SMOOTH;
  if (grads) mode |= SFM_MODE_GRAD;
  if (dbg) mode |= SFM_MODE_DEBUG;
  if (ig) mode |= SFM_MODE_IMG;
  if (pix) mode |= SFM_MODE_PIX;
  if (mr) mode |= SFM_MODE_PIX | SFM_MODE_MINREP;
  if (border) mode |= SFM_MODE_PIX | SFM_MODE_BORDER;
  const bool self_mask = geo && geo->self_mask != 0;
  if (self_mask) mode |= SFM_MODE_PIX;             // the per-pixel instances with the mask planes as weights
  if (vm) mode |= SFM_MODE_PIX | SFM_MODE_CLAMP;   // the weight planes a M (B h w) / n, the clamped L1
  const SfmStepPlan plan = sfm_plan_step(d, mode, num_sms());
  SfmWsLayout L;
  sfm_ws_layout(d, &L);
  char* ws = (char*)workspace;
  SfmFusedParams p{};
  SfmSmoothParams sm = plan.smooth;
  p.B = d->B; p.S = d->S; p.ns = d->n_scales;
  const double Bg = (double)(d->B_global > 0 ? d->B_global : d->B);
  for (int s = 0; s < d->n_scales; ++s) {
    const int h = d->H >> s, w = d->W >> s;           // native size: the smoothness terms
    p.h[s] = h; p.w[s] = w;
    p.tgt_pl[s] = s == 0 ? in->tgt : (const float*)(ws + L.off_tgt[s]);
    p.src_pl[s] = s == 0 ? in->src : (const float*)(ws + L.off_src[s]);
    p.disp[s] = in->disps[s];
    p.logits[s] = m.use_exp ? in->logits[s] : nullptr;
    p.gdisp[s] = grads ? grads->gdisps[s] : nullptr;
    p.glogits[s] = (grads && m.use_exp) ? grads->glogits[s] : nullptr;
    const double wgt = (double)d->smooth_reg / (double)(1 << s);
    p.sm_dx2[s] = (float)(wgt / (Bg * h * (w - 2)));
    p.sm_mix[s] = (float)(wgt / (Bg * (h - 1) * (w - 1)));
    p.sm_dy2[s] = (float)(wgt / (Bg * (h - 2) * w));
    p.sm_ex[s] = (float)(wgt / (Bg * h * (w - 1)));
    p.sm_ey[s] = (float)(wgt / (Bg * (h - 1) * w));
    sm.disp[s] = p.disp[s];
    sm.gdisp[s] = p.gdisp[s];
    sm.k_dx2[s] = p.sm_dx2[s]; sm.k_mix[s] = p.sm_mix[s]; sm.k_dy2[s] = p.sm_dy2[s];
    if (dbg) {
      p.dbg_P[s] = dbg->P[s]; p.dbg_u0[s] = dbg->u0[s]; p.dbg_v0[s] = dbg->v0[s]; p.dbg_inb[s] = dbg->inb[s];
    }
    if (ig) {
      p.gtgt[s] = !ig->gtgt ? nullptr : s == 0 ? ig->gtgt : (float*)(ws + L.off_gtgt[s]);
      p.gsrc[s] = !ig->gsrc ? nullptr : s == 0 ? ig->gsrc : (float*)(ws + L.off_gsrc[s]);
    }
    if (pix) {
      p.pix_w[s] = pix->weights[s];
      p.pix_map[s] = pix->losses[s];
    }
    if (mr) p.pix_w[s] = (const float*)(ws + L.off_mrw[s]);   // the one-hot weights, made by the select kernel
    if (self_mask || vm) {
      // M = 1 - D_diff, made by the geometry forward kernel (valid-pixel means: a M (B h w) / n, by the normalise
      // kernel); the maps d total / d M feed its backward kernel
      p.pix_w[s] = (const float*)(ws + L.off_geow[s]);
      p.pix_map[s] = (grads && self_mask) ? (float*)(ws + L.off_geomap[s]) : nullptr;
    }
  }
  auto photometric_consts = [&](int s) {              // from the size of the photometric terms of scale s
    const int h = p.h[s], w = p.w[s];
    p.inv_n3[s] = (float)(1.0 / (Bg * 3.0 * h * w));
    p.inv_n1[s] = (float)(1.0 / (Bg * h * w));
    p.hwf[s] = (float)((w - 1) / 2.0);
    p.hhf[s] = (float)((h - 1) / 2.0);
  };
  for (int s = 0; s < d->n_scales; ++s) photometric_consts(s);
  const bool tables = (d->flags & SFM_FLAG_TABLES_PROVIDED) != 0;
  p.proj = tables ? in->proj : (const float*)(ws + L.off_proj);
  p.kinv = tables ? in->kinv : (const float*)(ws + L.off_kinv);
  p.intrinsics = fr ? (const float*)(ws + L.off_k0) : in->intrinsics;
  p.poses = d->raw_pose_hw > 0 ? (const float*)(ws + L.off_posevec) : in->poses;
  p.raw_pose_hw = d->raw_pose_hw;
  p.pose_flags = d->flags & (SFM_FLAG_AXISANGLE_POSE | SFM_FLAG_POSE_INVERT_MASK);
  p.raw_disp_mask = d->raw_disp_scales;
  p.gy = gy;
  p.acc = (double*)(ws + L.off_acc);
  p.losses_out = losses_out;
  p.peer = SfmPeerDev{};
  if (peer) p.peer = *peer;
  p.gposes = grads ? grads->gposes : nullptr;
  p.smooth_reg = d->smooth_reg;
  p.exp_reg = m.use_exp ? d->exp_reg : 0.f;
  p.ssim_rate = d->ssim_rate;     // enters `total` even when the SSIM term itself is skipped (base_model.py:117)
  p.use_smooth = m.use_smooth ? 1 : 0;
  p.edge_smooth = (d->flags & SFM_FLAG_EDGE_AWARE_SMOOTH) ? 1 : 0;
  // prologue kernel: pyramid + tables + cell reset and, in the same grid, the second-order smoothness tasks (the
  // edge-aware variant reads the pyramid and is launched by sfm_launch_fused after it)
  sm.gy = gy;
  sm.raw_disp_mask = d->raw_disp_scales;
  sm.part = (float*)(ws + L.off_smpart);
  p.sm_part = sm.part;
  p.n_sm_part = sm.n_ctas;
  if (snip) {
    // per-snippet terms: the smoothness tasks write per-task losses instead of CTA partials (the epilogue sums each
    // snippet's tasks), every other loss partial goes to its snippet's cells
    p.snip_w = snip->weights;
    p.snip_losses = snip->losses;
    p.snip_cell0 = (int)L.snip_cell0;
    p.n_sm_part = 0;
    sm.snip_w = snip->weights;
    sm.task_part = (float*)(ws + L.off_smtask);
    p.sm_part = sm.task_part;
    p.sm_hseg = sm.n_ctas > 0 ? sm.hseg : 0;
  }
  // SFM_FLAG_MEAN_NORM_SMOOTH: the smoothness writers leave the loss of every (snippet, scale) in fixed slots -- the
  // prologue's per-task losses, or the edge-aware kernel's per-CTA partials -- and the fix-up kernel writes the
  // normalised loss where the epilogue reads the smoothness: into the snippets' smooth cells, or as its partials
  const bool mean_norm = (d->flags & SFM_FLAG_MEAN_NORM_SMOOTH) && m.use_smooth;
  SfmMeanNorm mn{};
  if (mean_norm) {
    mn.B = d->B; mn.ns = d->n_scales;
    const int chunks = (d->H * d->W + 2047) / 2048;
    mn.chunks = chunks < SFM_MN_SLOTS ? chunks : SFM_MN_SLOTS;
    for (int s = 0; s < d->n_scales; ++s) {
      mn.h[s] = p.h[s]; mn.w[s] = p.w[s];
      mn.disp[s] = in->disps[s];
      mn.gdisp[s] = p.gdisp[s];
    }
    mn.raw_disp_mask = d->raw_disp_scales;
    mn.gy = gy;
    mn.snip_w = snip ? snip->weights : nullptr;
    mn.mean_part = (float*)(ws + L.off_mnmean);
    if (plan.edge_smooth) {
      mn.edge_slots = (float*)(ws + L.off_mnedge);
      mn.loss_part = mn.edge_slots;
      for (int s = 0; s < d->n_scales; ++s) {
        mn.loss_off[s] = s * SFM_MN_SLOTS;
        mn.loss_stride[s] = d->n_scales * SFM_MN_SLOTS;
        mn.loss_cnt[s] = sfm_edge_smooth_ctas(p.h[0] * p.w[0]);
      }
    } else {
      sm.task_part = (float*)(ws + L.off_smtask);
      mn.loss_part = sm.task_part;
      for (int s = 0; s < d->n_scales; ++s) {
        mn.loss_off[s] = sm.tile_begin[s];
        mn.loss_stride[s] = mn.loss_cnt[s] = sm.tiles_x[s] * sm.tiles_y[s];
      }
    }
    mn.snip_loss = (float*)(ws + L.off_mnloss);
    if (snip) {
      mn.snip_cell = p.acc + L.snip_cell0 + 1;
      p.sm_hseg = 0;
    } else {
      p.sm_part = mn.snip_loss;
      p.n_sm_part = d->B;
    }
  }
  // SFM_FLAG_FULL_RES_MULTISCALE: `native` keeps the scales as the smoothness kernels see them, and every scale >= 1 of
  // the photometric step becomes a full-resolution scale (the caller's images, U_s(d_s) and its gradient plane in the
  // workspace, the activation already applied by the upsample kernel); the tables are built from the K_0 copy
  SfmFusedParams native;
  SfmFullRes f{};
  if (fr) {
    native = p;
    f.B = d->B; f.ns = d->n_scales; f.H = d->H; f.W = d->W;
    f.raw_disp_mask = d->raw_disp_scales;
    f.intrinsics = in->intrinsics;
    f.k0 = (float*)(ws + L.off_k0);
    f.zero_gup = plan.accum ? 1 : 0;
    f.accum = plan.accum ? 1 : 0;
    for (int s = 1; s < d->n_scales; ++s) {
      f.h[s] = p.h[s]; f.w[s] = p.w[s];
      f.disp[s] = in->disps[s];
      f.gdisp[s] = p.gdisp[s];
      f.up[s] = (float*)(ws + L.off_up[s]);
      f.gup[s] = grads ? (float*)(ws + L.off_gup[s]) : nullptr;
      p.h[s] = d->H; p.w[s] = d->W;
      p.tgt_pl[s] = in->tgt;
      p.src_pl[s] = in->src;
      p.disp[s] = f.up[s];
      p.gdisp[s] = f.gup[s];
      photometric_consts(s);
    }
    p.raw_disp_mask = d->raw_disp_scales & 1u;
  }
  // under SFM_FLAG_FULL_RES_MULTISCALE only the edge-aware smoothness reads the pyramid
  const bool pyramid = !reuse && (!fr || plan.edge_smooth);
  SfmPrepParams pp = prep_params(d, plan.band, ws, pyramid ? in->tgt : nullptr, in->src, p.intrinsics, in->poses,
                                 tables ? nullptr : (float*)(ws + L.off_proj), (float*)(ws + L.off_kinv), true);
  pp.n_mix_region = plan.n_mix_region;
  if (ig && ig->gsrc) {
    // the march accumulates the source gradients with reductions: scale 0 and the workspace levels start at 0
    SFM_CUDA_CHECK(cudaMemsetAsync(ig->gsrc, 0, (size_t)d->B * d->S * 3 * d->H * d->W * sizeof(float), st));
    if (L.gsrc_bytes) SFM_CUDA_CHECK(cudaMemsetAsync(ws + L.off_gsrc[1], 0, L.gsrc_bytes, st));
  }
  SfmGeoArgs ga{};
  if (geo) {
    ga.geometry_reg = geo->geometry_reg;
    int nf = 0, nb = 0;
    for (int s = 0; s < SFM_MAX_SCALES; ++s) {
      ga.fwd_begin[s] = nf;
      ga.bwd_begin[s] = nb;
      if (s >= d->n_scales) continue;
      const long long plane = (long long)p.h[s] * p.w[s];
      const int per = (int)((plane + 255) / 256);
      nf += d->B * d->S * per;
      nb += d->B * per;
      ga.src_disps[s] = geo->src_disps[s];
      ga.diff_maps[s] = geo->diff_maps[s];
      ga.gsrc_disps[s] = grads ? geo->gsrc_disps[s] : nullptr;
      ga.mask[s] = (self_mask || vm) ? (float*)(ws + L.off_geow[s]) : nullptr;
      if (vm) {
        ga.vm_mask[s] = (uint8_t*)(ws + L.off_vmmask[s]);
        ga.vm_out[s] = vm->masks[s];
      }
      ga.map[s] = self_mask ? p.pix_map[s] : nullptr;
      // gsrc_disps is accumulated with fp32 reductions
      if (ga.gsrc_disps[s]) SFM_CUDA_CHECK(cudaMemsetAsync(ga.gsrc_disps[s], 0, (size_t)d->B * d->S * plane * sizeof(float), st));
    }
    ga.fwd_begin[SFM_MAX_SCALES] = nf;
    ga.bwd_begin[SFM_MAX_SCALES] = nb;
    if (vm) {
      ga.vm = 1;
      ga.automask = vm->automask != 0 ? 1 : 0;
      ga.self_mask = self_mask ? 1 : 0;
      ga.groups = vm->groups;
      ga.min_count = vm->min_count;
      ga.counts = (int*)(ws + L.off_vmcount);
      ga.counts_out = vm->counts;
      // the counts are reset inside the step (a memset node under graph capture)
      SFM_CUDA_CHECK(cudaMemsetAsync(ga.counts, 0, (size_t)d->n_scales * d->S * vm->groups * sizeof(int32_t), st));
    }
  }
  if (fr && (rc = sfm_launch_full_res_upsample(f, st))) return rc;
  rc = sfm_launch_prep(pp, &sm, (grads ? 2 : 1) + ((snip || mean_norm) ? 2 : 0), st, p.pose_flags);
  if (rc) return rc;
  SfmMinRepArgs a{};
  if (mr) {
    a.automask = mr->automask != 0 ? 1 : 0;
    for (int s = 0; s < d->n_scales; ++s) a.selection[s] = mr->selection[s];
  }
  rc = sfm_launch_fused(p, plan, st, mr ? &a : nullptr, fr ? &native : nullptr, mean_norm ? &mn : nullptr,
                        (d->flags & SFM_FLAG_EDGE_MEAN_ABS) != 0, geo ? &ga : nullptr);
  if (rc || !fr || !grads) return rc;
  return sfm_launch_full_res_adjoint(f, st);
}

}  // namespace

extern "C" int sfm_loss_forward(const SfmDesc* desc, const SfmInputs* in, float* losses_out, const SfmDebug* debug,
                                void* workspace, void* stream) {
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  return run_loss(desc, in, losses_out, nullptr, nullptr, debug, workspace, (cudaStream_t)stream);
}

extern "C" int sfm_loss_backward(const SfmDesc* desc, const SfmInputs* in, const float* gy, const SfmGrads* grads,
                                 void* workspace, void* stream) {
  if (!grads) { sfm_set_error("grads is NULL"); return SFM_E_NULL_POINTER; }
  return run_loss(desc, in, nullptr, grads, gy, nullptr, workspace, (cudaStream_t)stream);
}

extern "C" int sfm_loss_forward_backward(const SfmDesc* desc, const SfmInputs* in, float* losses_out,
                                         const SfmGrads* grads, void* workspace, void* stream) {
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  if (!grads) { sfm_set_error("grads is NULL"); return SFM_E_NULL_POINTER; }
  return run_loss(desc, in, losses_out, grads, nullptr, nullptr, workspace, (cudaStream_t)stream);
}

extern "C" int sfm_loss_forward_backward_peer(const SfmDesc* desc, const SfmInputs* in, float* losses_out,
                                              const SfmGrads* grads, void* workspace, SfmPeer* peer, void* stream) {
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  if (!grads) { sfm_set_error("grads is NULL"); return SFM_E_NULL_POINTER; }
  if (!peer) { sfm_set_error("peer is NULL"); return SFM_E_NULL_POINTER; }
  const SfmPeerDev* dev = sfm_peer_dev(peer);
  if (!dev) { sfm_set_error("sfm_loss_forward_backward_peer: the peer object is not connected (sfm_peer_connect)"); return SFM_E_UNSUPPORTED; }
  return run_loss(desc, in, losses_out, grads, nullptr, nullptr, workspace, (cudaStream_t)stream, dev);
}

extern "C" int sfm_loss_forward_backward_images(const SfmDesc* desc, const SfmInputs* in, float* losses_out,
                                                const SfmGrads* grads, const SfmImageGrads* igrads, void* workspace,
                                                void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!(desc->flags & SFM_FLAG_IMAGE_GRADS)) {
    sfm_set_error("sfm_loss_forward_backward_images: desc->flags lacks SFM_FLAG_IMAGE_GRADS (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (desc->flags & SFM_FLAG_EDGE_AWARE_SMOOTH) {
    sfm_set_error("unsupported: image gradients through the edge-aware smoothness term (SFM_FLAG_EDGE_AWARE_SMOOTH)");
    return SFM_E_UNSUPPORTED;
  }
  if (desc->flags & SFM_FLAG_FULL_RES_MULTISCALE) {
    sfm_set_error("unsupported: image gradients together with SFM_FLAG_FULL_RES_MULTISCALE");
    return SFM_E_UNSUPPORTED;
  }
  if (!igrads || (!igrads->gtgt && !igrads->gsrc)) { sfm_set_error("igrads is NULL or has neither gtgt nor gsrc"); return SFM_E_NULL_POINTER; }
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  if (!grads) { sfm_set_error("grads is NULL"); return SFM_E_NULL_POINTER; }
  return run_loss(desc, in, losses_out, grads, nullptr, nullptr, workspace, (cudaStream_t)stream, nullptr, igrads);
}

extern "C" int sfm_loss_snippets(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms, float* losses_out,
                                 const SfmGrads* grads, const SfmImageGrads* igrads, void* workspace, SfmPeer* peer,
                                 void* stream) {
  return sfm_loss_weighted(desc, in, terms, nullptr, losses_out, grads, igrads, workspace, peer, stream);
}

extern "C" int sfm_loss_weighted(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms, const SfmPixelTerms* pix,
                                 float* losses_out, const SfmGrads* grads, const SfmImageGrads* igrads, void* workspace,
                                 SfmPeer* peer, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  const bool snip = terms && (terms->weights || terms->losses);
  if (snip && !(desc->flags & SFM_FLAG_SNIPPET_TERMS)) {
    sfm_set_error("sfm_loss_snippets: desc->flags lacks SFM_FLAG_SNIPPET_TERMS (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (igrads) {
    if (!(desc->flags & SFM_FLAG_IMAGE_GRADS)) {
      sfm_set_error("sfm_loss_snippets: igrads given but desc->flags lacks SFM_FLAG_IMAGE_GRADS (the workspace must be sized with it)");
      return SFM_E_INVALID_DESC;
    }
    if (desc->flags & SFM_FLAG_EDGE_AWARE_SMOOTH) {
      sfm_set_error("unsupported: image gradients through the edge-aware smoothness term (SFM_FLAG_EDGE_AWARE_SMOOTH)");
      return SFM_E_UNSUPPORTED;
    }
    if (desc->flags & SFM_FLAG_FULL_RES_MULTISCALE) {
      sfm_set_error("unsupported: image gradients together with SFM_FLAG_FULL_RES_MULTISCALE");
      return SFM_E_UNSUPPORTED;
    }
    if (!igrads->gtgt && !igrads->gsrc) { sfm_set_error("igrads has neither gtgt nor gsrc"); return SFM_E_NULL_POINTER; }
    if (!grads) { sfm_set_error("sfm_loss_snippets: igrads needs grads"); return SFM_E_NULL_POINTER; }
  }
  bool pixel = false;                  // per-pixel terms: some member of a scale < n_scales is set
  for (int s = 0; pix && s < desc->n_scales; ++s) pixel = pixel || pix->weights[s] || pix->losses[s];
  if (pixel && igrads) {
    sfm_set_error("unsupported: per-pixel terms (SfmPixelTerms) together with image gradients (igrads)");
    return SFM_E_UNSUPPORTED;
  }
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  const SfmPeerDev* dev = nullptr;
  if (peer && !(dev = sfm_peer_dev(peer))) {
    sfm_set_error("sfm_loss_snippets: the peer object is not connected (sfm_peer_connect)");
    return SFM_E_UNSUPPORTED;
  }
  return run_loss(desc, in, losses_out, grads, nullptr, nullptr, workspace, (cudaStream_t)stream, dev, igrads,
                  snip ? terms : nullptr, pixel ? pix : nullptr);
}

extern "C" int sfm_loss_min_reprojection(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms,
                                         const SfmMinReprojection* mr, float* losses_out, const SfmGrads* grads, void* workspace,
                                         SfmPeer* peer, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!(desc->flags & SFM_FLAG_MIN_REPROJECTION)) {
    sfm_set_error("sfm_loss_min_reprojection: desc->flags lacks SFM_FLAG_MIN_REPROJECTION (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (!(desc->ssim_rate >= 0.f && desc->ssim_rate <= 1.f)) {
    sfm_set_error("sfm_loss_min_reprojection: ssim_rate=%g outside [0, 1] (the selection needs a non-negative error)",
                  (double)desc->ssim_rate);
    return SFM_E_INVALID_DESC;
  }
  if (desc->exp_reg != 0.f) {
    sfm_set_error("unsupported: minimum reprojection together with the explainability branch (exp_reg != 0)");
    return SFM_E_UNSUPPORTED;
  }
  if (!mr) { sfm_set_error("SfmMinReprojection is NULL"); return SFM_E_NULL_POINTER; }
  if (mr->reserved_ != 0) { sfm_set_error("SfmMinReprojection.reserved_ must be 0"); return SFM_E_INVALID_DESC; }
  const bool snip = terms && (terms->weights || terms->losses);
  if (snip && !(desc->flags & SFM_FLAG_SNIPPET_TERMS)) {
    sfm_set_error("sfm_loss_min_reprojection: desc->flags lacks SFM_FLAG_SNIPPET_TERMS (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  const SfmPeerDev* dev = nullptr;
  if (peer && !(dev = sfm_peer_dev(peer))) {
    sfm_set_error("sfm_loss_min_reprojection: the peer object is not connected (sfm_peer_connect)");
    return SFM_E_UNSUPPORTED;
  }
  return run_loss(desc, in, losses_out, grads, nullptr, nullptr, workspace, (cudaStream_t)stream, dev, nullptr,
                  snip ? terms : nullptr, nullptr, mr);
}

extern "C" int sfm_loss_geometry(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms,
                                 const SfmGeometry* geo, float* losses_out, const SfmGrads* grads, void* workspace, SfmPeer* peer,
                                 void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!(desc->flags & SFM_FLAG_GEOMETRY_CONSISTENCY)) {
    sfm_set_error("sfm_loss_geometry: desc->flags lacks SFM_FLAG_GEOMETRY_CONSISTENCY (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (desc->exp_reg != 0.f) {
    sfm_set_error("unsupported: geometry consistency together with the explainability branch (exp_reg != 0)");
    return SFM_E_UNSUPPORTED;
  }
  const unsigned excl = desc->flags & (SFM_FLAG_FULL_RES_MULTISCALE | SFM_FLAG_BORDER_PADDING | SFM_FLAG_MIN_REPROJECTION);
  if (excl) {
    sfm_set_error("unsupported: geometry consistency together with %s",
                  (excl & SFM_FLAG_FULL_RES_MULTISCALE) ? "SFM_FLAG_FULL_RES_MULTISCALE"
                  : (excl & SFM_FLAG_BORDER_PADDING) ? "SFM_FLAG_BORDER_PADDING" : "SFM_FLAG_MIN_REPROJECTION");
    return SFM_E_UNSUPPORTED;
  }
  if (!geo) { sfm_set_error("SfmGeometry is NULL"); return SFM_E_NULL_POINTER; }
  for (int s = 0; s < desc->n_scales; ++s)
    if (!geo->src_disps[s]) { sfm_set_error("SfmGeometry.src_disps[%d] is NULL", s); return SFM_E_NULL_POINTER; }
  const bool snip = terms && (terms->weights || terms->losses);
  if (snip && !(desc->flags & SFM_FLAG_SNIPPET_TERMS)) {
    sfm_set_error("sfm_loss_geometry: desc->flags lacks SFM_FLAG_SNIPPET_TERMS (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  const SfmPeerDev* dev = nullptr;
  if (peer && !(dev = sfm_peer_dev(peer))) {
    sfm_set_error("sfm_loss_geometry: the peer object is not connected (sfm_peer_connect)");
    return SFM_E_UNSUPPORTED;
  }
  return run_loss(desc, in, losses_out, grads, nullptr, nullptr, workspace, (cudaStream_t)stream, dev, nullptr,
                  snip ? terms : nullptr, nullptr, nullptr, geo);
}

extern "C" int sfm_loss_geometry_valid_mean(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms,
                                            const SfmGeometry* geo, const SfmValidMean* vm, float* losses_out,
                                            const SfmGrads* grads, void* workspace, SfmPeer* peer, void* stream) {
  if (!vm) return sfm_loss_geometry(desc, in, terms, geo, losses_out, grads, workspace, peer, stream);
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!(desc->flags & SFM_FLAG_VALID_MEAN)) {
    sfm_set_error("sfm_loss_geometry_valid_mean: desc->flags lacks SFM_FLAG_VALID_MEAN (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (vm->groups < 1 || vm->groups > desc->B) {
    sfm_set_error("SfmValidMean.groups = %d outside [1, B = %d]", vm->groups, desc->B);
    return SFM_E_INVALID_DESC;
  }
  if (!(vm->min_count >= 0.f) || !isfinite(vm->min_count)) {
    sfm_set_error("SfmValidMean.min_count must be finite and >= 0");
    return SFM_E_INVALID_DESC;
  }
  if (peer) {
    sfm_set_error("unsupported: valid-pixel means with a peer (the counts are batch-global)");
    return SFM_E_UNSUPPORTED;
  }
  if (desc->B_global > 0 && desc->B_global != desc->B) {
    sfm_set_error("unsupported: valid-pixel means with B_global != B (the counts are batch-global)");
    return SFM_E_UNSUPPORTED;
  }
  if (!(desc->flags & SFM_FLAG_GEOMETRY_CONSISTENCY)) {
    sfm_set_error("sfm_loss_geometry_valid_mean: desc->flags lacks SFM_FLAG_GEOMETRY_CONSISTENCY (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (desc->exp_reg != 0.f) {
    sfm_set_error("unsupported: geometry consistency together with the explainability branch (exp_reg != 0)");
    return SFM_E_UNSUPPORTED;
  }
  const unsigned excl = desc->flags & (SFM_FLAG_FULL_RES_MULTISCALE | SFM_FLAG_BORDER_PADDING | SFM_FLAG_MIN_REPROJECTION);
  if (excl) {
    sfm_set_error("unsupported: geometry consistency together with %s",
                  (excl & SFM_FLAG_FULL_RES_MULTISCALE) ? "SFM_FLAG_FULL_RES_MULTISCALE"
                  : (excl & SFM_FLAG_BORDER_PADDING) ? "SFM_FLAG_BORDER_PADDING" : "SFM_FLAG_MIN_REPROJECTION");
    return SFM_E_UNSUPPORTED;
  }
  if (!geo) { sfm_set_error("SfmGeometry is NULL"); return SFM_E_NULL_POINTER; }
  for (int s = 0; s < desc->n_scales; ++s)
    if (!geo->src_disps[s]) { sfm_set_error("SfmGeometry.src_disps[%d] is NULL", s); return SFM_E_NULL_POINTER; }
  const bool snip = terms && (terms->weights || terms->losses);
  if (snip && !(desc->flags & SFM_FLAG_SNIPPET_TERMS)) {
    sfm_set_error("sfm_loss_geometry_valid_mean: desc->flags lacks SFM_FLAG_SNIPPET_TERMS (the workspace must be sized with it)");
    return SFM_E_INVALID_DESC;
  }
  if (!losses_out) { sfm_set_error("losses_out is NULL"); return SFM_E_NULL_POINTER; }
  return run_loss(desc, in, losses_out, grads, nullptr, nullptr, workspace, (cudaStream_t)stream, nullptr, nullptr,
                  snip ? terms : nullptr, nullptr, nullptr, geo, vm);
}

extern "C" int sfm_scale_image_grads(const SfmDesc* desc, const float* gy, const SfmImageGrads* igrads, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!gy) { sfm_set_error("gy is NULL"); return SFM_E_NULL_POINTER; }
  if (!igrads || (!igrads->gtgt && !igrads->gsrc)) { sfm_set_error("igrads is NULL or has neither gtgt nor gsrc"); return SFM_E_NULL_POINTER; }
  const long long img = 3ll * desc->H * desc->W;
  float* ptrs[2] = {igrads->gtgt, igrads->gsrc};
  const long long counts[2] = {desc->B * img, (long long)desc->B * desc->S * img};
  return sfm_launch_scale(ptrs, counts, 2, gy, (cudaStream_t)stream);
}

extern "C" int sfm_intrinsics_grad(const SfmDesc* desc, const SfmInputs* in, const void* workspace, float* gintrinsics,
                                   void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (desc->flags & SFM_FLAG_TABLES_PROVIDED) {
    sfm_set_error("unsupported: intrinsics gradient with SFM_FLAG_TABLES_PROVIDED (the step did not build proj / kinv from the intrinsics)");
    return SFM_E_UNSUPPORTED;
  }
  if (!in) { sfm_set_error("SfmInputs is NULL"); return SFM_E_NULL_POINTER; }
  if (!in->intrinsics || !in->poses) { sfm_set_error("intrinsics/poses pointer is NULL"); return SFM_E_NULL_POINTER; }
  if (!workspace) { sfm_set_error("workspace is NULL"); return SFM_E_NULL_POINTER; }
  if (((uintptr_t)workspace & 255) != 0) { sfm_set_error("workspace must be 256-byte aligned"); return SFM_E_INVALID_DESC; }
  if (!gintrinsics) { sfm_set_error("gintrinsics is NULL"); return SFM_E_NULL_POINTER; }
  SfmWsLayout L;
  sfm_ws_layout(desc, &L);
  const char* ws = (const char*)workspace;
  // the poses as the step saw them: under raw_pose_hw the vectors its prologue reduced into the workspace
  const float* poses = desc->raw_pose_hw > 0 ? (const float*)(ws + L.off_posevec) : in->poses;
  // under SFM_FLAG_FULL_RES_MULTISCALE every scale's projection was built from K_0 (the step's copy in the workspace), so
  // the per-scale gradients are folded into [:, 0]
  const bool fr = sfm_full_res(desc);
  rc = sfm_launch_intrinsics_grad(desc->B, desc->S, desc->n_scales, (const double*)(ws + L.off_acc) + 4, poses,
                                  fr ? (const float*)(ws + L.off_k0) : in->intrinsics, (desc->flags & SFM_FLAG_AXISANGLE_POSE) ? 1 : 0,
                                  (desc->flags & SFM_FLAG_POSE_INVERT_MASK) >> SFM_FLAG_POSE_INVERT_SHIFT, gintrinsics,
                                  (cudaStream_t)stream);
  if (rc || !fr) return rc;
  return sfm_launch_intrinsics_fold(desc->B, desc->n_scales, gintrinsics, (cudaStream_t)stream);
}

extern "C" int sfm_scale_intrinsics_grad(const SfmDesc* desc, const float* gy, float* gintrinsics, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!gy) { sfm_set_error("gy is NULL"); return SFM_E_NULL_POINTER; }
  if (!gintrinsics) { sfm_set_error("gintrinsics is NULL"); return SFM_E_NULL_POINTER; }
  const long long count = (long long)desc->B * desc->n_scales * 9;
  return sfm_launch_scale(&gintrinsics, &count, 1, gy, (cudaStream_t)stream);
}

extern "C" int sfm_scale_grads(const SfmDesc* desc, const float* gy, const SfmGrads* grads, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!gy) { sfm_set_error("gy is NULL"); return SFM_E_NULL_POINTER; }
  if ((rc = check_grads(desc, grads))) return rc;
  const Modes m = modes_of(desc);
  float* ptrs[2 * SFM_MAX_SCALES + 1];
  long long counts[2 * SFM_MAX_SCALES + 1];
  int n = 0;
  for (int s = 0; s < desc->n_scales; ++s) {
    const long long hw = (long long)(desc->H >> s) * (desc->W >> s);
    ptrs[n] = grads->gdisps[s]; counts[n++] = desc->B * hw;
    if (m.use_exp) { ptrs[n] = grads->glogits[s]; counts[n++] = (long long)desc->B * desc->S * hw; }
  }
  ptrs[n] = grads->gposes; counts[n++] = (long long)desc->B * desc->S * 6 * (desc->raw_pose_hw > 0 ? desc->raw_pose_hw : 1);
  return sfm_launch_scale(ptrs, counts, n, gy, (cudaStream_t)stream);
}

extern "C" int sfm_pyramid(const SfmDesc* desc, const float* tgt, const float* src, void* workspace, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!tgt || !src || !workspace) { sfm_set_error("sfm_pyramid: null pointer"); return SFM_E_NULL_POINTER; }
  const SfmPrepParams p = prep_params(desc, sfm_plan_band(desc), (char*)workspace, tgt, src, nullptr, nullptr, nullptr, nullptr, false);
  return sfm_launch_prep(p, nullptr, 0, (cudaStream_t)stream);
}

extern "C" int sfm_pyramid_export(const SfmDesc* desc, const void* workspace, int scale, float* tgt_out,
                                  float* src_out, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (scale < 1 || scale >= desc->n_scales) {
    sfm_set_error("sfm_pyramid_export: scale %d out of range (the workspace holds scales 1..%d; scale 0 is the input itself)", scale,
                  desc->n_scales - 1);
    return SFM_E_INVALID_DESC;
  }
  if (!workspace) { sfm_set_error("sfm_pyramid_export: null workspace"); return SFM_E_NULL_POINTER; }
  SfmWsLayout L;
  sfm_ws_layout(desc, &L);
  const char* ws = (const char*)workspace;
  // the pyramid levels are stored exactly in the output layout: (B,3,h,w) and (B,S,3,h,w)
  const size_t lvl = (size_t)3 * (desc->H >> scale) * (desc->W >> scale) * sizeof(float);
  if (tgt_out) SFM_CUDA_CHECK(cudaMemcpyAsync(tgt_out, ws + L.off_tgt[scale], desc->B * lvl, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (src_out) SFM_CUDA_CHECK(cudaMemcpyAsync(src_out, ws + L.off_src[scale], (size_t)desc->B * desc->S * lvl, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return 0;
}

extern "C" int sfm_build_tables(const SfmDesc* desc, const float* poses, const float* intrinsics, float* proj_out,
                                float* kinv_out, void* stream) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!poses || !intrinsics || !proj_out || !kinv_out) { sfm_set_error("sfm_build_tables: null pointer"); return SFM_E_NULL_POINTER; }
  const SfmPrepParams p = prep_params(desc, sfm_plan_band(desc), nullptr, nullptr, nullptr, intrinsics, poses, proj_out, kinv_out, false);
  return sfm_launch_prep(p, nullptr, 0, (cudaStream_t)stream, desc->flags & (SFM_FLAG_AXISANGLE_POSE | SFM_FLAG_POSE_INVERT_MASK));
}

extern "C" int sfm_ingest_u8(int B, int S, int H, int W, int n_scales, const uint8_t* frames, const float* K_in,
                             const SfmAugment* aug, float* tgt_out, float* src_out, float* intrinsics_out, void* stream) {
  if (B < 1 || S < 1 || S > SFM_MAX_SOURCES || n_scales < 1 || n_scales > SFM_MAX_SCALES) {
    sfm_set_error("sfm_ingest_u8: invalid B=%d S=%d n_scales=%d", B, S, n_scales);
    return SFM_E_INVALID_DESC;
  }
  if (H < 2 || W < 2 || (long long)B * (1 + S) * H * W >= (1ll << 31)) {
    sfm_set_error("sfm_ingest_u8: invalid shape H=%d W=%d", H, W);
    return SFM_E_INVALID_SHAPE;
  }
  if (!frames || !tgt_out || !src_out || (intrinsics_out && !K_in)) { sfm_set_error("sfm_ingest_u8: null pointer"); return SFM_E_NULL_POINTER; }
  return sfm_launch_ingest_u8(B, S, H, W, n_scales, frames, K_in, aug, tgt_out, src_out, intrinsics_out, (cudaStream_t)stream);
}

extern "C" size_t sfm_eval_depth_scratch_bytes(int B, int Hg, int Wg) {
  if (B < 1 || Hg < 1 || Wg < 1) return 0;
  return sfm_eval_scratch_bytes_impl(B, Hg, Wg);
}

extern "C" int sfm_eval_depth(int B, int h, int w, int Hg, int Wg, const float* pred_depth, const float* gt_depth,
                              const uint8_t* mask, float min_depth, float max_depth, float* errors_out, void* scratch,
                              void* stream) {
  if (B < 1 || h < 2 || w < 2 || Hg < 1 || Wg < 1) { sfm_set_error("sfm_eval_depth: invalid shape B=%d %dx%d -> %dx%d", B, h, w, Hg, Wg); return SFM_E_INVALID_SHAPE; }
  if (!(min_depth > 0.f) || !(max_depth >= min_depth)) { sfm_set_error("sfm_eval_depth: need 0 < min_depth <= max_depth"); return SFM_E_INVALID_DESC; }
  if (!pred_depth || !gt_depth || !mask || !errors_out || !scratch) { sfm_set_error("sfm_eval_depth: null pointer"); return SFM_E_NULL_POINTER; }
  return sfm_launch_eval_depth(B, h, w, Hg, Wg, pred_depth, gt_depth, mask, min_depth, max_depth, errors_out, scratch, (cudaStream_t)stream);
}

extern "C" int sfm_disp_activation(long long n, const float* x, float* disp, float* dact, void* stream) {
  if (n < 0) { sfm_set_error("sfm_disp_activation: n < 0"); return SFM_E_INVALID_SHAPE; }
  if (!x || (!disp && !dact)) { sfm_set_error("sfm_disp_activation: null pointer"); return SFM_E_NULL_POINTER; }
  return sfm_launch_disp_activation(n, x, disp, dact, (cudaStream_t)stream);
}

extern "C" int sfm_upsample_disparity(int N, int h, int w, int H, int W, const float* x, float* y, void* stream) {
  if (N < 1 || h < 1 || w < 1 || h > H || w > W || (long long)N * H * W >= (1ll << 31)) {
    sfm_set_error("sfm_upsample_disparity: invalid shape N=%d %dx%d -> %dx%d", N, h, w, H, W);
    return SFM_E_INVALID_SHAPE;
  }
  if (!x || !y) { sfm_set_error("sfm_upsample_disparity: null pointer"); return SFM_E_NULL_POINTER; }
  return sfm_launch_upsample_stage(N, h, w, H, W, x, y, (cudaStream_t)stream);
}

extern "C" int sfm_pose_reduce(int B, int S, int hw, const float* x, float* poses_out, void* stream) {
  if (B < 1 || S < 1 || S > SFM_MAX_SOURCES) { sfm_set_error("sfm_pose_reduce: invalid B=%d S=%d", B, S); return SFM_E_INVALID_DESC; }
  if (hw < 1 || hw > 128) { sfm_set_error("sfm_pose_reduce: unsupported hw=%d (1..128)", hw); return SFM_E_UNSUPPORTED; }
  if (!x || !poses_out) { sfm_set_error("sfm_pose_reduce: null pointer"); return SFM_E_NULL_POINTER; }
  return sfm_launch_pose_reduce(B, S, hw, x, poses_out, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------------
// host-buffer path
// ------------------------------------------------------------------------------------------------
struct SfmHostCtx {
  SfmDesc desc;
  cudaStream_t stream;
  void* workspace;
  float *d_tgt, *d_src, *d_K, *d_poses, *d_losses, *d_gposes;
  float* d_disp[SFM_MAX_SCALES];
  float* d_logits[SFM_MAX_SCALES];
  float* d_gdisp[SFM_MAX_SCALES];
  float* d_glogits[SFM_MAX_SCALES];
  // uint8 entry (sfm_loss_step_host_u8_submit): allocated on first use
  uint8_t* d_frames;
  SfmAugment* d_aug;
  float* d_Kin;
  std::vector<void*> allocs;
};

static int host_alloc(SfmHostCtx* c, void** p, size_t bytes) {
  SFM_CUDA_CHECK(cudaMalloc(p, bytes));
  c->allocs.push_back(*p);
  return 0;
}

extern "C" int sfm_host_ctx_destroy(SfmHostCtx* ctx) {
  if (!ctx) return 0;
  for (void* p : ctx->allocs) cudaFree(p);
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
  return 0;
}

extern "C" int sfm_host_ctx_create(const SfmDesc* desc, SfmHostCtx** ctx_out) {
  int rc = sfm_validate_desc(desc);
  if (rc) return rc;
  if (!ctx_out) { sfm_set_error("ctx_out is NULL"); return SFM_E_NULL_POINTER; }
  if (desc->flags & SFM_FLAG_FULL_RES_MULTISCALE) {
    sfm_set_error("unsupported: the host-buffer path with SFM_FLAG_FULL_RES_MULTISCALE");
    return SFM_E_UNSUPPORTED;
  }
  if (desc->flags & (SFM_FLAG_MEAN_NORM_SMOOTH | SFM_FLAG_EDGE_MEAN_ABS)) {
    sfm_set_error("unsupported: the host-buffer path with SFM_FLAG_MEAN_NORM_SMOOTH or SFM_FLAG_EDGE_MEAN_ABS");
    return SFM_E_UNSUPPORTED;
  }
  if (desc->flags & SFM_FLAG_BORDER_PADDING) {
    sfm_set_error("unsupported: the host-buffer path with SFM_FLAG_BORDER_PADDING");
    return SFM_E_UNSUPPORTED;
  }
  if (desc->flags & SFM_FLAG_AXISANGLE_POSE) {
    sfm_set_error("unsupported: the host-buffer path with SFM_FLAG_AXISANGLE_POSE");
    return SFM_E_UNSUPPORTED;
  }
  if (desc->flags & SFM_FLAG_GEOMETRY_CONSISTENCY) {
    sfm_set_error("unsupported: the host-buffer path with SFM_FLAG_GEOMETRY_CONSISTENCY");
    return SFM_E_UNSUPPORTED;
  }
  if (desc->flags & SFM_FLAG_VALID_MEAN) {
    sfm_set_error("unsupported: the host-buffer path with SFM_FLAG_VALID_MEAN");
    return SFM_E_UNSUPPORTED;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    sfm_set_error("no CUDA device: libsfmloss has no CPU fallback");
    return SFM_E_NO_DEVICE;
  }
  SfmHostCtx* c = new (std::nothrow) SfmHostCtx();
  if (!c) { sfm_set_error("out of host memory"); return SFM_E_INVALID_DESC; }
  c->desc = *desc;
  c->desc.flags &= ~(SFM_FLAG_TABLES_PROVIDED | SFM_FLAG_REUSE_PYRAMID);
  const SfmDesc* d = &c->desc;
  const Modes m = modes_of(d);
  const size_t img = (size_t)d->H * d->W * 3 * sizeof(float);
#define HA(ptr, bytes)                                                     \
  if ((rc = host_alloc(c, (void**)&(ptr), (bytes)))) { sfm_host_ctx_destroy(c); return rc; }
  if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
    sfm_set_error("cudaStreamCreate failed");
    delete c;
    return (int)cudaErrorUnknown;
  }
  HA(c->workspace, sfm_workspace_bytes(d));
  HA(c->d_tgt, d->B * img);
  HA(c->d_src, (size_t)d->B * d->S * img);
  HA(c->d_K, (size_t)d->B * d->n_scales * 9 * sizeof(float));
  const size_t pose_bytes = (size_t)d->B * d->S * 6 * (d->raw_pose_hw > 0 ? d->raw_pose_hw : 1) * sizeof(float);
  HA(c->d_poses, pose_bytes);
  HA(c->d_gposes, pose_bytes);
  HA(c->d_losses, 8 * sizeof(float));
  {
    // the per-scale arrays of one kind are carved back to back out of ONE allocation: when the caller's host arrays
    // are laid out the same way (scale s+1 right behind scale s) they travel in a single copy (host_submit)
    size_t tot = 0;
    for (int s = 0; s < d->n_scales; ++s) tot += (size_t)(d->H >> s) * (d->W >> s);
    float *bd = nullptr, *bg = nullptr, *bl = nullptr, *bgl = nullptr;
    HA(bd, d->B * tot * sizeof(float));
    HA(bg, d->B * tot * sizeof(float));
    if (m.use_exp) {
      HA(bl, (size_t)d->B * d->S * tot * sizeof(float));
      HA(bgl, (size_t)d->B * d->S * tot * sizeof(float));
    }
    size_t off = 0;
    for (int s = 0; s < d->n_scales; ++s) {
      const size_t hw = (size_t)(d->H >> s) * (d->W >> s);
      c->d_disp[s] = bd + d->B * off;
      c->d_gdisp[s] = bg + d->B * off;
      if (m.use_exp) {
        c->d_logits[s] = bl + (size_t)d->B * d->S * off;
        c->d_glogits[s] = bgl + (size_t)d->B * d->S * off;
      }
      off += hw;
    }
  }
#undef HA
  *ctx_out = c;
  return 0;
}

extern "C" int sfm_loss_step_host_wait(SfmHostCtx* c) {
  if (!c) { sfm_set_error("sfm_loss_step_host_wait: null context"); return SFM_E_NULL_POINTER; }
  SFM_CUDA_CHECK(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int sfm_loss_step_host(SfmHostCtx* c, const SfmInputs* in, float* losses_out, const SfmGrads* grads) {
  const int rc = sfm_loss_step_host_submit(c, in, losses_out, grads);
  return rc ? rc : sfm_loss_step_host_wait(c);
}

static int host_submit(SfmHostCtx* c, const SfmInputs* in, float* losses_out, const SfmGrads* grads, bool images_on_device);

extern "C" int sfm_loss_step_host_submit(SfmHostCtx* c, const SfmInputs* in, float* losses_out, const SfmGrads* grads) {
  return host_submit(c, in, losses_out, grads, false);
}

extern "C" int sfm_loss_step_host_u8_submit(SfmHostCtx* c, const uint8_t* frames, const float* K_in, const SfmAugment* aug,
                                            const SfmInputs* in, float* losses_out, const SfmGrads* grads) {
  if (!c || !frames || !K_in || !in) { sfm_set_error("sfm_loss_step_host_u8_submit: null pointer"); return SFM_E_NULL_POINTER; }
  const SfmDesc* d = &c->desc;
  const size_t n_frames = (size_t)d->B * (1 + d->S) * d->H * d->W * 3;
  if (aug) {
    // the crop window must lie inside the rescaled image (kitti_raw_transformed.py:36-50); the kernel trusts these
    for (int b = 0; b < d->B; ++b) {
      const SfmAugment& a = aug[b];
      if (a.out_h < d->H || a.out_w < d->W || a.off_y < 0 || a.off_x < 0 || a.off_y > a.out_h - d->H || a.off_x > a.out_w - d->W ||
          !(a.x_scaling > 0.0) || !(a.y_scaling > 0.0)) {
        sfm_set_error("sfm_loss_step_host_u8_submit: aug[%d] is invalid (out %dx%d, offset %d,%d for a %dx%d crop)", b, a.out_h, a.out_w,
                      a.off_y, a.off_x, d->H, d->W);
        return SFM_E_INVALID_DESC;
      }
    }
  }
  // each buffer is guarded on its own: a failed allocation leaves the others usable and is retried by the next call
  int rc0;
  if (!c->d_frames && (rc0 = host_alloc(c, (void**)&c->d_frames, n_frames))) return rc0;
  if (!c->d_aug && (rc0 = host_alloc(c, (void**)&c->d_aug, (size_t)d->B * sizeof(SfmAugment)))) return rc0;
  if (!c->d_Kin && (rc0 = host_alloc(c, (void**)&c->d_Kin, (size_t)d->B * 9 * sizeof(float)))) return rc0;
  cudaStream_t st = c->stream;
  SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_frames, frames, n_frames, cudaMemcpyHostToDevice, st));
  SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_Kin, K_in, (size_t)d->B * 9 * sizeof(float), cudaMemcpyHostToDevice, st));
  if (aug) SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_aug, aug, (size_t)d->B * sizeof(SfmAugment), cudaMemcpyHostToDevice, st));
  int rc = sfm_launch_ingest_u8(d->B, d->S, d->H, d->W, d->n_scales, c->d_frames, c->d_Kin, aug ? c->d_aug : nullptr, c->d_tgt,
                                c->d_src, c->d_K, st);
  if (rc) return rc;
  return host_submit(c, in, losses_out, grads, true);
}

static int host_submit(SfmHostCtx* c, const SfmInputs* in, float* losses_out, const SfmGrads* grads, bool images_on_device) {
  if (!c || !in || !losses_out || !grads) { sfm_set_error("sfm_loss_step_host: null pointer"); return SFM_E_NULL_POINTER; }
  const SfmDesc* d = &c->desc;
  SfmInputs chk = *in;
  if (images_on_device) { chk.tgt = c->d_tgt; chk.src = c->d_src; chk.intrinsics = c->d_K; }   // produced by the ingest kernel
  int rc = check_inputs(d, &chk, true);
  if (rc) return rc;
  if ((rc = check_grads(d, grads))) return rc;
  const Modes m = modes_of(d);
  cudaStream_t st = c->stream;
  const size_t img = (size_t)d->H * d->W * 3 * sizeof(float);
  if (!images_on_device) {
    SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_tgt, in->tgt, d->B * img, cudaMemcpyHostToDevice, st));
    SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_src, in->src, (size_t)d->B * d->S * img, cudaMemcpyHostToDevice, st));
    SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_K, in->intrinsics, (size_t)d->B * d->n_scales * 9 * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  const size_t pose_bytes = (size_t)d->B * d->S * 6 * (d->raw_pose_hw > 0 ? d->raw_pose_hw : 1) * sizeof(float);
  SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_poses, in->poses, pose_bytes, cudaMemcpyHostToDevice, st));
  SfmInputs din{};
  SfmGrads dg{};
  din.tgt = c->d_tgt; din.src = c->d_src; din.intrinsics = c->d_K; din.poses = c->d_poses;
  dg.gposes = c->d_gposes;
  // Every copy has a fixed cost of several microseconds (measured on B200: a 1 MB pinned H2D copy reaches 21 GB/s, a
  // 3 MB one 49 GB/s), so host arrays that lie back to back in scale order -- the device side always does -- travel
  // as ONE copy per kind instead of one per scale.
  size_t pix_tot = 0;
  for (int s = 0; s < d->n_scales; ++s) pix_tot += (size_t)(d->H >> s) * (d->W >> s);
  auto contiguous = [&](const float* const* a, size_t per_pixel) {
    for (int s = 0; s + 1 < d->n_scales; ++s)
      if (a[s + 1] != a[s] + per_pixel * (size_t)(d->H >> s) * (d->W >> s)) return false;
    return true;
  };
  const bool disp_1 = contiguous(in->disps, d->B), gdisp_1 = contiguous(grads->gdisps, d->B);
  const bool lg_1 = m.use_exp && contiguous(in->logits, (size_t)d->B * d->S);
  const bool glg_1 = m.use_exp && contiguous(grads->glogits, (size_t)d->B * d->S);
  if (disp_1) SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_disp[0], in->disps[0], d->B * pix_tot * sizeof(float), cudaMemcpyHostToDevice, st));
  if (lg_1) SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_logits[0], in->logits[0], (size_t)d->B * d->S * pix_tot * sizeof(float), cudaMemcpyHostToDevice, st));
  for (int s = 0; s < d->n_scales; ++s) {
    const size_t hw = (size_t)(d->H >> s) * (d->W >> s) * sizeof(float);
    if (!disp_1) SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_disp[s], in->disps[s], d->B * hw, cudaMemcpyHostToDevice, st));
    din.disps[s] = c->d_disp[s];
    dg.gdisps[s] = c->d_gdisp[s];
    if (m.use_exp) {
      if (!lg_1) SFM_CUDA_CHECK(cudaMemcpyAsync(c->d_logits[s], in->logits[s], (size_t)d->B * d->S * hw, cudaMemcpyHostToDevice, st));
      din.logits[s] = c->d_logits[s];
      dg.glogits[s] = c->d_glogits[s];
    }
  }
  rc = sfm_loss_forward_backward(d, &din, c->d_losses, &dg, c->workspace, st);
  if (rc) return rc;
  SFM_CUDA_CHECK(cudaMemcpyAsync(losses_out, c->d_losses, 5 * sizeof(float), cudaMemcpyDeviceToHost, st));
  SFM_CUDA_CHECK(cudaMemcpyAsync(grads->gposes, c->d_gposes, pose_bytes, cudaMemcpyDeviceToHost, st));
  if (gdisp_1) SFM_CUDA_CHECK(cudaMemcpyAsync(grads->gdisps[0], c->d_gdisp[0], d->B * pix_tot * sizeof(float), cudaMemcpyDeviceToHost, st));
  if (glg_1) SFM_CUDA_CHECK(cudaMemcpyAsync(grads->glogits[0], c->d_glogits[0], (size_t)d->B * d->S * pix_tot * sizeof(float), cudaMemcpyDeviceToHost, st));
  for (int s = 0; s < d->n_scales; ++s) {
    const size_t hw = (size_t)(d->H >> s) * (d->W >> s) * sizeof(float);
    if (!gdisp_1) SFM_CUDA_CHECK(cudaMemcpyAsync(grads->gdisps[s], c->d_gdisp[s], d->B * hw, cudaMemcpyDeviceToHost, st));
    if (m.use_exp && !glg_1)
      SFM_CUDA_CHECK(cudaMemcpyAsync(grads->glogits[s], c->d_glogits[s], (size_t)d->B * d->S * hw, cudaMemcpyDeviceToHost, st));
  }
  return 0;
}
