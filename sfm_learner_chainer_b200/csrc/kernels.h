// kernels.h -- kernel parameter blocks and launchers shared between the .cu translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sfmloss.h"

struct SfmPrepParams {
  int B, S, H, W, ns;
  int do_pyramid;    // 0: only tables / accumulator reset
  int build_tables;  // 0: caller supplied proj/kinv
  const float* tgt;
  const float* src;
  const float* intrinsics;
  const float* poses;
  float* tgt_pyr[SFM_MAX_SCALES];   // planar [B][3][h][w], written for scales >= 1 only
  float* src_pyr[SFM_MAX_SCALES];   // planar [B*S][3][h][w]
  float* proj_out;
  float* kinv_out;
  double* acc;
  int n_acc;
  int raw_pose_hw;   // > 0: `poses` is the raw poseout map (B, 6S, raw_pose_hw); the reduced vectors go to posevec_out
  float* posevec_out;
  int n_pyr_blocks, n_tail_blocks;   // filled by the launcher
  int n_mix_region;  // the smoothness CTAs are spread evenly over the first n_mix_region blocks after the tail blocks
  int band;          // full-resolution rows per pyramid CTA
};

// Second-order smoothness tasks that ride in the prologue kernel (smooth_task.cuh): strips x row segments of every
// (snippet, scale), one per warp of n_ctas 8-warp CTAs; CTA k writes its loss partial to part[k].  The planner fills
// the task geometry (ns .. tile_begin), the caller the rest.
struct SfmSmoothParams {
  int ns, hseg, n_tasks, n_ctas;
  int h[SFM_MAX_SCALES], w[SFM_MAX_SCALES];
  int tiles_x[SFM_MAX_SCALES], tiles_y[SFM_MAX_SCALES];
  int tile_begin[SFM_MAX_SCALES + 1];
  const float* disp[SFM_MAX_SCALES];
  float* gdisp[SFM_MAX_SCALES];
  float k_dx2[SFM_MAX_SCALES], k_mix[SFM_MAX_SCALES], k_dy2[SFM_MAX_SCALES];
  const float* gy;
  unsigned raw_disp_mask;
  float* part;       // [n_ctas] loss partials (workspace)
  // per-snippet terms (sm_mode 3 / 4): the gradient factor of snippet b is gy * snip_w[b] (snip_w nullptr: gy), and each
  // task t writes its loss to task_part[t] instead of the CTA partial (a CTA's tasks may belong to different snippets)
  const float* snip_w;
  float* task_part;
};

// sm_mode: 0 = no smoothness tasks, 1 = loss only, 2 = loss + gdisp; 3 / 4 = 1 / 2 with per-task losses (task_part)
int sfm_launch_prep(const SfmPrepParams& p, const SfmSmoothParams* sm, int sm_mode, cudaStream_t stream);
int sfm_launch_ingest_u8(int B, int S, int H, int W, int ns, const uint8_t* frames, const float* K_in, const SfmAugment* aug,
                         float* tgt, float* src, float* K_out, cudaStream_t stream);   // ingest.cu
size_t sfm_eval_scratch_bytes_impl(int B, int Hg, int Wg);                                  // eval.cu
int sfm_launch_eval_depth(int B, int h, int w, int Hg, int Wg, const float* pred, const float* gt, const uint8_t* mask, float lo,
                          float hi, float* out, void* scratch, cudaStream_t stream);
int sfm_launch_disp_activation(long long n, const float* x, float* disp, float* dact, cudaStream_t stream);
int sfm_launch_pose_reduce(int B, int S, int hw, const float* x, float* poses_out, cudaStream_t stream);

// Cross-GPU sum of the five loss partials inside the epilogue kernel, over NVLink peer memory (comm.cu: SfmPeer).
// Every rank owns a slot array [2 parities][nranks] that the OTHER ranks' epilogues write with plain peer stores;
// slots[r] is rank r's array as mapped into this process (CUDA IPC).  `counter` (local) numbers the steps.
constexpr int SFM_MAX_PEERS = 16;
struct SfmPeerSlot {
  float v[5];
  unsigned pad0, pad1;
  unsigned seq;          // step number the five values belong to (written last, after a system-scope fence)
};
struct SfmPeerDev {
  int nranks, rank;      // nranks == 0: no cross-GPU sum
  unsigned* counter;
  SfmPeerSlot* slots[SFM_MAX_PEERS];
};

// Warp tasks of a marching kernel: scale s holds tasks [task_begin[s], task_begin[s+1]), nseg[s] row segments of hseg
// rows each (L1 kernel: rows = 32-pixel runs, nstrip[s] of them; SSIM kernel: image rows, nstrip[s] column strips of
// SFM_SSIM_IW interior columns) per snippet.
constexpr int SFM_SSIM_IW = 28;
struct SfmTaskTable {
  int hseg;
  int nstrip[SFM_MAX_SCALES], nseg[SFM_MAX_SCALES];
  int task_begin[SFM_MAX_SCALES + 1];
};

// Fused loss kernel parameters (one launch covers every scale, source and snippet).
struct SfmFusedParams {
  int B, S, ns;
  int h[SFM_MAX_SCALES], w[SFM_MAX_SCALES];
  SfmTaskTable tasks;
  float hwf[SFM_MAX_SCALES], hhf[SFM_MAX_SCALES];     // (w-1)/2, (h-1)/2
  // images of every scale, planar fp32 [img][3][h][w]: scale 0 = the caller's tgt / src tensors themselves, scales >= 1 =
  // the pyramid in the workspace
  const float* tgt_pl[SFM_MAX_SCALES];
  const float* src_pl[SFM_MAX_SCALES];
  const float* disp[SFM_MAX_SCALES];
  const float* logits[SFM_MAX_SCALES];
  float* gdisp[SFM_MAX_SCALES];
  float* glogits[SFM_MAX_SCALES];
  const float* proj;        // [B][S][ns][12]
  const float* kinv;        // [B][ns][9]
  const float* intrinsics;  // [B][ns][9]
  const float* poses;       // [B][S][6] (the reduced vectors in the workspace when raw_pose_hw > 0)
  int raw_pose_hw;          // > 0: gposes has the raw map's shape (B, 6S, raw_pose_hw)
  unsigned raw_disp_mask;   // bit s: disp[s] is pre-activation, gdisp[s] the gradient w.r.t. it
  const float* gy;          // upstream gradient (device scalar) or nullptr
  double* acc;              // [4 + B*S*ns*12]
  const float* sm_part;     // loss partials of the smoothness CTAs of the prologue kernel (per-snippet terms: of its tasks)
  int n_sm_part;
  SfmPeerDev peer;          // nranks > 0: losses_out receives the sums over all ranks (epilogue kernel)
  float* losses_out;        // [5] or nullptr
  float* gposes;            // [B][S][6] or nullptr
  // loss weights per scale (host-computed in fp64, global batch in the denominators)
  float inv_n3[SFM_MAX_SCALES];      // 1 / (Bg*3*h*w)
  float inv_n1[SFM_MAX_SCALES];      // 1 / (Bg*h*w)
  float sm_dx2[SFM_MAX_SCALES];      // smooth_reg/2^s / (Bg*h*(w-2))
  float sm_mix[SFM_MAX_SCALES];      // smooth_reg/2^s / (Bg*(h-1)*(w-1))
  float sm_dy2[SFM_MAX_SCALES];      // smooth_reg/2^s / (Bg*(h-2)*w)
  float sm_ex[SFM_MAX_SCALES];       // smooth_reg/2^s / (Bg*h*(w-1))      edge-aware variant (compute_disp_smooth)
  float sm_ey[SFM_MAX_SCALES];       // smooth_reg/2^s / (Bg*(h-1)*w)
  int edge_smooth;                   // SFM_FLAG_EDGE_AWARE_SMOOTH
  float smooth_reg, exp_reg, ssim_rate;
  int use_smooth;
  // debug dumps (nullptr when unused)
  float* dbg_P[SFM_MAX_SCALES];
  int32_t* dbg_u0[SFM_MAX_SCALES];
  int32_t* dbg_v0[SFM_MAX_SCALES];
  uint8_t* dbg_inb[SFM_MAX_SCALES];
  // image gradients (sfm_loss_forward_backward_images; nullptr when not wanted): scale 0 = the caller's buffers, scales
  // >= 1 = the gradient levels in the workspace, pulled back into scale 0 by sfm_launch_image_pullback.  gsrc is
  // zeroed before the step and accumulated with fp32 reductions; gtgt is owned like gdisp (stored by the first pass).
  float* gtgt[SFM_MAX_SCALES];      // [B][3][h][w]
  float* gsrc[SFM_MAX_SCALES];      // [B*S][3][h][w]
  // per-snippet terms (sfm_loss_snippets; snip_cell0 == 0 when off).  The gradient factor of snippet b's tasks is
  // gy * snip_w[b] (snip_w nullptr: gy); its loss partials go to cells acc[snip_cell0 + 4b + k] (pixel, smooth, exp, ssim)
  // instead of acc[k], and the epilogue forms losses_out = sum_b w_b * cells_b and the rows snip_losses[b][5]
  const float* snip_w;
  float* snip_losses;               // [B][5] or nullptr
  int snip_cell0;
  // per-snippet terms: segment height of the prologue's smoothness tasks, whose losses sm_part then holds one per task
  // (0: no such tasks).  Their order is the planner's (plan_smooth): per scale, per snippet, strips x segments.
  int sm_hseg;
  // per-pixel terms (sfm_loss_weighted; nullptr when off), [B][S][h][w] per scale like logits.  pix_w[s] multiplies the
  // photometric terms of every (pixel, source) at scale s (nullptr: 1); pix_map[s] receives d losses_out[0] / d pix_w.
  // Appended last, so that no member the other kernels read moves.
  const float* pix_w[SFM_MAX_SCALES];
  float* pix_map[SFM_MAX_SCALES];
  // what pix_map receives for a masked or out-of-view (pixel, source): 0 (its share of the loss), or a negative marker in
  // the forward march of sfm_loss_min_reprojection, whose select kernel must tell "masked" from "error 0"
  float pix_map_masked;
};

// Launch helper: with pdl the kernel is a programmatic dependent launch on the previous kernel of the stream (its
// CTAs may be scheduled while the predecessor drains; the kernel itself orders its dependent accesses with
// cudaGridDependencySynchronize()).
template <typename K, typename... Args>
static inline cudaError_t sfm_launch_kernel(K kernel, dim3 grid, unsigned block, cudaStream_t stream, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = pdl ? attr : nullptr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

struct SfmPeer;
const SfmPeerDev* sfm_peer_dev(const SfmPeer* q);      // comm.cu; nullptr until connected

// Resident warps per SM the SSIM marching kernel is compiled for (__launch_bounds__), which the planner's cost model
// counts with: forward records in shared memory (168 registers) / in registers (250 registers).
constexpr int SFM_SSIM_MIN_WARPS = 12;
constexpr int SFM_SSIM_REG_MIN_WARPS = 8;
// image-gradient instances: with the bound of 12 the extra gradient field spilled; with 10 ptxas allocates 168 registers
// without spilling, so 12 warps per SM are still resident and the cost model stays as it is
constexpr int SFM_SSIM_IMG_MIN_WARPS = 10;

// Launch plan of one fused step (plan.cu, the whole launch policy).  The marching kernel instance is
// sfm_l1_march_kernel<exp, grad, accum, debug, raw, img, snip, pix, border> or
// sfm_ssim_march_kernel<grad, accum, debug, raw, nw, srec, img, snip, pix, border>.
struct SfmStepPlan {
  bool ssim;                           // kernel family
  bool exp, grad, accum, debug, raw;   // accum: a smoothness kernel has initialised gdisp
  bool img;                            // image gradients (grad, !debug; SSIM: nw = 1 with shared-memory records)
  bool pix;                            // per-pixel terms (!debug, !img; SSIM: nw = 1 with shared-memory records)
  bool border;                         // SFM_FLAG_BORDER_PADDING (pix, !exp): border-clamped sampler, reflection-padded SSIM
  bool minrep;                         // minimum reprojection (pix): a forward per-pixel march with the task table pre_tasks
                                       // and the select kernel run ahead of the march of this plan
  SfmTaskTable pre_tasks;
  int nw;                              // SSIM: warps per CTA (2: the two sources split over the warps of a CTA)
  bool srec;                           // SSIM: forward records in shared memory (false: in registers)
  bool edge_smooth;                    // the edge-aware smoothness kernel runs between the prologue and the march
  SfmTaskTable tasks;
  SfmSmoothParams smooth;              // second-order smoothness tasks of the prologue (n_ctas == 0: none)
  int band, n_mix_region;              // SfmPrepParams
};
// mode bits of the planner
enum { SFM_MODE_EXP = 1, SFM_MODE_SSIM = 2, SFM_MODE_GRAD = 4, SFM_MODE_DEBUG = 8, SFM_MODE_SMOOTH = 16, SFM_MODE_IMG = 32,
       SFM_MODE_PIX = 64, SFM_MODE_MINREP = 128, SFM_MODE_BORDER = 256 };
SfmStepPlan sfm_plan_step(const SfmDesc* d, int mode, int num_sms);
int sfm_plan_band(const SfmDesc* d);
// Minimum reprojection (sfm_loss_min_reprojection): the planes p.pix_w[s] are written by the forward march and turned
// into the one-hot weights by the select kernel, which also writes the optional selection maps.
struct SfmMinRepArgs {
  int automask;
  int8_t* selection[SFM_MAX_SCALES];
};
// Mean-normalised smoothness (SFM_FLAG_MEAN_NORM_SMOOTH, mean_norm.cu), per snippet b and native scale s: the sum kernel
// writes the per-CTA sums of the activated disparity, the fix-up kernel reduces them and the smoothness loss partials
// of (b, s) in a fixed order into m_bs and L_bs, stores the snippet's normalised loss sum_s L_bs / (m_bs + 1e-7) and, in
// gradient steps, rewrites the smoothness gradient in place as r G - gy w_b r^2 L_bs / (h w) f (r = 1 / (m_bs + 1e-7)).
struct SfmMeanNorm {
  int B, ns, chunks;                          // chunks: CTAs per snippet of both kernels (<= SFM_MN_SLOTS)
  int h[SFM_MAX_SCALES], w[SFM_MAX_SCALES];   // native sizes
  const float* disp[SFM_MAX_SCALES];          // the caller's maps (pre-activation for the raw bits)
  float* gdisp[SFM_MAX_SCALES];               // the caller's gradients, holding the smoothness gradient (nullptr: forward)
  unsigned raw_disp_mask;
  const float* gy;                            // device scalar or nullptr (1)
  const float* snip_w;                        // (B) snippet weights or nullptr
  float* mean_part;                           // [B][ns][SFM_MN_SLOTS]
  // loss partials of (b, s): loss_part[loss_off[s] + b * loss_stride[s] + k], k < loss_cnt[s]
  const float* loss_part;
  float* edge_slots;                          // edge-aware smoothness: where that kernel writes them (== loss_part)
  int loss_off[SFM_MAX_SCALES], loss_stride[SFM_MAX_SCALES], loss_cnt[SFM_MAX_SCALES];
  float* snip_loss;                           // [B] normalised loss of every snippet (the epilogue's smoothness partials)
  double* snip_cell;                          // per-snippet terms: snippet b's smooth cell at snip_cell[4 b] (else nullptr)
};
int sfm_launch_mean_norm_sum(const SfmMeanNorm& m, cudaStream_t stream);   // a dependent launch behind the prologue
int sfm_launch_mean_norm_fix(const SfmMeanNorm& m, bool grad, cudaStream_t stream);   // behind the smoothness writers
// native: with SFM_FLAG_FULL_RES_MULTISCALE, the parameters of the native-resolution scales (dims, disparity, gradient,
// pyramid, raw bits), read by the edge-aware smoothness kernel and by the epilogue's layout of the smoothness tasks.
// mn: SFM_FLAG_MEAN_NORM_SMOOTH with a smoothness term (nullptr otherwise); edge_mean_abs: SFM_FLAG_EDGE_MEAN_ABS
int sfm_launch_fused(SfmFusedParams& p, const SfmStepPlan& plan, cudaStream_t stream, const SfmMinRepArgs* mr = nullptr,
                     const SfmFusedParams* native = nullptr, const SfmMeanNorm* mn = nullptr, bool edge_mean_abs = false);
// smooth.cu; slots (SFM_FLAG_MEAN_NORM_SMOOTH): the per-CTA loss partials [B][ns][SFM_MN_SLOTS] instead of the cells
int sfm_launch_edge_smooth(const SfmFusedParams& p, bool grad, bool mean_abs, float* slots, cudaStream_t stream);
extern thread_local cudaEvent_t sfm_ev_start, sfm_ev_stop;   // profiling hook (sfm_set_kernel_events)

int sfm_launch_scale(float* const* ptrs, const long long* counts, int n, const float* gy, cudaStream_t stream);
// adds the gradient levels p.gtgt[s] / p.gsrc[s] (s >= 1) into the full-resolution p.gtgt[0] / p.gsrc[0] through the
// adjoint of the pyramid (fused_loss.cu); a dependent launch behind the epilogue
int sfm_launch_image_pullback(const SfmFusedParams& p, int H, int W, cudaStream_t stream);
// gintrinsics (B,ns,3,3) from the dL/dP cells (SfmWsLayout::off_acc + 4 doubles) and the poses / intrinsics the step
// used (fused_loss.cu); a dependent launch behind the step's last kernel
int sfm_launch_intrinsics_grad(int B, int S, int ns, const double* cells, const float* poses, const float* intrinsics,
                               float* gintrinsics, cudaStream_t stream);

// Full-resolution multi-scale (SFM_FLAG_FULL_RES_MULTISCALE, full_res.cu): the scales >= 1 of the step are full-resolution
// scales whose disparity up[s] = U_s(disp[s]) and gradient gup[s] live in the workspace.
struct SfmFullRes {
  int B, ns, H, W;
  int h[SFM_MAX_SCALES], w[SFM_MAX_SCALES];   // native sizes
  const float* disp[SFM_MAX_SCALES];          // the caller's maps (pre-activation for the raw bits)
  float* gdisp[SFM_MAX_SCALES];               // the caller's gradients (nullptr: forward only)
  float* up[SFM_MAX_SCALES];                  // [B][H][W], s >= 1
  float* gup[SFM_MAX_SCALES];                 // [B][H][W], s >= 1 (nullptr: forward only)
  unsigned raw_disp_mask;                     // the caller's raw bits (only s >= 1 are read)
  const float* intrinsics;                    // the caller's (B, ns, 3, 3)
  float* k0;                                  // (B, ns, 3, 3): K_0 at every scale
  int zero_gup;                               // the march accumulates into gup: the upsample kernel zeroes it
  int accum;                                  // a smoothness kernel wrote gdisp: the adjoint adds to it
};
struct SfmUpGrid {
  int blk_begin[SFM_MAX_SCALES + 1];          // adjoint blocks of scale s: [blk_begin[s], blk_begin[s+1])
};
// first in the step's chain, without PDL: U_s(d_s), the zeroed gradient planes and the K_0 copy
int sfm_launch_full_res_upsample(const SfmFullRes& f, cudaStream_t stream);
// last, a dependent launch behind the epilogue: gdisp[s] (+)= U_s^T(gup[s]) (times d disp / d x for the raw bits)
int sfm_launch_full_res_adjoint(const SfmFullRes& f, cudaStream_t stream);
// gintrinsics[:, 0] = sum over the scales, [:, 1:] = 0; a dependent launch behind the intrinsics-gradient kernel
int sfm_launch_intrinsics_fold(int B, int ns, float* gintrinsics, cudaStream_t stream);
int sfm_launch_upsample_stage(int N, int h, int w, int H, int W, const float* x, float* y, cudaStream_t stream);
