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
};

// sm_mode: 0 = no smoothness tasks, 1 = loss only, 2 = loss + gdisp
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
  const float* sm_part;     // loss partials of the smoothness CTAs of the prologue kernel
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

// Launch plan of one fused step (plan.cu, the whole launch policy).  The marching kernel instance is
// sfm_l1_march_kernel<exp, grad, accum, debug, raw> or sfm_ssim_march_kernel<grad, accum, debug, raw, nw, srec>.
struct SfmStepPlan {
  bool ssim;                           // kernel family
  bool exp, grad, accum, debug, raw;   // accum: a smoothness kernel has initialised gdisp
  int nw;                              // SSIM: warps per CTA (2: the two sources split over the warps of a CTA)
  bool srec;                           // SSIM: forward records in shared memory (false: in registers)
  bool edge_smooth;                    // the edge-aware smoothness kernel runs between the prologue and the march
  SfmTaskTable tasks;
  SfmSmoothParams smooth;              // second-order smoothness tasks of the prologue (n_ctas == 0: none)
  int band, n_mix_region;              // SfmPrepParams
};
// mode bits of the planner
enum { SFM_MODE_EXP = 1, SFM_MODE_SSIM = 2, SFM_MODE_GRAD = 4, SFM_MODE_DEBUG = 8, SFM_MODE_SMOOTH = 16 };
SfmStepPlan sfm_plan_step(const SfmDesc* d, int mode, int num_sms);
int sfm_plan_band(const SfmDesc* d);
int sfm_launch_fused(SfmFusedParams& p, const SfmStepPlan& plan, cudaStream_t stream);
int sfm_launch_edge_smooth(const SfmFusedParams& p, bool grad, cudaStream_t stream);   // smooth.cu
extern thread_local cudaEvent_t sfm_ev_start, sfm_ev_stop;   // profiling hook (sfm_set_kernel_events)

int sfm_launch_scale(float* const* ptrs, const long long* counts, int n, const float* gy, cudaStream_t stream);
