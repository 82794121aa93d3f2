/*
 * sfmloss.h -- C ABI of libsfmloss.so: the SfM-Learner view-synthesis loss path on B200 (sm_100a).
 *
 * This is the drop-in boundary for the hot path of pfnet/sfm-learner-chainer.  Every entry point
 * cites the reference interface it replaces (paths relative to the reference repo root).
 * The reference-side binding (ctypes + Chainer FunctionNode) is shown in INTEGRATION.md.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no torch / cupy types.
 *  - All tensors are float32, C-contiguous, resident on the CURRENT CUDA device; the caller owns
 *    every buffer (CuPy memory pool, torch allocator, cudaMalloc ...).  The library never frees or
 *    retains caller pointers after a call returns, except inside an SfmHostCtx it created itself.
 *  - Every call is asynchronous on `stream` (0 = legacy default stream), performs no host
 *    synchronisation and no D2H copy, and is capturable in a CUDA graph (the *_host entry point is
 *    the exception: it copies and synchronises by contract).
 *  - Return value: 0 = OK, < 0 = SFM_E_* argument error, > 0 = cudaError_t.  The message of the
 *    last failure on the calling thread is available from sfm_last_error().
 *  - There is NO CPU fallback: without a CUDA device the compute entry points return an error.
 */
#ifndef SFMLOSS_H_
#define SFMLOSS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SFM_VERSION 102           /* major*100 + minor */
#define SFM_MAX_SCALES 4          /* base_model.py:66 (len(pred_depthes) == 4) */
#define SFM_MAX_SOURCES 8         /* seq_len-1; shipped configs use 2 and 4 */

/* error codes */
#define SFM_OK 0
#define SFM_E_INVALID_DESC (-1)
#define SFM_E_INVALID_SHAPE (-2)
#define SFM_E_NULL_POINTER (-3)
#define SFM_E_UNSUPPORTED (-4)
#define SFM_E_NO_DEVICE (-5)
#define SFM_E_COMM (-6)           /* a collective failed (NCCL error in sfm_last_error) */

/* SfmDesc.flags */
#define SFM_FLAG_TABLES_PROVIDED 0x1u /* caller supplies proj/kinv tables (bit-exact tests; the reference
                                         itself builds P on the host, transform.py:76-90) */
#define SFM_FLAG_REUSE_PYRAMID 0x2u   /* workspace already holds this batch's image pyramid (sfm_pyramid); in->tgt / in->src
                                         are still read (scale 0 is never copied) */
#define SFM_FLAG_NO_TMA 0x4u          /* reserved (accepted and ignored: the marching kernels stage nothing through TMA) */
#define SFM_FLAG_EDGE_AWARE_SMOOTH 0x8u /* the smoothness term is compute_disp_smooth(curr_tgt_img, pred_disps[ns])
                                         (base_model.py:144-155), the edge-aware alternative the reference keeps
                                         commented out at its call site (:78-80), instead of compute_smooth_loss */
#define SFM_FLAG_IMAGE_GRADS 0x10u    /* the workspace also holds fp32 gradient levels of the pyramid (scales >= 1) for
                                         sfm_loss_forward_backward_images; every other entry point accepts the flag and
                                         behaves exactly as without it */
#define SFM_FLAG_SNIPPET_TERMS 0x20u  /* the workspace also holds 4 fp64 loss cells per snippet and one float per smoothness
                                         task for sfm_loss_snippets; every other entry point accepts the flag and behaves
                                         exactly as without it */
#define SFM_FLAG_MIN_REPROJECTION 0x40u /* the workspace also holds B*S*sum_s h_s*w_s floats, the per-(pixel, source) error /
                                         weight planes of sfm_loss_min_reprojection; every other entry point accepts the
                                         flag and behaves exactly as without it */
#define SFM_FLAG_FULL_RES_MULTISCALE 0x80u /* Monodepth2's full-resolution multi-scale loss (Godard et al., ICCV 2019, §3
                                         "multi-scale estimation"): the photometric terms of every scale are computed at
                                         full resolution on the upsampled disparity; see "Full-resolution multi-scale"
                                         below.  Changes the loss and sizes the workspace */
#define SFM_FLAG_MEAN_NORM_SMOOTH 0x100u /* Monodepth2's mean-normalised smoothness: the smoothness term of every scale is
                                         evaluated on d_s / (mean(d_s) + 1e-7); see "Mean-normalised smoothness" below.
                                         Changes the loss and sizes the workspace */
#define SFM_FLAG_EDGE_MEAN_ABS 0x200u /* with SFM_FLAG_EDGE_AWARE_SMOOTH: Monodepth2's edge weight exp(-mean_c |dI_c|) instead
                                         of the reference's exp(-|mean_c dI_c|) (else SFM_E_INVALID_DESC) */
#define SFM_FLAG_BORDER_PADDING 0x400u /* Monodepth2's image borders: border-clamped sampling without the out-of-view mask
                                         and reflection-padded SSIM windows; see "Border padding" below.  Changes the
                                         loss; does not size the workspace */
#define SFM_FLAG_AXISANGLE_POSE 0x800u /* Monodepth2's pose: `poses` rows are (v0, v1, v2, tx, ty, tz), an axis-angle
                                         vector and a translation, instead of the Euler vector; see "Axis-angle pose"
                                         below.  Does not size the workspace */
#define SFM_FLAG_GEOMETRY_CONSISTENCY 0x1000u /* the workspace also holds the self-discovered mask planes and the per-pixel
                                         map planes of sfm_loss_geometry (B*S*sum_s h_s*w_s floats each); see "Geometry
                                         consistency" below.  Every other entry point accepts the flag and behaves exactly
                                         as without it */
#define SFM_FLAG_POSE_INVERT_SHIFT 16   /* flags bits 16..23: with SFM_FLAG_AXISANGLE_POSE, bit 16 + i inverts the
                                         transform of source i (Monodepth2's frame ids < 0) */
#define SFM_FLAG_POSE_INVERT(i) (1u << (SFM_FLAG_POSE_INVERT_SHIFT + (i)))
#define SFM_FLAG_POSE_INVERT_MASK (0xffu << SFM_FLAG_POSE_INVERT_SHIFT)

/*
 * Problem descriptor.  Mirrors the reference's model flags (base_model.py:37-39:
 * smooth_reg, exp_reg, ssim_rate; experiments/sfm_learner_v1*.yml `architecture:` blocks) and the
 * tensor shapes SFMLearner.__call__ receives (base_model.py:48-58).
 * A flag equal to 0 disables its term (any non-zero value, negative included, enables it) exactly like the
 * Python truthiness tests at base_model.py:75,86,103,112;
 * the explainability branch and SSIM are mutually exclusive as in the reference (:103-115).
 */
typedef struct SfmDesc {
  int32_t B;         /* snippets held by this process                                  */
  int32_t S;         /* source views per snippet (seq_len - 1)                         */
  int32_t H, W;      /* full resolution; scale s is (H >> s, W >> s)                   */
  int32_t n_scales;  /* 1..SFM_MAX_SCALES                                              */
  int32_t B_global;  /* batch every F.mean divides by (0 = B); > B when snippet-sharded */
  float smooth_reg;
  float exp_reg;
  float ssim_rate;
  uint32_t flags;
  /* Producer-side fusion at the seam with the two CNNs (both default to 0 = off):
   * raw_disp_scales  bit s set: disps[s] holds the PRE-activation output of DispNet's `dispout` convolution
   *                  and the kernels apply disp = DISP_SCALING * sigmoid(x) + MIN_DISP themselves
   *                  (models/disp_net.py:7-8,104,110,116,122); gdisps[s] is then the gradient w.r.t. x.
   *                  Scale 0 (disp1) is consumed by the loss alone; disp2..4 are also fed back into the
   *                  decoder (disp_net.py:105,111,117), so a drop-in normally sets bit 0 only.
   * raw_pose_hw      n > 0: poses holds PoseNet's `poseout` map (B, 6*S, n) with n = h'*w' spatial positions
   *                  and the kernels apply pose = 0.01 * mean over n (models/pose_net.py:51-53); gposes then
   *                  has the same (B, 6*S, n) shape.  n <= 128.                                             */
  uint32_t raw_disp_scales;
  int32_t raw_pose_hw;
} SfmDesc;

/* Inputs of one loss evaluation.  Shapes as produced by the reference's nets and dataset:
 *   tgt        (B,3,H,W)            base_model.py:48
 *   src        (B,S,3,H,W)          base_model.py:57-58 (== stacked (B,3S,H,W))
 *   intrinsics (B,n_scales,3,3)     datasets/kitti/kitti_raw_transformed.py:76-93
 *   disps[s]   (B,1,H>>s,W>>s)      models/disp_net.py:124   (disparity, NOT depth; pre-activation map when
 *                                   bit s of desc->raw_disp_scales is set)
 *   poses      (B,S,6)              models/pose_net.py:52-54 (rx,ry,rz,tx,ty,tz per source); (B,6*S,n) raw
 *                                   `poseout` map when desc->raw_pose_hw = n > 0
 *   logits[s]  (B,S,H>>s,W>>s)      models/pose_net.py:56-67; may be NULL when exp_reg == 0
 *   proj       (B,S,n_scales,3,4)   only with SFM_FLAG_TABLES_PROVIDED: K4.T rows 0..2 (transform.py:86-88)
 *   kinv       (B,n_scales,3,3)     only with SFM_FLAG_TABLES_PROVIDED: inverse intrinsics (transform.py:105)
 */
typedef struct SfmInputs {
  const float* tgt;
  const float* src;
  const float* intrinsics;
  const float* disps[SFM_MAX_SCALES];
  const float* poses;
  const float* logits[SFM_MAX_SCALES];
  const float* proj;
  const float* kinv;
} SfmInputs;

/* Gradients w.r.t. the network outputs (base_model.py:59-63 are the producers).  Same shapes as the
 * corresponding inputs.  glogits may be NULL when exp_reg == 0. */
typedef struct SfmGrads {
  float* gdisps[SFM_MAX_SCALES];
  float* gposes;
  float* glogits[SFM_MAX_SCALES];
} SfmGrads;

/* Gradients w.r.t. the two images (sfm_loss_forward_backward_images), same shapes as SfmInputs.tgt / .src:
 *   gtgt (B,3,H,W), gsrc (B,S,3,H,W).  Either may be NULL (that gradient is not computed), not both. */
typedef struct SfmImageGrads {
  float* gtgt;
  float* gsrc;
} SfmImageGrads;

/* Optional per-(scale, source) dumps of the warp for stage-level parity tests (may be NULL):
 *   P[s]   (B,S,3,h,w) f32  warped image            (transform.py:189)
 *   u0[s]  (B,S,h,w)   i32  floor(u), v0 likewise   (integer work: must be bit-exact)
 *   inb[s] (B,S,h,w)   u8   strict in-bounds flag   (transform.py:128-131)               */
typedef struct SfmDebug {
  float* P[SFM_MAX_SCALES];
  int32_t* u0[SFM_MAX_SCALES];
  int32_t* v0[SFM_MAX_SCALES];
  uint8_t* inb[SFM_MAX_SCALES];
} SfmDebug;

int sfm_version(void);
const char* sfm_last_error(void);

/* Bytes of device scratch a call needs (image pyramid of the scales >= 1, planar like the inputs; projection
 * tables; fp64 reduction cells; with SFM_FLAG_IMAGE_GRADS also the fp32 gradient levels of the pyramid).  The caller allocates it (any 256-byte aligned device pointer) and passes it to
 * every call with the same descriptor.  Scale 0 is read straight from in->tgt / in->src. */
size_t sfm_workspace_bytes(const SfmDesc* desc);

/* losses_out: device float[5] = total, pixel, smooth, exp, ssim  (chainer.report keys,
 * base_model.py:119-123).  Under snippet sharding they are this shard's partial sums; add across
 * ranks (one allreduce of 5 floats). */

/* Forward only.  Replaces SFMLearner.__call__'s loss loop, base_model.py:64-118
 * (F.resize_images :71-72, projective_inverse_warp transform.py:156-193, compute_smooth_loss :169-185,
 * compute_exp_reg_loss :157-167, compute_ssim :126-142). */
int sfm_loss_forward(const SfmDesc* desc, const SfmInputs* in, float* losses_out, const SfmDebug* debug,
                     void* workspace, void* stream);

/* Backward only (recomputes the forward).  Replaces loss.backward() through the graph recorded by
 * base_model.py:64-118.  gy: device float* holding dL/dloss, or NULL for 1. */
int sfm_loss_backward(const SfmDesc* desc, const SfmInputs* in, const float* gy, const SfmGrads* grads,
                      void* workspace, void* stream);

/* Fused single pass: losses and gradients (for upstream gradient 1) in one sweep.  This is what the
 * Chainer adapter calls from forward(); its backward() only rescales (sfm_scale_grads). */
int sfm_loss_forward_backward(const SfmDesc* desc, const SfmInputs* in, float* losses_out,
                              const SfmGrads* grads, void* workspace, void* stream);

/* grads *= *gy (device scalar).  No-op on the device when *gy == 1. */
int sfm_scale_grads(const SfmDesc* desc, const float* gy, const SfmGrads* grads, void* stream);

/* sfm_loss_forward_backward plus the gradients of the reported total (losses_out[0]) w.r.t. the images, for callers
 * whose images come out of a differentiable module.  The images are treated as differentiable throughout: the
 * reference's `.data` on the pyramid (base_model.py:71-72) and on mu_y / sigma_y (:131,:134) are lifted, so igrads is
 * the derivative of the reported value.  The all-zero mask (:96) is piecewise constant and has derivative 0.
 * desc->flags must contain SFM_FLAG_IMAGE_GRADS (else SFM_E_INVALID_DESC; the workspace is sized with it); with
 * SFM_FLAG_EDGE_AWARE_SMOOTH it returns SFM_E_UNSUPPORTED (that term depends on the target image).  Losses, gdisps
 * and glogits are bitwise those of sfm_loss_forward_backward.  gtgt is bitwise reproducible from run to run; gsrc
 * is accumulated with fp32 atomics and its last bits vary with their order.  Under snippet sharding (B_global > B)
 * a shard's image gradients are final. */
int sfm_loss_forward_backward_images(const SfmDesc* desc, const SfmInputs* in, float* losses_out, const SfmGrads* grads,
                                     const SfmImageGrads* igrads, void* workspace, void* stream);

/* igrads *= *gy (device scalar), the NULL members skipped.  No-op on the device when *gy == 1. */
int sfm_scale_image_grads(const SfmDesc* desc, const float* gy, const SfmImageGrads* igrads, void* stream);

/* d(reported total)/d intrinsics (B,n_scales,3,3) times the call's gy, from the dL/dP cells that the last
 * gradient-producing call (sfm_loss_backward, _forward_backward, _forward_backward_peer, _forward_backward_images)
 * left in `workspace`: same desc, inputs and stream, before the next call on that workspace.  For callers that learn
 * their camera.  K_s = intrinsics[:, s] is treated as differentiable in both places the reference uses it: the
 * projection K4.[R|t] (transform.py:86-88) and pixel2cam's batch_inv(K) (:105).  Per (snippet, scale) it is
 *   sum_i [ A_i R_i^T + g_i t_i^T - K_s^-T R_i^T K_s^T A_i ],   [A_i | g_i] = dL/dP of source i at scale s,
 * evaluated in fp64 on the device (a dependent launch; graph-capturable).  Under snippet sharding (B_global > B) a
 * shard's gradient is final.  With SFM_FLAG_TABLES_PROVIDED it returns SFM_E_UNSUPPORTED: the step then did not build
 * the projection and K^-1 from the intrinsics. */
int sfm_intrinsics_grad(const SfmDesc* desc, const SfmInputs* in, const void* workspace, float* gintrinsics, void* stream);

/* gintrinsics *= *gy (device scalar).  No-op on the device when *gy == 1. */
int sfm_scale_intrinsics_grad(const SfmDesc* desc, const float* gy, float* gintrinsics, void* stream);

/* Per-snippet weights and per-snippet loss values (sfm_loss_snippets).  Every term of the loss is a sum over the
 * snippets, total = sum_b l_b with the 1/B_global means inside each l_b, so the weighted loss sum_b w_b * l_b is linear
 * in the weights and d total / d w_b = l_b[0].  Weights held in device memory let one captured CUDA graph run batches
 * with fewer real snippets: pad to the captured B with copies of a real snippet, keep B_global = B and pass
 * w_b = B / B_real for the real snippets and 0 for the padding.  Any float is accepted (0 and negative ones included);
 * a non-finite weight propagates. */
typedef struct SfmSnippetTerms {
  const float* weights;  /* (B) device: w_b, or NULL = all 1 */
  float* losses;         /* (B,5) device: l_b = total, pixel, smooth, exp, ssim of snippet b (unweighted, with the
                            1/B_global means), or NULL */
} SfmSnippetTerms;


/* Profiling hook (bench.py's roofline measurement): while set (non-NULL cudaEvent_t handles), every
 * sfm_loss_* call on this thread records `start` right before and `stop` right after the fused loss
 * kernel, on the call's stream.  Pass NULL, NULL to clear. */
int sfm_set_kernel_events(void* start_event, void* stop_event);

/* Image pyramid only (F.resize_images from full resolution, base_model.py:70-72; scales 1..n_scales-1, scale 0 is
 * the identity and is never copied) into the workspace; sfm_pyramid_export copies one level (scale >= 1) back
 * out for tests: tgt_out (B,3,h,w), src_out (B,S,3,h,w). */
int sfm_pyramid(const SfmDesc* desc, const float* tgt, const float* src, void* workspace, void* stream);
int sfm_pyramid_export(const SfmDesc* desc, const void* workspace, int scale, float* tgt_out, float* src_out,
                       void* stream);

/* Projection tables on the device: proj_out (B,S,n_scales,3,4), kinv_out (B,n_scales,3,3).
 * Replaces proj_tgt_to_src / pose_vec2mat / euler2mat (transform.py:11-91) and F.batch_inv(K) (:105),
 * including the five blocking host<->device copies per (scale, source) of models/utils.py:33-84. */
int sfm_build_tables(const SfmDesc* desc, const float* poses, const float* intrinsics, float* proj_out,
                     float* kinv_out, void* stream);

/* Stage API of the producer-side fusions (the same device code the fused kernels inline; the parity tests
 * use it to show raw-input mode == activation stage + plain mode bit for bit):
 * sfm_disp_activation: disp[k] = DISP_SCALING * sigmoid(x[k]) + MIN_DISP (disp_net.py:104) for n elements,
 * optional dact[k] = d disp / d x.   sfm_pose_reduce: x (B, 6*S, hw) -> poses (B, S, 6) = 0.01 * mean
 * (pose_net.py:52-53). */
int sfm_disp_activation(long long n, const float* x, float* disp, float* dact, void* stream);
int sfm_pose_reduce(int B, int S, int hw, const float* x, float* poses_out, void* stream);

/* Data layer in front of the loss path, as one device gather (datasets/kitti/kitti_raw_dataset.py:12-14
 * load_as_float_norm; datasets/kitti/kitti_raw_transformed.py:23-74 data_augmentation and :76-93
 * get_multi_scale_intrinsics).  The caller draws the random numbers exactly as the reference does and passes
 * them per snippet; NULL `aug` = no augmentation (validation split). */
typedef struct SfmAugment {
  int32_t out_h, out_w;        /* size after random scaling: int(H * y_scaling), int(W * x_scaling)  (:36-37)  */
  int32_t off_y, off_x;        /* random crop offsets in the rescaled image                         (:49-50)  */
  int32_t flip;                /* != 0: horizontal flip                                             (:63-65)  */
  int32_t reserved_;
  double x_scaling, y_scaling; /* np.random.uniform(1, 1.15, 2), used for the intrinsics            (:34-42)  */
} SfmAugment;
/* frames (B, 1+S, H, W, 3) uint8 HWC on the device, frame 0 of a snippet = target (imread order); K_in (B,3,3);
 * aug: device array of B SfmAugment or NULL.  Outputs: tgt_out (B,3,H,W), src_out (B,S,3,H,W) float32 in
 * [-1, 1]; intrinsics_out (B,n_scales,3,3) or NULL. */
int sfm_ingest_u8(int B, int S, int H, int W, int n_scales, const uint8_t* frames, const float* K_in,
                  const SfmAugment* aug, float* tgt_out, float* src_out, float* intrinsics_out, void* stream);

/* Inference-side depth evaluation of one batch (evaluate.py:94-103 + kitti_eval/depth_util.py:6-22), on the
 * device: pred_depth (B,1,h,w) is resized to the ground truth's (Hg,Wg) (F.resize_images), clipped to
 * [min_depth, max_depth], masked, scaled by median(gt)/median(pred) (exact medians) and compared.
 * gt_depth (B,Hg,Wg) float32, mask (B,Hg,Wg) uint8 (non-zero = valid; masked depths must be positive).
 * errors_out: device float[8] = abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3 (depth_util.py:22) and the scale
 * factor.  scratch: sfm_eval_depth_scratch_bytes(B,Hg,Wg) bytes of device memory.  Asynchronous on `stream`. */
size_t sfm_eval_depth_scratch_bytes(int B, int Hg, int Wg);
int sfm_eval_depth(int B, int h, int w, int Hg, int Wg, const float* pred_depth, const float* gt_depth,
                   const uint8_t* mask, float min_depth, float max_depth, float* errors_out, void* scratch,
                   void* stream);

/* Stage API: projective_inverse_warp(imgs, depthes, poses, K) of transform.py:156-165 on N images of
 * one resolution.  imgs (N,3,h,w) NCHW, depth (N,h*w) [the reference passes it broadcast to 3 rows],
 * poses (N,6), K (N,3,3); proj (N,3,4) / kinv (N,3,3) optional overrides (NULL = built on device).
 * Outputs: out (N,3,h,w); optional u0,v0 (N,h,w) int32 and inb (N,h,w) uint8. */
int sfm_warp_forward(int N, int h, int w, const float* imgs, const float* depth, const float* poses,
                     const float* K, const float* proj, const float* kinv, float* out, int32_t* u0,
                     int32_t* v0, uint8_t* inb, void* stream);
/* Backward of the above for upstream gy (N,3,h,w): gdepth (N,h*w), gposes (N,6), optional gimgs
 * (N,3,h,w; the reference discards it, base_model.py:71-72 `.data`).  scratch: device buffer of
 * sfm_warp_backward_scratch_bytes(N) bytes. */
size_t sfm_warp_backward_scratch_bytes(int N);
int sfm_warp_backward(int N, int h, int w, const float* imgs, const float* depth, const float* poses,
                      const float* K, const float* gy, float* gdepth, float* gposes, float* gimgs,
                      void* scratch, void* stream);

/* SpatialTransformerSamplerInterp (models/spational_transformer_sampler_interp.py:9-159, the repo-local
 * sampler the live path leaves commented out, transform.py:190-191): grid in PIXEL units, indices
 * clamped to the image.  x (B,C,H,W), grid (B,2,oH,oW) -> y (B,C,oH,oW);  backward returns ggrid
 * (B,2,oH,oW) and gx = zeros (:148). */
int sfm_sampler_interp_forward(int B, int C, int H, int W, int oH, int oW, const float* x, const float* grid,
                               float* y, void* stream);
int sfm_sampler_interp_backward(int B, int C, int H, int W, int oH, int oW, const float* x, const float* grid,
                                const float* gy, float* gx, float* ggrid, void* stream);

/* Host-buffer convenience path (what a CPU-resident caller, e.g. a Chainer numpy run or the end-to-end
 * benchmark, uses): owns device buffers, copies inputs H2D, runs sfm_loss_forward_backward, copies
 * losses and gradients D2H and synchronises.  All pointers in `in`, `grads` and `losses_out` are HOST
 * pointers here (pinned memory makes the copies asynchronous). */
typedef struct SfmHostCtx SfmHostCtx;
int sfm_host_ctx_create(const SfmDesc* desc, SfmHostCtx** ctx_out);
int sfm_host_ctx_destroy(SfmHostCtx* ctx);
int sfm_loss_step_host(SfmHostCtx* ctx, const SfmInputs* in, float* losses_out, const SfmGrads* grads);
/* The same step split in two, for callers that keep several steps in flight (a data loader that prepares
 * step k+1 while step k runs): _submit enqueues the H2D copies, the kernels and the D2H copies on the context's
 * own stream and returns; _wait blocks until they are done.  The host buffers of a submitted step must stay
 * valid (and, for the outputs, untouched) until _wait returns.  With two contexts used alternately the copies of
 * one step overlap the kernels of the other (pinned memory required for the overlap).  Host arrays of one kind (disps,
 * logits, gdisps, glogits) that lie back to back in scale order are moved in ONE copy each (every copy has a fixed cost of
 * several microseconds); separate arrays work the same, one copy per scale. */
int sfm_loss_step_host_submit(SfmHostCtx* ctx, const SfmInputs* in, float* losses_out, const SfmGrads* grads);
int sfm_loss_step_host_wait(SfmHostCtx* ctx);

/* The host-buffer step fed by the data layer's raw material: `frames` (B, 1+S, H, W, 3) uint8 HWC, `K_in` (B,3,3)
 * and `aug` (B SfmAugment or NULL) are HOST pointers; the images and intrinsics of `in` are ignored (sfm_ingest_u8
 * produces them on the device), its disps / poses / logits are host pointers as in sfm_loss_step_host_submit.
 * The H2D copy carries 1 byte per image sample instead of 4.  Complete with sfm_loss_step_host_wait. */
int sfm_loss_step_host_u8_submit(SfmHostCtx* ctx, const uint8_t* frames, const float* K_in, const SfmAugment* aug,
                                 const SfmInputs* in, float* losses_out, const SfmGrads* grads);

/* ---- Multi-GPU: the path shards by snippet (SfmDesc.B_global), gradients need no communication, and the five loss
 * partials are completed by ONE all-reduce (sum, float32) per step.  Replaces the reduce of Chainer's
 * MultiprocessParallelUpdater (config_utils.py:123-126, unused by the shipped configs) for this path.
 * One process per GPU.  The communicator wraps an NCCL communicator (bound at run time with dlopen, so the library
 * loads without NCCL; sfm_nccl_set_library names the shared object when the process has not loaded one already):
 *   rank 0:      sfm_comm_unique_id(id)            -> 128 opaque bytes, handed to the other ranks by the host program
 *                                                     (MPI, torch.distributed, a file ...)
 *   every rank:  sfm_comm_create(id, nranks, rank, &comm)     collective, on the rank's current device
 *   every step:  sfm_allreduce_partials(comm, losses, 5, stream)   in place on the device array `losses`; enqueued on
 *                                                     `stream` (after the loss call that wrote it), asynchronous,
 *                                                     capturable in a CUDA graph together with the step
 *   at the end:  sfm_comm_destroy(comm)           after every CUDA graph that captured the all-reduce has been destroyed
 *                                                 (such a graph holds a reference on the NCCL communicator)          */
#define SFM_NCCL_UNIQUE_ID_BYTES 128
typedef struct SfmComm SfmComm;
int sfm_nccl_set_library(const char* path);
int sfm_nccl_version(void);                /* ncclGetVersion code (e.g. 22809), 0 when NCCL cannot be loaded */
int sfm_comm_unique_id(void* id_out);
int sfm_comm_create(const void* unique_id, int nranks, int rank, SfmComm** comm_out);
int sfm_comm_destroy(SfmComm* comm);
int sfm_allreduce_partials(SfmComm* comm, float* losses, int count, void* stream);

/* The same sum WITHOUT a collective call: the epilogue kernel of the step exchanges the five partials over NVLink
 * peer memory itself (every rank owns a small slot array that the other ranks' epilogues write with peer stores; CUDA
 * IPC maps the arrays across the processes) and adds them in rank order, so losses_out holds bitwise the same global
 * sums on every rank when the step's kernels are done -- no extra launch, no library latency on the step.
 *   every rank:  sfm_peer_create(nranks, rank, &peer, handle)   -> 64 opaque bytes (a cudaIpcMemHandle_t)
 *   host side:   all-gather the handles of all ranks in rank order (nranks x 64 bytes)
 *   every rank:  sfm_peer_connect(peer, all_handles); then a host barrier before the first step
 *   every step:  sfm_loss_forward_backward_peer(desc, in, losses_out, grads, workspace, peer, stream)
 *                (graph-capturable; every rank must run the same number of steps: step k of one rank waits, inside the
 *                 epilogue kernel and for at most ~2 s, for step k of the others; on that timeout the losses are NaN)
 *   at the end:  a host barrier, then sfm_peer_destroy(peer)
 * One node, one process per GPU, up to 16 ranks, GPUs with peer access (NVLink / NVSwitch).                        */
#define SFM_IPC_HANDLE_BYTES 64
typedef struct SfmPeer SfmPeer;
int sfm_peer_create(int nranks, int rank, SfmPeer** peer_out, void* ipc_handle_out);
int sfm_peer_connect(SfmPeer* peer, const void* all_handles);
int sfm_peer_destroy(SfmPeer* peer);
int sfm_loss_forward_backward_peer(const SfmDesc* desc, const SfmInputs* in, float* losses_out, const SfmGrads* grads,
                                   void* workspace, SfmPeer* peer, void* stream);

/* losses_out = sum_b w_b * l_b (under `peer`: summed over the ranks as sfm_loss_forward_backward_peer does), and every
 * gradient is that of losses_out[0].  grads == NULL: forward only.  igrads: as sfm_loss_forward_backward_images (needs
 * SFM_FLAG_IMAGE_GRADS and grads; not with SFM_FLAG_EDGE_AWARE_SMOOTH).  peer: as sfm_loss_forward_backward_peer (may be
 * NULL); terms->losses stays per rank.  A non-NULL member of `terms` needs SFM_FLAG_SNIPPET_TERMS in desc->flags (else
 * SFM_E_INVALID_DESC); terms == NULL or both members NULL is the plain step of the same grads / igrads / peer.  The
 * weighted sums run in fp64 in a fixed snippet order; with all weights 1 the gradients are bitwise those of the plain
 * step and the losses agree to rounding.  sfm_intrinsics_grad after this call returns the weighted gradient. */
int sfm_loss_snippets(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms, float* losses_out,
                      const SfmGrads* grads, const SfmImageGrads* igrads, void* workspace, SfmPeer* peer, void* stream);

/* Per-pixel weights and per-pixel loss maps (sfm_loss_weighted).  M_s = weights[s] is a (B,S,h_s,w_s) array laid out
 * like logits[s]; it multiplies the per-pixel photometric terms of source i at scale s, broadcast over the 3 channels,
 * and the means keep their denominators B_global*3*h*w (as the explainability weighting does):
 *   pixel_loss += mean(E * sigma(l) * M)   (exp branch; mean(E * M) otherwise)
 *   ssim_loss  += mean(clip((1 - SSIM) / 2, 0, 1) * (1 - m_zero) * M)
 * The smoothness term and the explainability regulariser are not weighted.  Every gradient (gdisps, gposes, glogits and
 * the dL/dP cells, hence sfm_intrinsics_grad) is that of the weighted total.  The loss is linear in M, so the map
 *   losses[s][b,i,y,x] = d losses_out[0] / d M
 *     = w_b * [ (1 - ssim_rate) * sigma(l) * sum_c E_c + ssim_rate * sum_c clip(raw_c, 0, 1) * (1 - m_zero) ] / (B_global*3*h_s*w_s)
 * (sigma = 1 without the exp branch, the SSIM part only when SSIM runs, w_b the snippet weight or 1) is each pixel's
 * share of the photometric loss: sum M * map = (1 - ssim_rate) * pixel + ssim_rate * ssim.  Uses: validity or semantic
 * masks (moving objects, the ego-vehicle, rectification borders, sky), per-source confidence maps, learned weight maps
 * (their gradient is the map), and per-pixel loss maps for validation and outlier search.  Any float weight is
 * accepted, 0 and negative ones included; a non-finite weight propagates.  The maps are written with plain stores, each
 * pixel once: bitwise reproducible from run to run. */
typedef struct SfmPixelTerms {
  const float* weights[SFM_MAX_SCALES];  /* (B,S,h_s,w_s) device, or NULL = 1 at that scale */
  float* losses[SFM_MAX_SCALES];         /* (B,S,h_s,w_s) device: d losses_out[0] / d weights, or NULL */
} SfmPixelTerms;

/* sfm_loss_snippets with per-pixel terms.  pix == NULL, or every member of the scales < n_scales NULL, is exactly
 * sfm_loss_snippets of the other arguments (members of scales >= n_scales are ignored).  Maps may be requested with or
 * without weights and with or without grads (grads == NULL: forward only, the validation use).  Composes with snippet
 * terms, the peer sum (the maps stay per rank), raw disparity / pose, edge-aware smoothness, SFM_FLAG_TABLES_PROVIDED,
 * SFM_FLAG_REUSE_PYRAMID and sfm_intrinsics_grad afterwards.  Per-pixel terms together with igrads return
 * SFM_E_UNSUPPORTED.  With all weights 1 (or NULL) the losses are bitwise those of the step without per-pixel terms run
 * with the same plan, and so are gdisps and glogits without SSIM (with SSIM gdisps agree to the last bits). */
int sfm_loss_weighted(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms, const SfmPixelTerms* pix,
                      float* losses_out, const SfmGrads* grads, const SfmImageGrads* igrads, void* workspace, SfmPeer* peer,
                      void* stream);

/* Per-pixel minimum reprojection and auto-masking over the source views (Godard et al., "Digging Into Self-Supervised
 * Monocular Depth Estimation", ICCV 2019), sfm_loss_min_reprojection.  The reference's photometric loss is a mean over
 * the source views of every (pixel, source) error; here each target pixel is scored on the one source that explains it
 * best, so a pixel occluded in one source is scored on a source where it is visible, and (auto-masking) a pixel is
 * dropped when an UNWARPED source already matches the target at least as well (a static camera, objects that move with
 * the camera).  Per scale s, snippet b, target pixel p, source i, with r = ssim_rate:
 *   reprojection error  e_i(p) = (1 - r) * sum_c E_c + r * sum_c clip((1 - SSIM_c) / 2, 0, 1) * (1 - m)
 *                       the per-pixel map of sfm_loss_weighted without its 1/(B_global*3*h*w) factor, without gy and
 *                       without snippet weights; the SSIM part only when SSIM runs (ssim_rate != 0).
 *   candidates          source i is a candidate at p only where its all-zero mask m (base_model.py:96) is 0; every
 *                       out-of-view pixel is masked (the x2 rule makes the warped value exactly 0).  A masked source is
 *                       NOT a candidate with error 0 (it would always win).
 *   identity error      e_id_i(p): the same formula with the warped image replaced by source i's own pyramid level at p
 *                       (scale 0: the caller's tensor), no mask, the same 3x3 zero-padded windows as the reference SSIM.
 *   selection           sel(p) = -2 when p has no candidate; else i* = argmin over the candidates of e_i(p), ties to the
 *                       lowest index; with automask, sel(p) = -1 when e_i*(p) >= min_i e_id_i(p) (a strict < keeps the
 *                       pixel), else sel(p) = i*.  The selection uses neither snippet weights nor gy, so a negative
 *                       snippet weight cannot turn the minimum into a maximum.
 *   loss                the loss of sfm_loss_weighted with the one-hot weights M_i(p) = [sel(p) = i].  The means keep their
 *                       denominators, so the photometric part is the mean over the pixels of the per-pixel minimum;
 *                       losses_out[1] (pixel) and [4] (ssim) are the L1 and SSIM parts of the chosen terms; smoothness
 *                       (either kind) is unchanged.  Every gradient (gdisps, gposes, the dL/dP cells, hence
 *                       sfm_intrinsics_grad afterwards) is that of this total; the selection is piecewise constant and
 *                       has derivative 0.
 * Auto-masked pixels contribute 0 to the reported value, as the paper's mask mu does.  Monodepth2's code instead adds the
 * identity error of those pixels to the reported value; that part carries no disparity, pose or intrinsics gradient, so
 * the gradients are the same either way and only the reported value differs.
 * Computed in two marches on the device (graph-capturable): a forward march writes every e_i into the workspace planes,
 * a select kernel computes the identity errors and turns the planes into the one-hot weights, and the march of
 * sfm_loss_weighted runs with them. */
typedef struct SfmMinReprojection {
  int32_t automask;                       /* != 0: auto-masking on */
  int32_t reserved_;                      /* 0 (else SFM_E_INVALID_DESC) */
  int8_t* selection[SFM_MAX_SCALES];      /* (B,h_s,w_s) device: sel(p) in {-2, -1, 0 .. S-1}, or NULL */
} SfmMinReprojection;

/* sfm_loss_snippets with minimum reprojection (and auto-masking) over the sources.  desc->flags must contain
 * SFM_FLAG_MIN_REPROJECTION (else SFM_E_INVALID_DESC; the workspace is sized with it), mr must not be NULL and
 * desc->ssim_rate must lie in [0, 1] (else SFM_E_INVALID_DESC: the selection needs a non-negative error).  grads == NULL:
 * forward only (the losses and the selection, the validation use).  Composes with snippet terms (their weights apply to
 * the loss, not to the selection), the peer sum (the selection stays per rank), raw disparity / pose, edge-aware
 * smoothness, SFM_FLAG_TABLES_PROVIDED, SFM_FLAG_REUSE_PYRAMID and sfm_intrinsics_grad afterwards.  The explainability
 * branch (exp_reg != 0) returns SFM_E_UNSUPPORTED: auto-masking replaces it, and sigma(l) would enter the selection.
 * Image gradients and caller per-pixel weights (SfmPixelTerms) have no argument here, as per-pixel terms exclude image
 * gradients in sfm_loss_weighted. */
int sfm_loss_min_reprojection(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms,
                              const SfmMinReprojection* mr, float* losses_out, const SfmGrads* grads, void* workspace,
                              SfmPeer* peer, void* stream);

/* Full-resolution multi-scale (SFM_FLAG_FULL_RES_MULTISCALE; Monodepth2, Godard et al., ICCV 2019, §3).  Low-resolution
 * photometric terms produce holes and texture-copy artefacts, so every coarse disparity is upsampled to the input size
 * and its photometric terms are computed there.  With the flag, for every scale s < n_scales:
 *   upsampling     U_s(d) = d_s upsampled to (H, W) with the fp32 arithmetic of torch's
 *                  F.interpolate(d, size=(H, W), mode='bilinear', align_corners=False): scale = (float)h_s / H,
 *                  src = max((Y + 0.5f) * scale - 0.5f, 0), y0 = (int)src, y1 = y0 + (y0 < h_s - 1), l1 = src - y0,
 *                  l0 = 1 - l1, the same for x, value ly0 * (lx0 * d[y0,x0] + lx1 * d[y0,x1]) + ly1 * (lx0 * d[y1,x0] +
 *                  lx1 * d[y1,x1]).  scale is h_s / H, not 2^-s (they differ when H is not a multiple of 2^s).  Scale 0 is
 *                  the identity and is never copied.
 *   photometric    the terms of scale s are those of scale 0 with disps[0] replaced by U_s(d_s): warped with
 *                  K_0 = intrinsics[:, 0] and the caller's tgt / src, over H x W pixels, means over B_global*3*H*W, the
 *                  same mask, SSIM windows and x2 out-of-view rule.
 *   smoothness     (second-order, or edge-aware with the target pyramid level) stays on d_s at its native resolution
 *                  with its smooth_reg / 2^s weight, unchanged.
 *   loss           the scales are summed as the reference does; Monodepth2's 1 / num_scales is a constant the caller
 *                  applies.
 *   gradients      those of this total: gdisps[s] = U_s^T(d total / d U_s(d_s)) + the smoothness gradient, at
 *                  (B,1,h_s,w_s); gposes through K_0 at every scale.  The adjoint is a gather without atomics, so gdisps
 *                  are bitwise reproducible from run to run.
 *   raw disparity  with bit s >= 1 of raw_disp_scales the activation is applied at native resolution before the
 *                  upsampling (Monodepth2's order) and gdisps[s] is multiplied by its derivative at the native pixel.
 *                  Bit 0 is unchanged.
 *   shapes         every per-scale map of the photometric terms grows to H x W: SfmPixelTerms weights and maps (B,S,H,W),
 *                  the selections of sfm_loss_min_reprojection (B,H,W), the debug dumps (B,S,3,H,W) / (B,S,H,W), and the
 *                  min-reprojection workspace planes.
 *   intrinsics     keeps its (B,n_scales,3,3) shape; only [:, 0] is read by the photometric terms.  With
 *                  SFM_FLAG_TABLES_PROVIDED the caller's proj / kinv must be those of K_0 at every scale.
 *                  sfm_intrinsics_grad after such a step returns the sum over the scales at [:, 0] and zeros at [:, 1:].
 * Supported: sfm_loss_forward (with debug dumps), _backward, _forward_backward, _peer, sfm_loss_snippets,
 * sfm_loss_weighted, sfm_loss_min_reprojection (with automask, the Monodepth2 configuration), SFM_FLAG_REUSE_PYRAMID,
 * SFM_FLAG_TABLES_PROVIDED, edge-aware smoothness, raw pose and CUDA-graph capture.  SFM_E_UNSUPPORTED: exp_reg != 0 (the
 * logits live at scale resolution, and auto-masking replaces the branch), image gradients
 * (sfm_loss_forward_backward_images, igrads) and sfm_host_ctx_create.  n_scales == 1 with the flag is the step without it.
 * The workspace holds B*H*W floats per scale >= 1 for the upsampled disparity and as many for its gradient, and a copy
 * of K_0 per scale.
 *
 * sfm_upsample_disparity: the upsampling U on its own (the device code the step uses), x (N,1,h,w) -> y (N,1,H,W),
 * for tests and callers that want the upsampled maps. */
int sfm_upsample_disparity(int N, int h, int w, int H, int W, const float* x, float* y, void* stream);

/* Mean-normalised smoothness (SFM_FLAG_MEAN_NORM_SMOOTH; Monodepth2, Godard et al., ICCV 2019, after Wang et al., CVPR
 * 2018).  Without it the smoothness term rewards shrinking the disparity; dividing by the mean removes that degenerate
 * solution.  With the flag, for every snippet b and scale s < n_scales:
 *   mean           m_bs = mean of the activated disparity d_s of snippet b over its native h_s x w_s plane (the raw bits of
 *                  raw_disp_scales are activated first; under SFM_FLAG_FULL_RES_MULTISCALE the native plane, not the
 *                  upsampled one, as Monodepth2 does), accumulated in a fixed order.
 *   smoothness     the term of either kind (second-order, or edge-aware with either edge weight) is evaluated on
 *                  d_s / (m_bs + 1e-7), with its smooth_reg / 2^s and 1 / B_global factors unchanged.  Every such term is
 *                  positively homogeneous of degree 1 in d, so with r_bs = 1 / (m_bs + 1e-7) and L_bs the unnormalised term
 *                  the loss is r_bs * L_bs and its disparity gradient r_bs * dL_bs/dd_j - r_bs^2 * L_bs / (h_s * w_s), times
 *                  d disp / d x at the pixel for a raw bit, times gy and the snippet weight.
 *   photometric    untouched.
 * Composes with every entry point of the fused step (sfm_loss_forward, _backward, _forward_backward, _peer,
 * sfm_loss_snippets, sfm_loss_weighted, sfm_loss_min_reprojection with or without SFM_FLAG_FULL_RES_MULTISCALE,
 * sfm_intrinsics_grad afterwards, CUDA-graph capture) and, with second-order smoothness, sfm_loss_forward_backward_images.
 * The means are per snippet, so snippet sharding needs no communication.  No float atomics feed the result: gdisps stay
 * bitwise reproducible from run to run.  smooth_reg == 0 with the flag is the step without it.  sfm_host_ctx_create
 * returns SFM_E_UNSUPPORTED with this flag or SFM_FLAG_EDGE_MEAN_ABS.
 * Workspace: with the flag it also holds B*n_scales*32 floats of disparity partials, as many of edge-aware loss partials,
 * B floats of per-snippet smoothness losses and (unless SFM_FLAG_SNIPPET_TERMS already holds it) the per-task loss array
 * of the second-order term; each array 256-byte aligned.  Without the flag the workspace is unchanged.
 *
 * Edge weight (SFM_FLAG_EDGE_MEAN_ABS, needs SFM_FLAG_EDGE_AWARE_SMOOTH): exp(-((|D0| + |D1|) + |D2|) / 3) with D_c the
 * neighbour difference of channel c of the target image, Monodepth2's form, instead of exp(-|((D0 + D1) + D2) / 3|).  The
 * two differ where the channel differences have opposite signs.  The weight depends on the image range: Monodepth2's
 * images are in [0, 1], the reference's in [-1, 1]. */

/* Border padding (SFM_FLAG_BORDER_PADDING; Monodepth2, Godard et al., ICCV 2019: F.grid_sample(..., padding_mode="border")
 * with the align-corners mapping, and the SSIM module's ReflectionPad2d(1) + AvgPool2d(3, 1)).  The reference zero-pads
 * and masks pixels that leave the view; Monodepth2 scores them against the clamped border.  With the flag:
 *   coordinates    the projection chain is unchanged up to xn, yn (the same 1e-10 and individually rounded fp32
 *                  operations); the x2 rule is skipped.  u = clamp(((xn+1)*(w-1))/2, 0, w-1), v likewise.
 *   sampling       bilinear with taps u0 = min(floor(u), w-2), weight u - u0 on u0+1, the same for v: every tap is inside
 *                  the image (at u = w-1 the value is 1 * I[w-1] + 0 * I[w-2]).
 *   gradient       d u / d xn = (w-1)/2 for 0 < ((xn+1)*(w-1))/2 < w-1 strictly, 0 otherwise (torch's
 *                  clip_coordinates_set_grad, equality at either end included); v likewise.
 *   mask           no all-zero mask.  Only a pixel whose projection is degenerate -- |z| outside [2^-58, 2^126], or a
 *                  non-finite xn or yn -- is masked: value 0, gradient 0, pix_map_masked in the per-pixel maps and no
 *                  candidate of the minimum reprojection.
 *   SSIM           the 3x3 windows of the warped image and of the target use reflection padding by one pixel (row /
 *                  column -1 is 1, h / w is h-2 / w-2), still divided by 9; the backward is the adjoint of that padding.
 *                  The identity error of sfm_loss_min_reprojection uses the same windows.
 *   unchanged      means and denominators, the smoothness term (either kind, any normalisation), the loss rows, the
 *                  intrinsics gradient and the peer sum.
 * Supported: sfm_loss_forward (without debug dumps), _backward, _forward_backward, _peer, sfm_loss_snippets,
 * sfm_loss_weighted, sfm_loss_min_reprojection, SFM_FLAG_FULL_RES_MULTISCALE, mean-normalised and edge-aware smoothness,
 * raw disparity and pose, SFM_FLAG_REUSE_PYRAMID, SFM_FLAG_TABLES_PROVIDED, sfm_intrinsics_grad afterwards and CUDA-graph
 * capture.  SFM_E_UNSUPPORTED: exp_reg != 0, image gradients, debug dumps and sfm_host_ctx_create. */

/* Axis-angle pose (SFM_FLAG_AXISANGLE_POSE; Monodepth2, Godard et al., ICCV 2019: layers.py rot_from_axisangle,
 * get_translation_matrix and transformation_from_parameters, followed literally).  Monodepth2's PoseDecoder emits
 * 0.01 * mean over its output map, which is what raw_pose_hw applies, so its raw `poseout` map composes unchanged.
 * For a pose row (v, t):
 *   rotation       theta = |v|_2, a = v / (theta + 1e-7), c = cos theta, s = sin theta, C = 1 - c,
 *                  R = C a a^T + s [a]_x + c I, entry by entry as rot_from_axisangle; no angle clipping.  For theta below
 *                  ~1e-7 R is not exactly orthonormal, as in Monodepth2.
 *   transform      T = [R | t], or with bit 16 + i of flags (SFM_FLAG_POSE_INVERT(i)) for source i, T = [R^T | -R^T t]
 *                  (Monodepth2 runs the pose network on the swapped pair for a source that precedes the target and
 *                  inverts the result: frame ids [0, -1, 1] with sources [-1, +1] give the mask 0b01).
 *   evaluation     theta, a, sin / cos, R and -R^T t in fp64, each operation individually rounded; R and t rounded to
 *                  fp32 once; P_s = K4_s . T as for the Euler pose (the same fp32 order and non-finite guard).
 *   gradient       gposes is the derivative of this formula in fp64, with torch's convention d theta / d v = 0 at
 *                  theta = 0.  With SFM_FLAG_TABLES_PROVIDED gposes goes through this chain, as it goes through the
 *                  Euler chain without the flag.  sfm_intrinsics_grad uses the R and t of the transform (fp32-rounded,
 *                  inverted where the mask says so).
 * An invert bit without SFM_FLAG_AXISANGLE_POSE, or for a source >= S, is SFM_E_INVALID_DESC.  The flag works with every
 * fused entry point, sfm_build_tables, sfm_intrinsics_grad, raw pose maps and CUDA-graph capture; sfm_host_ctx_create
 * returns SFM_E_UNSUPPORTED.  The stage warp (sfm_warp_forward / sfm_warp_backward) has no descriptor and stays Euler. */

/* Geometry consistency (SC-SfMLearner: Bian et al., "Unsupervised Scale-consistent Depth and Ego-motion Learning from
 * Monocular Video", NeurIPS 2019), sfm_loss_geometry.  Without it the depth and pose of SfM-Learner drift in scale from
 * snippet to snippet; the term ties the depth of the target to the predicted depth of every source frame.  Per scale s,
 * snippet b, target pixel p and source i:
 *   projection     the step's own: the same fp32 operations as the photometric term, so the taps, the strict in-view
 *                  flag inb (transform.py:128-131) and the bilinear weights w1..w4 are bitwise those of the warp.
 *   validity       a pair is valid iff inb.  An invalid pair contributes nothing to the geometry term and has M = 1 (its
 *                  photometric term is already masked by the x2 rule).
 *   computed depth z' = q2, the third row of P_s . [X, Y, Z, 1] before the + 1e-10 (the source-camera depth: row 2 of K is
 *                  (0, 0, 1)).  sfm_intrinsics_grad afterwards therefore stays exact.
 *   projected depth D' = ((w1 * 1/d'00 + w2 * 1/d'01) + w3 * 1/d'10) + w4 * 1/d'11, d' = src_disps[s] of (b, i), the
 *                  reciprocals as the march forms 1/disp (correctly rounded), products and sums individually rounded.
 *   depth diff     D_diff = clip(|z' - D'| / (z' + D'), 0, 1) in fp32.  Derivative with torch's conventions: sign(0) = 0,
 *                  and the clip passes the gradient on the closed interval [0, 1] and blocks it outside.  A point behind
 *                  the source camera that still projects into view (z' + D' <= 0, or z' < 0) clips and has gradient 0.
 *   geometry term  L_geo = sum_s sum_i sum_{b, p valid} D_diff / (B_global * h_s * w_s): no 2^-s and no 1/S, as the
 *                  released code sums over the sources.  The step adds geometry_reg * L_geo to the total; snippet weights
 *                  and gy apply to it as to every other term.
 *   self-mask      (self_mask != 0) the photometric terms are those of sfm_loss_weighted with M_i(p) = 1 - D_diff_i(p),
 *                  L1 and SSIM parts, with its denominators; the gradient includes the product-rule term through M.
 *   reporting      losses_out[0] (total) includes geometry_reg * L_geo; losses_out[3] REPORTS geometry_reg * L_geo: that
 *                  slot is the explainability regulariser's, which this entry point excludes, so it carries the geometry
 *                  term here (also in the rows of SfmSnippetTerms and in the peer sum).  losses_out[1] and [4] are the
 *                  (masked) L1 and SSIM parts, [2] the smoothness term.
 *   gradients      gdisps, gposes, the dL/dP cells (hence sfm_intrinsics_grad afterwards) and gsrc_disps are those of
 *                  this total.  gdisps are bitwise reproducible from run to run; gsrc_disps are accumulated with fp32
 *                  atomics after the step zeroes them, and their last bits vary with the order, as gsrc's do.
 * Computed as prologue -> (smoothness kernels) -> geometry forward (D_diff, M, the loss) -> the march (per-pixel instances
 * with the M planes under the self-mask, the plain ones without it) -> geometry backward -> epilogue; graph-capturable. */
typedef struct SfmGeometry {
  const float* src_disps[SFM_MAX_SCALES];  /* (B,S,h_s,w_s) device, activated disparity of every source frame */
  float* gsrc_disps[SFM_MAX_SCALES];       /* (B,S,h_s,w_s) device: d total / d src_disps (overwritten), or NULL */
  float* diff_maps[SFM_MAX_SCALES];        /* (B,S,h_s,w_s) device: D_diff (0 for invalid pairs), or NULL */
  float geometry_reg;                      /* SC-SfMLearner's w3 (0.5 in its released setting) */
  int32_t self_mask;                       /* != 0: the photometric terms are weighted by M = 1 - D_diff */
} SfmGeometry;

/* sfm_loss_snippets with the geometry consistency term and, optionally, the self-discovered mask.  desc->flags must
 * contain SFM_FLAG_GEOMETRY_CONSISTENCY (else SFM_E_INVALID_DESC; the workspace is sized with it), geo must not be NULL
 * and geo->src_disps[s] must be set for every s < n_scales (else SFM_E_NULL_POINTER).  grads == NULL: forward only (the
 * losses and diff_maps; gsrc_disps is then not written).  Composes with snippet terms, the peer sum (diff_maps stay per
 * rank), raw target disparity (raw_disp_scales) and raw pose, the axis-angle pose with its invert bits, either smoothness
 * with SFM_FLAG_MEAN_NORM_SMOOTH / SFM_FLAG_EDGE_MEAN_ABS, SFM_FLAG_TABLES_PROVIDED, SFM_FLAG_REUSE_PYRAMID,
 * sfm_intrinsics_grad afterwards and CUDA-graph capture.  src_disps are activated disparities (raw source maps are not
 * supported).  SFM_E_UNSUPPORTED: exp_reg != 0 (the self-mask replaces the explainability branch and its slot carries the
 * geometry term), SFM_FLAG_FULL_RES_MULTISCALE, SFM_FLAG_BORDER_PADDING or SFM_FLAG_MIN_REPROJECTION in the same call;
 * sfm_host_ctx_create with the flag.  Image gradients and debug dumps have no argument here.
 * SC-SfMLearner applies the pair loss in both directions; the reverse direction is a second call on a batch of B*S
 * snippets with S = 1 (target = source frame i, source = the target frame, disparities swapped, the inverse pose: with
 * SFM_FLAG_AXISANGLE_POSE the same rows with the invert bit flipped), which also supplies the smoothness of the sources
 * (INTEGRATION.md §6). */
int sfm_loss_geometry(const SfmDesc* desc, const SfmInputs* in, const SfmSnippetTerms* terms, const SfmGeometry* geo,
                      float* losses_out, const SfmGrads* grads, void* workspace, SfmPeer* peer, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SFMLOSS_H_ */
