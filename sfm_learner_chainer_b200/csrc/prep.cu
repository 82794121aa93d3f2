// prep.cu -- per-step prologue kernel: image pyramid (F.resize_images, base_model.py:70-72), scales >= 1 only and
// planar like the caller's tensors (scale 0 is the identity and is never copied: the loss kernels read it from
// the caller's tensors), the 3x4 projection tables (proj_tgt_to_src, transform.py:64-91) and inverse intrinsics
// (F.batch_inv, transform.py:105), the reset of the fp64 reduction cells the fused loss kernel accumulates into --
// and, in the same grid, the second-order smoothness tasks (smooth_task.cuh): they depend on the caller's disparity
// alone and are issue-bound while the pyramid CTAs are memory-bound, so CTAs of both kinds are interleaved in one
// launch and share the SMs (as separate dependent launches they ran almost back to back: a dependent grid is only
// released when the last wave of its predecessor has started).
#include "common.cuh"
#include "kernels.h"
#include "smooth_task.cuh"

namespace {

constexpr int kPrepThreads = 256;
constexpr int kMaxCand = 8;       // candidate rows per (band, scale): band / step + 3 <= 8 for bands of up to 8 rows

// One row of a coarser scale owned by this band: its index, top tap row and the float64 row weights.
struct PrepRow {
  int y, v0;
  double va, vb;
};

// Pyramid CTA = (image, band of BAND full-resolution rows).  It produces every coarser-scale row whose top tap
// row v0 lies in the band, so the full-resolution planes are read from HBM once (scale 1 touches every
// full-resolution row; the coarser scales re-read them through L1/L2 while they are hot) instead of once per
// scale.  A thread owns one output COLUMN of one scale: it derives the column's float64 coordinate and weights
// once and then walks the (at most BAND/2 + 1) rows of that scale in the band, so the loads of different rows
// are independent and every warp of the CTA is busy at once; threads along x make the planar 4-byte stores fully
// coalesced.  The rows a band owns are found once per CTA (shared-memory list).
// Coordinates follow Chainer's resize_images: u = linspace(0, W-1, w_s) in float64 (x*step, last
// element pinned to W-1), u0 = clip(floor(u), 0, W-2), weights are float64 products cast to fp32,
// y = ((w1*a + w2*b) + w3*c) + w4*d in fp32.
// Block roles: [0, n_tail) tables + cell reset; then the n_pyr_blocks pyramid CTAs and the n_sm smoothness CTAs, the
// latter spread evenly over the first R = n_mix_region blocks (block i < R is a smoothness CTA when
// floor((i+1) n_sm / R) > floor(i n_sm / R)): the long, issue-bound smoothness CTAs start early and the short,
// memory-bound pyramid CTAs fill the SMs around them and run on alone at the end.
// SM: 0 = no smoothness tasks, 1 = loss only, 2 = loss and gdisp; 3 / 4 = 1 / 2 with per-task losses instead of the CTA
// partial (a CTA's tasks may belong to different snippets).  No early programmatic-launch trigger: the dependent
// fused kernel's CTAs would pile up on whichever SMs are free first (measured, see the launch policy notes in DESIGN.md).
// AA: SFM_FLAG_AXISANGLE_POSE, the tables of Monodepth2's axis-angle pose, bit i of pose_inv inverting source i's.  Its
// own instances: the inlined fp64 chain changes the register allocation of the whole kernel, so the Euler instances keep
// the parent's code (and pose_inv, the trailing argument, is not read there).
template <int SM, bool AA>
__global__ void __launch_bounds__(kPrepThreads) sfm_prep_kernel(const __grid_constant__ SfmPrepParams p,
                                                                const __grid_constant__ SfmSmoothParams sm, unsigned pose_inv) {
  int blk = blockIdx.x;
  if (blk < p.n_tail_blocks) {
    // ---- tables + accumulator reset (a handful of leading CTAs)
    const int t = blk * kPrepThreads + threadIdx.x;
    const int n_proj = p.build_tables ? p.B * p.S * p.ns : 0;
    const int n_kinv = p.build_tables ? p.B * p.ns : 0;
    if (t < n_proj) {
      const int s = t % p.ns;
      const int i = (t / p.ns) % p.S;
      const int b = t / (p.ns * p.S);
      float K[9], pose[6], P[12];
      for (int k = 0; k < 9; ++k) K[k] = p.intrinsics[((size_t)b * p.ns + s) * 9 + k];
      if (p.raw_pose_hw > 0) {
        // producer-side fusion: pose = 0.01 * mean_{h', w'}(poseout)   (pose_net.py:52-53; channel 6i+k of snippet b)
        for (int k = 0; k < 6; ++k)
          pose[k] = sfm_pose_component(p.poses + (((size_t)b * p.S + i) * 6 + k) * p.raw_pose_hw, p.raw_pose_hw);
        if (s == 0 && p.posevec_out)
          for (int k = 0; k < 6; ++k) p.posevec_out[((size_t)b * p.S + i) * 6 + k] = pose[k];
      } else {
        for (int k = 0; k < 6; ++k) pose[k] = p.poses[((size_t)b * p.S + i) * 6 + k];
      }
      if constexpr (AA)
        sfm_build_proj_axisangle(pose, (pose_inv >> i) & 1u, K, P);
      else
        sfm_build_proj(pose, K, P);
      // A non-finite pose or intrinsic would make every pixel of this (snippet, source) pair project to NaN: out of view
      // by the strict test of transform.py:128-131, but with NaN in the backward's 0 * P products.  Such a pair gets a
      // finite projection that sends every pixel out of view instead (q = (1e30, 1e30, 1)): losses and gradients of the
      // pair are exactly 0 (documented deviation: the reference propagates NaN).
      bool finite = true;
      for (int k = 0; k < 12; ++k) finite = finite && (fabsf(P[k]) <= 3.0e38f);
      if (!finite) {
        for (int k = 0; k < 12; ++k) P[k] = 0.f;
        P[3] = 1e30f; P[7] = 1e30f; P[11] = 1.f;
      }
      for (int k = 0; k < 12; ++k) p.proj_out[(size_t)t * 12 + k] = P[k];
    } else if (t < n_proj + n_kinv) {
      const int j = t - n_proj;
      float K[9], inv[9];
      for (int k = 0; k < 9; ++k) K[k] = p.intrinsics[(size_t)j * 9 + k];
      sfm_inv3(K, inv);
      for (int k = 0; k < 9; ++k) p.kinv_out[(size_t)j * 9 + k] = inv[k];
    } else {
      const int j = t - n_proj - n_kinv;
      if (j < p.n_acc) p.acc[j] = 0.0;
    }
    return;
  }

  blk -= p.n_tail_blocks;
  if (SM != 0) {
    const long long R = p.n_mix_region;
    const int k0 = (blk < R) ? (int)(((long long)blk * sm.n_ctas) / R) : sm.n_ctas;
    const int k1 = (blk < R) ? (int)(((long long)(blk + 1) * sm.n_ctas) / R) : sm.n_ctas;
    if (k1 > k0) {
      // ---- smoothness CTA k0: one task per warp
      __shared__ float s_part[kPrepThreads / 32];
      const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
      const int t = k0 * (kPrepThreads / 32) + warp;
      if (SM >= 3) {
        if (t < sm.n_tasks) sfm_smooth_task<SM == 4, true>(sm, t, lane);
        return;
      }
      float loss = (t < sm.n_tasks) ? sfm_smooth_task<SM == 2>(sm, t, lane) : 0.f;
      loss = sfm_warp_sum(loss);
      if (lane == 0) s_part[warp] = loss;
      __syncthreads();
      if (threadIdx.x == 0) {
        float tot = 0.f;
#pragma unroll
        for (int k = 0; k < kPrepThreads / 32; ++k) tot += s_part[k];
        sm.part[k0] = tot;
      }
      return;
    }
    blk -= k0;
  }

  // ---- pyramid
  __shared__ PrepRow s_rows[SFM_MAX_SCALES - 1][kMaxCand];
  __shared__ int s_nrows[SFM_MAX_SCALES - 1];
  const int band_rows = p.band;
  const int n_bands = (p.H + band_rows - 1) / band_rows;
  const int img = blk / n_bands;            // [0, B): target b ; [B, B + B*S): source (b, i)
  const int band = blk - img * n_bands;
  const int Y0 = band * band_rows, Y1 = min(Y0 + band_rows, p.H);
  const bool is_src = img >= p.B;
  const int H = p.H, W = p.W;
  const size_t plane = (size_t)H * W;
  const float* __restrict__ base = is_src ? p.src + (size_t)(img - p.B) * 3 * plane : p.tgt + (size_t)img * 3 * plane;
  if (threadIdx.x < SFM_MAX_SCALES - 1) s_nrows[threadIdx.x] = 0;
  __syncthreads();
  if (threadIdx.x < (p.ns - 1) * kMaxCand) {
    const int s = 1 + threadIdx.x / kMaxCand, k = threadIdx.x % kMaxCand;
    const int h = H >> s;
    const double stepy = (h > 1) ? __ddiv_rn((double)(H - 1), (double)(h - 1)) : 0.0;
    // candidate rows: those whose v0 can fall in [Y0, Y1); the exact test follows
    const int y_lo = (stepy > 0.0) ? max(0, (int)((double)Y0 / stepy) - 1) : 0;
    const int y_hi = (stepy > 0.0) ? min(h, (int)((double)Y1 / stepy) + 2) : h;
    const int y = y_lo + k;
    if (y < y_hi) {
      const double v = (y == h - 1 && h > 1) ? (double)(H - 1) : __dmul_rn((double)y, stepy);
      const int v0 = min(max((int)floor(v), 0), H - 2);
      if (v0 >= Y0 && v0 < Y1) {
        const int slot = atomicAdd(&s_nrows[s - 1], 1);
        PrepRow e;
        e.y = y; e.v0 = v0;
        e.va = __dsub_rn((double)(v0 + 1), v);
        e.vb = __dsub_rn(v, (double)v0);
        s_rows[s - 1][slot] = e;
      }
    }
  }
  __syncthreads();
  int col_end[SFM_MAX_SCALES];               // columns of the scales 1.. laid end to end
  col_end[0] = 0;
#pragma unroll
  for (int s = 1; s < SFM_MAX_SCALES; ++s) col_end[s] = col_end[s - 1] + ((s < p.ns) ? (W >> s) : 0);
  for (int c = threadIdx.x; c < col_end[SFM_MAX_SCALES - 1]; c += kPrepThreads) {
    int s = 1;
#pragma unroll
    for (int q = 1; q < SFM_MAX_SCALES - 1; ++q)
      if (c >= col_end[q]) s = q + 1;
    const int x = c - col_end[s - 1];
    const int nr = s_nrows[s - 1];
    if (nr == 0) continue;
    const int h = H >> s, w = W >> s;
    const size_t oplane = (size_t)h * w;
    float* __restrict__ out = (is_src ? p.src_pyr[s] + (size_t)(img - p.B) * 3 * oplane : p.tgt_pyr[s] + (size_t)img * 3 * oplane) + x;
    const double stepx = (w > 1) ? __ddiv_rn((double)(W - 1), (double)(w - 1)) : 0.0;
    const double u = (x == w - 1 && w > 1) ? (double)(W - 1) : __dmul_rn((double)x, stepx);
    const int u0 = min(max((int)floor(u), 0), W - 2);
    const double ua = __dsub_rn((double)(u0 + 1), u), ub = __dsub_rn(u, (double)u0);
    const float* __restrict__ col = base + u0;
    for (int r = 0; r < nr; ++r) {
      const PrepRow e = s_rows[s - 1][r];
      const float w1 = (float)__dmul_rn(ua, e.va), w2 = (float)__dmul_rn(ub, e.va);
      const float w3 = (float)__dmul_rn(ua, e.vb), w4 = (float)__dmul_rn(ub, e.vb);
      const float* __restrict__ r0 = col + (size_t)e.v0 * W;
      float* __restrict__ orow = out + (size_t)e.y * w;
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        const float* pl = r0 + ch * plane;
        orow[ch * oplane] = sfm_blend(w1, w2, w3, w4, __ldg(pl), __ldg(pl + 1), __ldg(pl + W), __ldg(pl + W + 1));
      }
    }
  }
}

__global__ void sfm_disp_activation_kernel(const float* __restrict__ x, float* __restrict__ disp, float* __restrict__ dact,
                                           long long n) {
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    float da;
    const float d = sfm_disp_act(__ldg(x + i), da);
    if (disp) disp[i] = d;
    if (dact) dact[i] = da;
  }
}

__global__ void sfm_pose_reduce_kernel(const float* __restrict__ x, float* __restrict__ out, int n_comp, int hw) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_comp) out[t] = sfm_pose_component(x + (size_t)t * hw, hw);
}

}  // namespace

template <bool AA>
int launch_prep(const SfmPrepParams& p, const SfmSmoothParams& sm, int sm_mode, unsigned grid, unsigned pose_inv,
                cudaStream_t stream) {
  const auto kernel = sm_mode == 4 ? sfm_prep_kernel<4, AA> : sm_mode == 3 ? sfm_prep_kernel<3, AA> : sm_mode == 2 ? sfm_prep_kernel<2, AA>
                    : sm_mode == 1 ? sfm_prep_kernel<1, AA> : sfm_prep_kernel<0, AA>;
  SFM_CUDA_CHECK(sfm_launch_kernel(kernel, grid, kPrepThreads, stream, false, p, sm, pose_inv));
  return 0;
}

int sfm_launch_prep(const SfmPrepParams& p_in, const SfmSmoothParams* sm_in, int sm_mode, cudaStream_t stream,
                    unsigned pose_flags) {
  SfmPrepParams p = p_in;
  const SfmSmoothParams sm = sm_in ? *sm_in : SfmSmoothParams{};
  if (sm.n_ctas <= 0) sm_mode = 0;
  p.n_pyr_blocks = (p.do_pyramid && p.ns > 1) ? p.B * (1 + p.S) * ((p.H + p.band - 1) / p.band) : 0;
  const long long n_tail = (p.build_tables ? (long long)p.B * p.S * p.ns + (long long)p.B * p.ns : 0) + p.n_acc;
  p.n_tail_blocks = (int)((n_tail + kPrepThreads - 1) / kPrepThreads);
  const unsigned grid = (unsigned)(p.n_tail_blocks + p.n_pyr_blocks + (sm_mode ? sm.n_ctas : 0));
  if (grid == 0) return 0;                        // e.g. sfm_pyramid with a single scale: nothing to build
  const unsigned inv = (pose_flags & SFM_FLAG_POSE_INVERT_MASK) >> SFM_FLAG_POSE_INVERT_SHIFT;
  return (p.build_tables && (pose_flags & SFM_FLAG_AXISANGLE_POSE)) ? launch_prep<true>(p, sm, sm_mode, grid, inv, stream)
                                                                    : launch_prep<false>(p, sm, sm_mode, grid, 0u, stream);
}

int sfm_launch_disp_activation(long long n, const float* x, float* disp, float* dact, cudaStream_t stream) {
  if (n <= 0) return 0;
  const long long blocks = (n + 255) / 256;
  sfm_disp_activation_kernel<<<(unsigned)(blocks > SFM_REF_SMS * 16 ? SFM_REF_SMS * 16 : blocks), 256, 0, stream>>>(x, disp, dact, n);
  SFM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

int sfm_launch_pose_reduce(int B, int S, int hw, const float* x, float* poses_out, cudaStream_t stream) {
  const int n = B * S * 6;
  sfm_pose_reduce_kernel<<<(n + 127) / 128, 128, 0, stream>>>(x, poses_out, n, hw);
  SFM_CUDA_CHECK(cudaGetLastError());
  return 0;
}

