// mean_norm.cu -- Monodepth2's mean-normalised smoothness (SFM_FLAG_MEAN_NORM_SMOOTH; Godard et al., ICCV 2019, after
// Wang et al., CVPR 2018): the smoothness term of snippet b at scale s is evaluated on d / (m_bs + 1e-7), m_bs the mean of
// the activated disparity over the native plane.
//
// Every smoothness term here (second-order, edge-aware with either weight) is |linear combination of d| times a weight
// independent of d, so the unnormalised loss L_bs is positively homogeneous of degree 1 in d.  With r = 1 / (m_bs + 1e-7)
// and N = h_s * w_s:
//   loss       L_bs(r d) = r L_bs(d)
//   gradient   d/dd_j [r L_bs(d)] = r G_j - r^2 L_bs / N,   G_j = dL_bs/dd_j
// so the smoothness kernels keep computing G and L on the unnormalised disparity, and the correction is uniform over
// the plane (times d disp / d x for a raw bit, gy and the snippet weight, which G already carries).
//
// Two kernels, both one CTA row per snippet: the sum kernel (behind the prologue, it reads the disparity alone) writes
// per-CTA sums of the disparity of every scale to fixed slots; the fix-up kernel (behind the smoothness writers, ahead of
// the march, which accumulates the photometric gradient on top) reduces those and the smoothness loss partials of
// (b, s) in a fixed order, stores the snippet's normalised loss and rewrites the smoothness gradient in place.  No
// atomics: the losses and gdisp are bitwise reproducible from run to run.
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int kThreads = 256;

// CTA sum in a fixed order: warp butterflies, then the warp sums in warp order (the same value on every thread)
__device__ __forceinline__ float cta_sum(float v, float* sh) {
  v = sfm_warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int k = 0; k < kThreads / 32; ++k) t += sh[k];
  return t;
}

__global__ void __launch_bounds__(kThreads) sfm_mean_norm_sum_kernel(const __grid_constant__ SfmMeanNorm p) {
  __shared__ float sh[kThreads / 32];
  const int b = blockIdx.y;
  float sums[SFM_MAX_SCALES];
#pragma unroll
  for (int s = 0; s < SFM_MAX_SCALES; ++s) {
    float v = 0.f;
    if (s < p.ns) {
      const int plane = p.h[s] * p.w[s];
      const bool raw = (p.raw_disp_mask >> s) & 1u;
      const float* __restrict__ D = p.disp[s] + (size_t)b * plane;
      for (int i = blockIdx.x * kThreads + threadIdx.x; i < plane; i += gridDim.x * kThreads) {
        const float x = __ldg(D + i);
        float f;
        v += raw ? sfm_disp_act(x, f) : x;
      }
    }
    sums[s] = cta_sum(v, sh);
  }
  // the sums overlap the prologue; the slots are written once it is done, so that completing this grid implies
  // completing the prologue for the dependent launches behind it
  cudaGridDependencySynchronize();
  if (threadIdx.x == 0)
#pragma unroll
    for (int s = 0; s < SFM_MAX_SCALES; ++s)
      if (s < p.ns) p.mean_part[((size_t)b * p.ns + s) * SFM_MN_SLOTS + blockIdx.x] = sums[s];
}

template <bool GRAD>
__global__ void __launch_bounds__(kThreads) sfm_mean_norm_fix_kernel(const __grid_constant__ SfmMeanNorm p) {
  __shared__ double s_r[SFM_MAX_SCALES], s_l[SFM_MAX_SCALES];
  const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float gyv = (GRAD && p.gy) ? __ldg(p.gy) : 1.f;
  if (GRAD && p.snip_w) gyv *= __ldg(p.snip_w + b);
  cudaGridDependencySynchronize();          // disparity sums, smoothness gradient and loss partials
  // warp s: m_bs and L_bs, lane L adding the slots L, L + 32, ... and a fixed butterfly combining the lanes, so every
  // CTA of the snippet forms bitwise the same values
  if (warp < p.ns) {
    const int s = warp;
    double m = 0.0, l = 0.0;
    const float* mp = p.mean_part + ((size_t)b * p.ns + s) * SFM_MN_SLOTS;
    for (int k = lane; k < p.chunks; k += 32) m += (double)__ldcg(mp + k);
    const float* lp = p.loss_part + p.loss_off[s] + (size_t)b * p.loss_stride[s];
    for (int k = lane; k < p.loss_cnt[s]; k += 32) l += (double)__ldcg(lp + k);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      m += __shfl_xor_sync(0xffffffffu, m, o);
      l += __shfl_xor_sync(0xffffffffu, l, o);
    }
    if (lane == 0) {
      s_r[s] = 1.0 / (m / ((double)p.h[s] * p.w[s]) + 1e-7);
      s_l[s] = l;
    }
  }
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double t = 0.0;
    for (int s = 0; s < p.ns; ++s) t += s_r[s] * s_l[s];
    if (p.snip_cell) p.snip_cell[4 * (size_t)b] = t;
    else p.snip_loss[b] = (float)t;
  }
  if constexpr (GRAD) {
#pragma unroll 1
    for (int s = 0; s < p.ns; ++s) {
      const int plane = p.h[s] * p.w[s];
      const float r = (float)s_r[s];
      const float c = (float)((double)gyv * s_r[s] * s_r[s] * s_l[s] / plane);
      const bool raw = (p.raw_disp_mask >> s) & 1u;
      const float* __restrict__ D = p.disp[s] + (size_t)b * plane;
      float* __restrict__ G = p.gdisp[s] + (size_t)b * plane;
      for (int i = blockIdx.x * kThreads + threadIdx.x; i < plane; i += gridDim.x * kThreads) {
        float f = 1.f;
        if (raw) sfm_disp_act(__ldg(D + i), f);
        G[i] = r * G[i] - c * f;
      }
    }
  }
}

}  // namespace

int sfm_launch_mean_norm_sum(const SfmMeanNorm& m, cudaStream_t stream) {
  SFM_CUDA_CHECK(sfm_launch_kernel(sfm_mean_norm_sum_kernel, dim3((unsigned)m.chunks, (unsigned)m.B), kThreads, stream, true, m));
  return 0;
}

int sfm_launch_mean_norm_fix(const SfmMeanNorm& m, bool grad, cudaStream_t stream) {
  // forward only: one CTA per snippet forms the loss
  SFM_CUDA_CHECK(sfm_launch_kernel(grad ? sfm_mean_norm_fix_kernel<true> : sfm_mean_norm_fix_kernel<false>,
                                   dim3(grad ? (unsigned)m.chunks : 1u, (unsigned)m.B), kThreads, stream, true, m));
  return 0;
}
