// full_res.cu -- the two kernels around the fused step under SFM_FLAG_FULL_RES_MULTISCALE (include/sfmloss.h), Monodepth2's
// full-resolution multi-scale loss:
//   upsample -> prologue -> [edge-aware smoothness] -> [forward march -> select] -> march -> epilogue -> adjoint
// The march itself is unchanged: every scale s >= 1 is handed to it as a full-resolution scale (the caller's images, the
// upsampled disparity U_s(d_s) and a full-resolution gradient plane in the workspace, tables built from K_0).  The upsample
// kernel writes those planes and the K_0 copy; the adjoint kernel maps the gradient planes back to the native maps.
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int kUpThreads = 256;

// One axis of torch's upsample_bilinear2d with align_corners=False for an output of n_out points from n points, in the
// fp32 arithmetic of its CPU kernel (area_pixel_compute_scale / area_pixel_compute_source_index, no contraction):
// src = max((X + 0.5) * scale - 0.5, 0), i0 = (int)src, i1 = i0 + (i0 < n - 1), l1 = src - i0, l0 = 1 - l1.
struct UpTap {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ UpTap up_tap(int X, int n, float scale) {
  const float src = fmaxf(__fsub_rn(__fmul_rn(__fadd_rn((float)X, 0.5f), scale), 0.5f), 0.f);
  UpTap t;
  t.i0 = (int)src;
  t.i1 = t.i0 + (t.i0 < n - 1 ? 1 : 0);
  t.l1 = __fsub_rn(src, (float)t.i0);
  t.l0 = __fsub_rn(1.f, t.l1);
  return t;
}
__device__ __forceinline__ float up_scale(int n, int n_out) { return __fdiv_rn((float)n, (float)n_out); }

// U(d) at full-resolution pixel (Y, X) of one (h, w) map; RAW: d is the pre-activation map, activated at the four taps
template <bool RAW>
__device__ __forceinline__ float up_value(const float* __restrict__ d, int h, int w, int H, int W, int Y, int X) {
  const UpTap ty = up_tap(Y, h, up_scale(h, H)), tx = up_tap(X, w, up_scale(w, W));
  const float* r0 = d + (size_t)ty.i0 * w;
  const float* r1 = d + (size_t)ty.i1 * w;
  float d00 = __ldg(r0 + tx.i0), d01 = __ldg(r0 + tx.i1), d10 = __ldg(r1 + tx.i0), d11 = __ldg(r1 + tx.i1);
  if (RAW) {
    float f;
    d00 = sfm_disp_act(d00, f); d01 = sfm_disp_act(d01, f); d10 = sfm_disp_act(d10, f); d11 = sfm_disp_act(d11, f);
  }
  const float top = __fadd_rn(__fmul_rn(tx.l0, d00), __fmul_rn(tx.l1, d01));
  const float bot = __fadd_rn(__fmul_rn(tx.l0, d10), __fmul_rn(tx.l1, d11));
  return __fadd_rn(__fmul_rn(ty.l0, top), __fmul_rn(ty.l1, bot));
}

// Grid: x over the B*H*W full-resolution pixels, y = scale - 1.  Writes U_s(d_s), zeroes the gradient plane when the
// march accumulates into it, and (y == 0) copies K_0 over the scales.  Launched without PDL ahead of the prologue kernel,
// so everything after it sees its writes through plain stream order.
__global__ void __launch_bounds__(kUpThreads) sfm_full_res_upsample_kernel(const __grid_constant__ SfmFullRes f) {
  const int s = 1 + blockIdx.y;
  const long long k = (long long)blockIdx.x * kUpThreads + threadIdx.x;
  if (blockIdx.y == 0 && k < (long long)f.B * f.ns * 9) {
    const int b = (int)(k / (f.ns * 9)), e = (int)(k % 9);
    f.k0[k] = __ldg(f.intrinsics + (size_t)b * f.ns * 9 + e);
  }
  const long long plane = (long long)f.H * f.W;
  if (k >= f.B * plane) return;
  const int b = (int)(k / plane), pix = (int)(k - b * plane), Y = pix / f.W, X = pix - Y * f.W;
  const float* d = f.disp[s] + (size_t)b * f.h[s] * f.w[s];
  f.up[s][k] = ((f.raw_disp_mask >> s) & 1u) ? up_value<true>(d, f.h[s], f.w[s], f.H, f.W, Y, X)
                                             : up_value<false>(d, f.h[s], f.w[s], f.H, f.W, Y, X);
  if (f.zero_gup) f.gup[s][k] = 0.f;
}

// Taps of U along one axis that read native index i: the contiguous range of output points whose (i0, i1) contains i,
// with the weight l0 [i0 == i] + l1 [i1 == i].  `lo` is a point at or before the first of them.
__device__ __forceinline__ int up_first(int i, float scale) {
  return max(0, (int)floorf(((float)i - 0.5f) / scale - 0.5f) - 2);
}

// Adjoint U_s^T in gather form: one thread per native pixel (b, y, x) of a scale s >= 1 (block ranges blk_begin) walks
// the fine rows and columns whose taps include it in increasing order and adds g * wx per row, then wy * row sum, with
// the forward's fp32 weights.  No atomics: the result is bitwise reproducible.  Raw scales multiply by d disp / d x at the
// native pixel.  A dependent launch behind the epilogue: the march's writes are two launches back, and both the epilogue
// and this kernel wait for their predecessor before they end.
__global__ void __launch_bounds__(kUpThreads) sfm_full_res_adjoint_kernel(const __grid_constant__ SfmFullRes f,
                                                                          const SfmUpGrid g) {
  int s = 1;
#pragma unroll
  for (int q = 2; q < SFM_MAX_SCALES; ++q)
    if (q < f.ns && (int)blockIdx.x >= g.blk_begin[q]) s = q;
  const int h = f.h[s], w = f.w[s], H = f.H, W = f.W;
  const long long k = (long long)(blockIdx.x - g.blk_begin[s]) * kUpThreads + threadIdx.x;
  const long long plane = (long long)h * w;
  cudaGridDependencySynchronize();                         // the march (behind the epilogue) has written the planes
  if (k >= f.B * plane) return;
  const int b = (int)(k / plane), pix = (int)(k - b * plane), y = pix / w, x = pix - y * w;
  const float sy = up_scale(h, H), sx = up_scale(w, W);
  const float* __restrict__ G = f.gup[s] + (size_t)b * H * W;
  const int X0 = up_first(x, sx);
  float acc = 0.f;
  for (int Y = up_first(y, sy); Y < H; ++Y) {
    const UpTap ty = up_tap(Y, h, sy);
    if (ty.i0 > y) break;
    if (ty.i0 != y && ty.i1 != y) continue;
    const float wy = __fadd_rn(ty.i0 == y ? ty.l0 : 0.f, ty.i1 == y ? ty.l1 : 0.f);
    const float* __restrict__ row = G + (size_t)Y * W;
    float r = 0.f;
    for (int X = X0; X < W; ++X) {
      const UpTap tx = up_tap(X, w, sx);
      if (tx.i0 > x) break;
      if (tx.i0 != x && tx.i1 != x) continue;
      const float wx = __fadd_rn(tx.i0 == x ? tx.l0 : 0.f, tx.i1 == x ? tx.l1 : 0.f);
      r = __fmaf_rn(__ldcg(row + X), wx, r);
    }
    acc = __fmaf_rn(wy, r, acc);
  }
  const size_t o = (size_t)b * plane + pix;
  if ((f.raw_disp_mask >> s) & 1u) {
    float dact;
    sfm_disp_act(__ldg(f.disp[s] + o), dact);
    acc = acc * dact;
  }
  f.gdisp[s][o] = f.accum ? f.gdisp[s][o] + acc : acc;
}

// sfm_intrinsics_grad after a full-resolution step: every scale's contribution belongs to K_0.  One thread per (b, entry)
// adds them in scale order into [:, 0] and zeroes [:, 1:]; a dependent launch behind the intrinsics-gradient kernel.
__global__ void sfm_intrinsics_fold_kernel(int B, int ns, float* __restrict__ gK) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  cudaGridDependencySynchronize();
  if (t >= B * 9) return;
  float* q = gK + (size_t)(t / 9) * ns * 9 + t % 9;
  float v = q[0];
  for (int s = 1; s < ns; ++s) {
    v += q[s * 9];
    q[s * 9] = 0.f;
  }
  q[0] = v;
}

__global__ void __launch_bounds__(kUpThreads) sfm_upsample_stage_kernel(int N, int h, int w, int H, int W, const float* __restrict__ x,
                                                                        float* __restrict__ y) {
  const long long k = (long long)blockIdx.x * kUpThreads + threadIdx.x;
  const long long plane = (long long)H * W;
  if (k >= N * plane) return;
  const int n = (int)(k / plane), pix = (int)(k - n * plane), Y = pix / W, X = pix - Y * W;
  y[k] = up_value<false>(x + (size_t)n * h * w, h, w, H, W, Y, X);
}

}  // namespace

int sfm_launch_full_res_upsample(const SfmFullRes& f, cudaStream_t stream) {
  const long long n = (long long)f.B * f.H * f.W;
  const long long nk = (long long)f.B * f.ns * 9;
  const dim3 grid((unsigned)(((n > nk ? n : nk) + kUpThreads - 1) / kUpThreads), (unsigned)(f.ns - 1));
  SFM_CUDA_CHECK(sfm_launch_kernel(sfm_full_res_upsample_kernel, grid, kUpThreads, stream, false, f));
  return 0;
}

int sfm_launch_full_res_adjoint(const SfmFullRes& f, cudaStream_t stream) {
  SfmUpGrid g{};
  int nb = 0;
  for (int s = 0; s < SFM_MAX_SCALES; ++s) {
    g.blk_begin[s] = nb;
    if (s >= 1 && s < f.ns) nb += (int)(((long long)f.B * f.h[s] * f.w[s] + kUpThreads - 1) / kUpThreads);
  }
  g.blk_begin[SFM_MAX_SCALES] = nb;
  SFM_CUDA_CHECK(sfm_launch_kernel(sfm_full_res_adjoint_kernel, (unsigned)nb, kUpThreads, stream, true, f, g));
  return 0;
}

int sfm_launch_intrinsics_fold(int B, int ns, float* gintrinsics, cudaStream_t stream) {
  SFM_CUDA_CHECK(sfm_launch_kernel(sfm_intrinsics_fold_kernel, (unsigned)((B * 9 + 127) / 128), 128, stream, true, B, ns, gintrinsics));
  return 0;
}

int sfm_launch_upsample_stage(int N, int h, int w, int H, int W, const float* x, float* y, cudaStream_t stream) {
  const long long n = (long long)N * H * W;
  if (n == 0) return 0;
  sfm_upsample_stage_kernel<<<(unsigned)((n + kUpThreads - 1) / kUpThreads), kUpThreads, 0, stream>>>(N, h, w, H, W, x, y);
  SFM_CUDA_CHECK(cudaGetLastError());
  return 0;
}
