// smooth.cu -- second-order disparity smoothness (compute_smooth_loss, base_model.py:169-185), forward
// and backward, for all snippets and scales in one launch.
//
//   dx = D[:, 1:] - D[:, :-1] ; dy = D[1:, :] - D[:-1, :]
//   loss_s = smooth_reg/2^s * ( mean|dx2| + mean|dxdy| + mean|dydx| + mean|dy2| )        (:181-185, :76)
//
// The term depends on the disparity alone, so it runs ahead of the fused photometric kernel -- as warp tasks
// inside the prologue kernel (smooth_task.cuh, prep.cu): it writes gdisp completely (every pixel, zero where no
// term touches it) and the fused kernel then accumulates the photometric gradient on top.
//
// Marching formulation (same shape as the SSIM kernel): a warp owns a strip of 28 interior columns (+2
// halo columns per side) x hseg rows and streams the disparity rows y0-2 .. y1+1 through registers, lane =
// column.  Horizontal neighbours come from warp shuffles (6 per row), vertical ones from short register
// rings.  With S2x, S2y, M the signed weights of the second differences (0 where the difference does not
// exist) the gradient is the gather
//   G(y,x) = [S2x(y,x-2) - 2 S2x(y,x-1) + S2x(y,x)] + [S2y(y-2,x) - 2 S2y(y-1,x) + S2y(y,x)]
//          + [M(y,x) - M(y,x-1)] - [M(y-1,x) - M(y-1,x-1)]
// so there is no scatter and no atomic on gdisp.
#include "smooth_task.cuh"

namespace {

// Edge-aware first-order smoothness, compute_disp_smooth (base_model.py:144-155; the alternative the reference
// keeps commented out at its call site, :78-80; SfmDesc flag SFM_FLAG_EDGE_AWARE_SMOOTH):
//   loss_s = smooth_reg/2^s * ( mean(|d_dx| * exp(-|mean_c i_dx|)) + mean(|d_dy| * exp(-|mean_c i_dy|)) )
// with d = disparity, i = target image of the scale (the pyramid level, no gradient).  One thread per pixel in
// gather form: its right / down differences give the loss terms it owns, and together with the left / up ones
// the gradient, so there is no scatter and no atomic on gdisp.  Needs the pyramid, so unlike the second-order
// kernel above it starts after the prep kernel.
// SNIP: per-snippet terms (gradient factor gy * w_b, the loss to snippet b's smooth cell), an instance of its own.
// MEAN_ABS (SFM_FLAG_EDGE_MEAN_ABS): Monodepth2's weight exp(-mean_c |i_dx|).  SLOTS (SFM_FLAG_MEAN_NORM_SMOOTH): the CTA
// writes its loss partial to slots[blockIdx.y][blockIdx.x] instead of adding it to a cell, so that the mean
// normalisation (mean_norm.cu) reads the loss of every (snippet, scale) in a fixed order; the gradient factor is
// gy * w_b whenever snippet weights are given.
template <bool GRAD, bool SNIP, bool MEAN_ABS = false, bool SLOTS = false>
__global__ void __launch_bounds__(256) sfm_edge_smooth_kernel(const __grid_constant__ SfmFusedParams p, float* slots) {
  const int s = blockIdx.y % p.ns, b = blockIdx.y / p.ns;
  const int h = p.h[s], w = p.w[s], plane = h * w;
  const bool raw = (p.raw_disp_mask >> s) & 1u;
  const float* __restrict__ D = p.disp[s] + (size_t)b * plane;
  const float* __restrict__ T = p.tgt_pl[s] + (size_t)b * 3 * plane;      // planar (3, h, w)
  float* __restrict__ G = GRAD ? p.gdisp[s] + (size_t)b * plane : nullptr;
  const float kx = p.sm_ex[s], ky = p.sm_ey[s];
  float gyv = (GRAD && p.gy) ? __ldg(p.gy) : 1.f;
  if ((SNIP || SLOTS) && GRAD && p.snip_w) gyv *= __ldg(p.snip_w + b);
  cudaGridDependencySynchronize();          // pyramid and loss cells (prep kernel)
  auto disp_at = [&](int i, float& f) {
    const float v = __ldg(D + i);
    f = 1.f;
    return raw ? sfm_disp_act(v, f) : v;
  };
  // exp(-|mean_c (b - a)|): F.mean over the three channels = ((d0 + d1) + d2) / 3, F.absolute, F.exp
  struct Px { float x, y, z; };
  auto tex = [&](int i) { Px v; v.x = __ldg(T + i); v.y = __ldg(T + plane + i); v.z = __ldg(T + 2 * plane + i); return v; };
  // MEAN_ABS: exp(-((|b0 - a0| + |b1 - a1|) + |b2 - a2|) / 3)
  auto edge = [&](const Px& a, const Px& c) {
    if (MEAN_ABS) {
      const float m = __fdiv_rn(__fadd_rn(__fadd_rn(fabsf(__fsub_rn(c.x, a.x)), fabsf(__fsub_rn(c.y, a.y))), fabsf(__fsub_rn(c.z, a.z))), 3.f);
      return expf(-m);
    }
    const float m = __fdiv_rn(__fadd_rn(__fadd_rn(__fsub_rn(c.x, a.x), __fsub_rn(c.y, a.y)), __fsub_rn(c.z, a.z)), 3.f);
    return expf(-fabsf(m));
  };
  float loss = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < plane; i += gridDim.x * blockDim.x) {
    const int y = i / w, x = i - y * w;
    float f0, fd;
    const float d0 = disp_at(i, f0);
    const Px t0 = tex(i);
    float g = 0.f;
    if (x + 1 < w) {
      const float dd = __fsub_rn(disp_at(i + 1, fd), d0), e = edge(t0, tex(i + 1));
      loss += fabsf(dd) * e * kx;
      g -= sfm_sign_times(dd, kx) * e;
    }
    if (y + 1 < h) {
      const float dd = __fsub_rn(disp_at(i + w, fd), d0), e = edge(t0, tex(i + w));
      loss += fabsf(dd) * e * ky;
      g -= sfm_sign_times(dd, ky) * e;
    }
    if (GRAD) {
      if (x > 0) g += sfm_sign_times(__fsub_rn(d0, disp_at(i - 1, fd)), kx) * edge(tex(i - 1), t0);
      if (y > 0) g += sfm_sign_times(__fsub_rn(d0, disp_at(i - w, fd)), ky) * edge(tex(i - w), t0);
      G[i] = raw ? (gyv * g) * f0 : gyv * g;
    }
  }
  __shared__ float part[8];
  loss = sfm_warp_sum(loss);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = loss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += part[k];
    if (SLOTS) slots[(size_t)blockIdx.y * SFM_MN_SLOTS + blockIdx.x] = t;
    else if (t != 0.f) atomicAdd(p.acc + (SNIP ? p.snip_cell0 + 4 * (size_t)b + 1 : 1), (double)t);
  }
}

}  // namespace

int sfm_launch_edge_smooth(const SfmFusedParams& p, bool grad, bool mean_abs, float* slots, cudaStream_t stream) {
  const dim3 grid((unsigned)sfm_edge_smooth_ctas(p.h[0] * p.w[0]), (unsigned)(p.B * p.ns));
  auto kernel = p.snip_cell0 ? (grad ? sfm_edge_smooth_kernel<true, true> : sfm_edge_smooth_kernel<false, true>)
                             : (grad ? sfm_edge_smooth_kernel<true, false> : sfm_edge_smooth_kernel<false, false>);
  if (slots)
    kernel = mean_abs ? (grad ? sfm_edge_smooth_kernel<true, false, true, true> : sfm_edge_smooth_kernel<false, false, true, true>)
                      : (grad ? sfm_edge_smooth_kernel<true, false, false, true> : sfm_edge_smooth_kernel<false, false, false, true>);
  else if (mean_abs)
    kernel = p.snip_cell0 ? (grad ? sfm_edge_smooth_kernel<true, true, true> : sfm_edge_smooth_kernel<false, true, true>)
                          : (grad ? sfm_edge_smooth_kernel<true, false, true> : sfm_edge_smooth_kernel<false, false, true>);
  SFM_CUDA_CHECK(sfm_launch_kernel(kernel, grid, 256, stream, true, p, slots));
  return 0;
}
