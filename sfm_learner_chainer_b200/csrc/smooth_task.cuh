// smooth_task.cuh -- one warp task of the second-order disparity smoothness term (compute_smooth_loss,
// base_model.py:169-185; see smooth.cu for the formulation).  The tasks run inside the prologue kernel
// (prep.cu) next to the pyramid CTAs: the term depends on the caller's disparity alone, the pyramid CTAs are
// memory-bound and these tasks issue-bound, so one grid holding both overlaps them completely.
#pragma once
#include "common.cuh"
#include "kernels.h"

namespace {

constexpr int SM_IW = SFM_SMOOTH_IW;         // interior columns per strip

// -> this lane's part of the task's loss (to be summed over the warp by the caller)
template <bool GRAD>
__device__ __forceinline__ float sfm_smooth_task(const SfmSmoothParams& p, int t, const int lane) {
  // ---- task decode (uniform): strips x row segments of every (snippet, scale)
  int s = 0;
#pragma unroll
  for (int q = 1; q < SFM_MAX_SCALES; ++q)
    if (q < p.ns && t >= p.tile_begin[q]) s = q;
  t -= p.tile_begin[s];
  const int h = p.h[s], w = p.w[s];
  const int seg = t % p.tiles_y[s];
  t /= p.tiles_y[s];
  const int strip = t % p.tiles_x[s];
  const int b = t / p.tiles_x[s];
  const int y0 = seg * p.hseg, y1 = min(y0 + p.hseg, h);
  const int xx = strip * SM_IW - 2 + lane;
  const bool col_in = (xx >= 0) && (xx < w);
  const bool col_own = (lane >= 2) && (lane < 2 + SM_IW) && (xx < w);
  const float* __restrict__ D = p.disp[s] + (size_t)b * h * w;
  float* __restrict__ G = GRAD ? p.gdisp[s] + (size_t)b * h * w : nullptr;
  const float k_dx2 = p.k_dx2[s], k_mix = p.k_mix[s], k_dy2 = p.k_dy2[s];
  const float gyv = (GRAD && p.gy) ? __ldg(p.gy) : 1.f;
  const bool x_dx2 = col_in && (xx <= w - 3);          // dx2(., xx) exists
  const bool x_mix = col_in && (xx <= w - 2);          // cell (., xx) exists
  float loss = 0.f;
  // rings (row index relative to the row r being loaded)
  float d1 = 0.f;                   // D[r-1]
  float ex1 = 0.f;                  // ex[r-1]
  float ey2 = 0.f;                  // ey[r-2] = D[r-1] - D[r-2]
  float sy3 = 0.f, sy4 = 0.f;       // S2y[r-3], S2y[r-4]
  float n2 = 0.f, n3 = 0.f;         // N[r-2], N[r-3],  N[y] = M(y,x) - M(y,x-1)
  float gx1 = 0.f, gx2 = 0.f;       // Gx[r-1], Gx[r-2]
  // producer-side fusion (SfmDesc.raw_disp_scales): D holds the pre-activation map, the disparity is formed on
  // load and the gradient is written w.r.t. the raw map (factor ring f0..f2 = d disp / d x of rows r..r-2)
  const bool raw = (p.raw_disp_mask >> s) & 1u;
  float f_next = 1.f, f1 = 1.f, f2 = 1.f;
  auto load = [&](int r, float& f) {
    f = 1.f;
    if (!(col_in && r >= 0 && r < h)) return 0.f;
    const float v = __ldg(D + (size_t)r * w + xx);
    return raw ? sfm_disp_act(v, f) : v;
  };
  float d_next = load(y0 - 2, f_next);
#pragma unroll 1
  for (int r = y0 - 2; r < y1 + 2; ++r) {
    const float d0 = d_next, f0 = f_next;
    d_next = load(r + 1, f_next);
    const bool r_in = (r >= 0) && (r < h);
    // ---- horizontal terms of row r
    const float ex0 = __fsub_rn(__shfl_down_sync(0xffffffffu, d0, 1), d0);                 // D[r][x+1] - D[r][x]
    const float dx2 = __fsub_rn(__shfl_down_sync(0xffffffffu, ex0, 1), ex0);
    const bool vx = r_in && x_dx2;
    const float sx = vx ? sfm_sign_times(dx2, k_dx2) : 0.f;
    if (vx && col_own && r >= y0 && r < y1) loss += fabsf(dx2) * k_dx2;
    const float sxm1 = __shfl_up_sync(0xffffffffu, sx, 1), sxm2 = __shfl_up_sync(0xffffffffu, sx, 2);
    const float gx0 = (sxm2 - 2.f * sxm1) + sx;
    // ---- vertical terms: dy2 at row r-2
    const float ey1 = __fsub_rn(d0, d1);                                                    // D[r] - D[r-1]
    const float dy2 = __fsub_rn(ey1, ey2);
    const int ry = r - 2;
    const bool vy = col_in && (ry >= 0) && (ry <= h - 3);
    const float sy2 = vy ? sfm_sign_times(dy2, k_dy2) : 0.f;
    if (vy && col_own && ry >= y0 && ry < y1) loss += fabsf(dy2) * k_dy2;
    // ---- mixed terms of cell (r-1, x): dxdy = ex[r] - ex[r-1] ; dydx = ey[r-1][x+1] - ey[r-1][x]
    const float a = __fsub_rn(ex0, ex1);
    const float bq = __fsub_rn(__shfl_down_sync(0xffffffffu, ey1, 1), ey1);
    const int rm = r - 1;
    const bool vm = x_mix && (rm >= 0) && (rm <= h - 2);
    const float m1 = vm ? (sfm_sign_times(a, k_mix) + sfm_sign_times(bq, k_mix)) : 0.f;
    if (vm && col_own && rm >= y0 && rm < y1) loss += (fabsf(a) + fabsf(bq)) * k_mix;
    const float n1 = m1 - __shfl_up_sync(0xffffffffu, m1, 1);
    // ---- gradient of pixel (r-2, x)
    if (GRAD) {
      const float g = (gx2 + ((sy4 - 2.f * sy3) + sy2)) + (n2 - n3);
      if (col_own && ry >= y0 && ry < y1) G[(size_t)ry * w + xx] = raw ? (gyv * g) * f2 : gyv * g;
    }
    f2 = f1; f1 = f0;
    d1 = d0; ex1 = ex0; ey2 = ey1;
    sy4 = sy3; sy3 = sy2;
    n3 = n2; n2 = n1;
    gx2 = gx1; gx1 = gx0;
  }
  return loss;
}

}  // namespace
