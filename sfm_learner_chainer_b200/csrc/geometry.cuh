// geometry.cuh -- the two kernels of sfm_loss_geometry (include/sfmloss.h): SC-SfMLearner's geometry consistency term and
// self-discovered mask.  Included by fused_loss.cu after min_reprojection.cuh (shares Geo, pair_project, sfm_blend,
// rcp_newton and the fp64 dL/dP cells).
//
// The step is  prologue -> (smoothness kernels) -> geometry forward -> march -> geometry backward -> epilogue.
//   forward   one thread per (pixel, source): projects the target pixel exactly as the march does (pair_project on the
//             same X, Y, Z), so the in-view flag, the taps and the bilinear weights are bitwise the warp's; blends 1/d' of
//             the source disparity at the four taps into D', writes D_diff (diff_maps), M = 1 - D_diff (the march's
//             pix_w under the self-mask; 1 for an invalid pair) and adds geometry_reg * inv_n1 * sum D_diff into the
//             explainability cell of the batch or of the snippet (the slot this entry point reports the term in).
//   march     unchanged kernels: the per-pixel instances with pix_w = M and pix_map = the map planes under the self-mask,
//             the plain instances without it.
//   backward  one thread per target pixel, the sources in a fixed order: the upstream of D_diff is
//             gy w_b geometry_reg inv_n1 - map (the map, d total / d M, already holds gy w_b; only under the self-mask),
//             chained through z' = q2 and D' into the target's gdisp (read-modify-write, one store per pixel: bitwise
//             reproducible), the 12 dL/dP cells of (snippet, source, scale) (the march's layout, so the epilogue's pose
//             chain and sfm_intrinsics_grad see the whole gradient) and gsrc_disps (fp32 atomics).
// PDL: the epilogue reads the smoothness partials ahead of its own cudaGridDependencySynchronize(), relying on "launched
// => the kernel before it passed its dependency wait" holding transitively back to the prologue.  Both kernels therefore
// call cudaGridDependencySynchronize() before cudaTriggerProgrammaticLaunchCompletion().
#pragma once

namespace {

constexpr int kGeoThreads = 256;
constexpr int kGeoWarps = kGeoThreads / 32;

__device__ __forceinline__ int geo_scale(const int* begin, int ns) {
  int s = 0;
#pragma unroll
  for (int q = 1; q < SFM_MAX_SCALES; ++q)
    if (q < ns && (int)blockIdx.x >= begin[q]) s = q;
  return s;
}

// Camera point of target pixel pix of (b, s) as the march computes it: depth = 1/disp (the activation applied for a raw
// bit), ray = Kinv.(x, y, 1) individually rounded.  dsc = d(-depth)/d(disp input) / depth, as the march's.
__device__ __forceinline__ void geo_camera(const SfmFusedParams& p, int s, int b, int pix, int w, float& X, float& Y,
                                           float& Z, float& dsc) {
  const int plane = p.h[s] * w;
  float d = __ldg(p.disp[s] + (size_t)b * plane + pix), dact = 1.f;
  const bool raw = (p.raw_disp_mask >> s) & 1u;
  if (raw) d = sfm_disp_act(d, dact);
  const float depth = rcp_newton(d);
  dsc = raw ? depth * dact : depth;
  const int y = pix / w;
  const float yf = (float)y, xf = (float)(pix - y * w);
  const float* k = p.kinv + ((size_t)b * p.ns + s) * 9;
  const float rx = __fadd_rn(__fadd_rn(__fmul_rn(__ldg(k + 0), xf), __fmul_rn(__ldg(k + 1), yf)), __ldg(k + 2));
  const float ry = __fadd_rn(__fadd_rn(__fmul_rn(__ldg(k + 3), xf), __fmul_rn(__ldg(k + 4), yf)), __ldg(k + 5));
  const float rz = __fadd_rn(__fadd_rn(__fmul_rn(__ldg(k + 6), xf), __fmul_rn(__ldg(k + 7), yf)), __ldg(k + 8));
  X = __fmul_rn(depth, rx);
  Y = __fmul_rn(depth, ry);
  Z = __fmul_rn(depth, rz);
}

// The geometry record of one in-view (pixel, source): the weights and reciprocal taps of D', and the clipped ratio
struct GeoRec {
  float w1, w2, w3, w4;
  float i00, i01, i10, i11;   // 1/d' at the taps
  float a, rc, ratio;         // z' - D', 1/(z' + D'), |a| / (z' + D') unclipped
};

__device__ __forceinline__ void geo_eval(const float* __restrict__ sd, const Geo& g, const PairFwd& f, GeoRec& r) {
  r.w1 = __fmul_rn(f.wa, f.wc); r.w2 = __fmul_rn(f.wb, f.wc);
  r.w3 = __fmul_rn(f.wa, f.wd); r.w4 = __fmul_rn(f.wb, f.wd);
  const float* q = sd + f.idx;
  r.i00 = rcp_newton(__ldg(q));
  r.i01 = rcp_newton(__ldg(q + 1));
  r.i10 = rcp_newton(__ldg(q + g.w));
  r.i11 = rcp_newton(__ldg(q + g.w + 1));
  const float Dp = sfm_blend(r.w1, r.w2, r.w3, r.w4, r.i00, r.i01, r.i10, r.i11);
  r.a = __fsub_rn(f.q2, Dp);
  const float c = __fadd_rn(f.q2, Dp);
  r.ratio = __fdiv_rn(fabsf(r.a), c);
  r.rc = __fdiv_rn(1.f, c);
}

// Loads the 3x4 projection of (b, i, s)
__device__ __forceinline__ void geo_proj(const SfmFusedParams& p, int b, int i, int s, float* P) {
  const float* q = p.proj + (((size_t)b * p.S + i) * p.ns + s) * 12;
#pragma unroll
  for (int k = 0; k < 12; ++k) P[k] = __ldg(q + k);
}

__global__ void __launch_bounds__(kGeoThreads) sfm_geometry_forward_kernel(const __grid_constant__ SfmFusedParams p,
                                                                           const __grid_constant__ SfmGeoArgs a) {
  __shared__ float s_part[kGeoWarps];
  const int s = geo_scale(a.fwd_begin, p.ns);
  const int w = p.w[s], plane = p.h[s] * w, S = p.S;
  const int per = (plane + kGeoThreads - 1) / kGeoThreads;
  const int rel = (int)blockIdx.x - a.fwd_begin[s];
  const int bi = rel / per, b = bi / S, i = bi - b * S;
  const int pix = (rel - bi * per) * kGeoThreads + (int)threadIdx.x;
  const bool act = pix < plane;
  // the tables (prologue) are built and the cells reset; the march behind this kernel reads the mask planes
  cudaGridDependencySynchronize();
  cudaTriggerProgrammaticLaunchCompletion();
  float diff = 0.f;
  if (act) {
    float X, Y, Z, dsc;
    geo_camera(p, s, b, pix, w, X, Y, Z, dsc);
    float P[12];
    geo_proj(p, b, i, s, P);
    const Geo g = make_geo(p, s);
    PairFwd f;
    pair_project(P, X, Y, Z, g, f);
    if (f.inb) {
      GeoRec r;
      geo_eval(a.src_disps[s] + (size_t)bi * plane, g, f, r);
      diff = fminf(fmaxf(r.ratio, 0.f), 1.f);
    }
    const size_t o = (size_t)bi * plane + pix;
    if (a.diff_maps[s]) a.diff_maps[s][o] = diff;
    if (a.mask[s]) a.mask[s][o] = __fsub_rn(1.f, diff);
  }
  // loss partial: warp sums, then the block's warps in order, one fp64 atomic per block
  const float ws = sfm_warp_sum(diff);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = ws;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < kGeoWarps; ++k) t += s_part[k];
    if (t != 0.f) {
      const double wgt = (double)a.geometry_reg * (double)p.inv_n1[s];
      atomicAdd(p.acc + (p.snip_cell0 ? p.snip_cell0 + 4 * (size_t)b : 0) + 2, (double)t * wgt);
    }
  }
}

__global__ void __launch_bounds__(kGeoThreads) sfm_geometry_backward_kernel(const __grid_constant__ SfmFusedParams p,
                                                                            const __grid_constant__ SfmGeoArgs a) {
  __shared__ float s_red[kGeoWarps][12];
  const int s = geo_scale(a.bwd_begin, p.ns);
  const int w = p.w[s], plane = p.h[s] * w, S = p.S;
  const int per = (plane + kGeoThreads - 1) / kGeoThreads;
  const int rel = (int)blockIdx.x - a.bwd_begin[s];
  const int b = rel / per;
  const int pix = (rel - b * per) * kGeoThreads + (int)threadIdx.x;
  const bool act = pix < plane;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // the march has stored gdisp and the maps
  cudaGridDependencySynchronize();
  cudaTriggerProgrammaticLaunchCompletion();
  float gyv = p.gy ? __ldg(p.gy) : 1.f;
  if (p.snip_w) gyv *= __ldg(p.snip_w + b);
  const float wgeo = gyv * a.geometry_reg * p.inv_n1[s];
  float X = 0.f, Y = 0.f, Z = 0.f, dsc = 0.f;
  if (act) geo_camera(p, s, b, pix, w, X, Y, Z, dsc);
  const Geo g = make_geo(p, s);
  float gdd = 0.f;
  for (int i = 0; i < S; ++i) {
    const size_t bi = (size_t)b * S + i;
    float P[12];
    geo_proj(p, b, i, s, P);
    float acc[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) acc[k] = 0.f;
    if (act) {
      PairFwd f;
      pair_project(P, X, Y, Z, g, f);
      if (f.inb) {
        GeoRec r;
        geo_eval(a.src_disps[s] + bi * plane, g, f, r);
        float up = wgeo;
        if (a.map[s]) up -= __ldcg(a.map[s] + bi * plane + pix);
        // clip: the gradient passes on the closed interval [0, 1]; sign(0) = 0
        const bool pass = (r.ratio >= 0.f) && (r.ratio <= 1.f);
        const float sa = (r.a > 0.f) ? 1.f : (r.a < 0.f) ? -1.f : 0.f;
        const float gz = pass ? up * (sa - r.ratio) * r.rc : 0.f;      // d / d z'
        const float gD = pass ? up * (-sa - r.ratio) * r.rc : 0.f;     // d / d D'
        // D' through the sampler's coordinates, as the march's backward; z' = q2 directly
        const float gu = gD * (f.wc * (r.i01 - r.i00) + f.wd * (r.i11 - r.i10));
        const float gv = gD * (f.wa * (r.i10 - r.i00) + f.wb * (r.i11 - r.i01));
        const float gq0 = gu * f.r, gq1 = gv * f.r;
        const float gq2 = gz - (gq0 * f.q0 + gq1 * f.q1) * f.r;
        gdd += gq0 * (f.q0 - P[3]) + gq1 * (f.q1 - P[7]) + gq2 * (f.q2 - P[11]);
        acc[0] = gq0 * X; acc[1] = gq0 * Y; acc[2] = gq0 * Z; acc[3] = gq0;
        acc[4] = gq1 * X; acc[5] = gq1 * Y; acc[6] = gq1 * Z; acc[7] = gq1;
        acc[8] = gq2 * X; acc[9] = gq2 * Y; acc[10] = gq2 * Z; acc[11] = gq2;
        float* gs = a.gsrc_disps[s];
        if (gs && gD != 0.f) {
          float* q = gs + bi * plane + f.idx;
          atomicAdd(q, -(gD * r.w1) * r.i00 * r.i00);
          atomicAdd(q + 1, -(gD * r.w2) * r.i01 * r.i01);
          atomicAdd(q + w, -(gD * r.w3) * r.i10 * r.i10);
          atomicAdd(q + w + 1, -(gD * r.w4) * r.i11 * r.i11);
        }
      }
    }
    // dL/dP of (b, i, s): warp reduce-scatter, then the block's warps in order, one fp64 atomic per entry and block
    float v[16];
#pragma unroll
    for (int k = 0; k < 12; ++k) v[k] = acc[k];
    v[12] = v[13] = v[14] = v[15] = 0.f;
    const float tot = reduce_scatter16(v, lane);
    if ((lane & 1) == 0 && (lane >> 1) < 12) s_red[warp][lane >> 1] = tot;
    __syncthreads();
    if (threadIdx.x < 12) {
      float t = 0.f;
#pragma unroll
      for (int k = 0; k < kGeoWarps; ++k) t += s_red[k][threadIdx.x];
      if (t != 0.f) atomicAdd(p.acc + 4 + (bi * p.ns + s) * 12 + threadIdx.x, (double)t);
    }
    __syncthreads();
  }
  if (act && p.gdisp[s]) {
    float* gp = p.gdisp[s] + (size_t)b * plane + pix;
    *gp = *gp - gdd * dsc;
  }
}

}  // namespace
