// min_reprojection.cuh -- select kernel of sfm_loss_min_reprojection (include/sfmloss.h): per-pixel minimum reprojection
// and auto-masking over the source views.  Included by fused_loss.cu after ssim_march.cuh (shares its packed SSIM
// arithmetic).
//
// The step is  prologue -> forward march -> select -> march -> epilogue.  The forward march is the per-pixel instance of
// the forward mode with gy = 1 and no snippet weights: it writes the map of every (pixel, source) into the workspace
// planes, which is inv_n3 * e_i(p), and p.pix_map_masked (< 0) where the source is masked.  The select kernel reads the
// S planes of a pixel, computes the identity errors as a stencil over the target and source pyramid levels in the same
// arithmetic as the march (L1, and the 3x3 SSIM on raw window sums, both scaled like the map), writes the one-hot weights
// over the planes in place and the optional selection map.  The march of sfm_loss_weighted then runs with those weights.
#pragma once

namespace {

constexpr int kSelectThreads = 256;

// Blocks of the select grid: scale s holds blocks [blk_begin[s], blk_begin[s+1]), one thread per pixel of B x h x w.
struct SfmSelectGrid {
  int blk_begin[SFM_MAX_SCALES + 1];
};

// target pixel (b, y, x) of scale s, three channels; 0 outside the image (the zero padding of the reference's SSIM pool)
__device__ __forceinline__ V3 sel_tap(const float* __restrict__ img, int plane, int h, int w, int y, int x) {
  if (y < 0 || y >= h || x < 0 || x >= w) return v3s(0.f);
  const float* q = img + y * w + x;
  return v3(__ldg(q), __ldg(q + plane), __ldg(q + 2 * plane));
}

// SSIM: the identity error includes the clipped SSIM term of the same 3x3 zero-padded windows as the march
template <bool SSIM>
__global__ void __launch_bounds__(kSelectThreads) sfm_min_reprojection_select_kernel(const __grid_constant__ SfmFusedParams p,
                                                                                     const SfmSelectGrid g, const SfmMinRepArgs a) {
  int s = 0;
#pragma unroll
  for (int q = 1; q < SFM_MAX_SCALES; ++q)
    if (q < p.ns && (int)blockIdx.x >= g.blk_begin[q]) s = q;
  const int h = p.h[s], w = p.w[s], plane = h * w, S = p.S;
  const long long k = (long long)(blockIdx.x - g.blk_begin[s]) * kSelectThreads + threadIdx.x;
  const bool act = k < (long long)p.B * plane;
  const int b = act ? (int)(k / plane) : 0, pix = act ? (int)(k - (long long)b * plane) : 0;
  const int y = pix / w, x = pix - y * w;
  // the forward march wrote the planes; the cells it accumulated into are reset below
  cudaGridDependencySynchronize();
  cudaTriggerProgrammaticLaunchCompletion();
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    // the forward march ran without snippet terms, so its partials are in the batch cells pixel, exp, ssim; the smooth
    // cell belongs to the edge-aware smoothness kernel (which ran before it) and is left alone
    p.acc[0] = 0.0;
    p.acc[2] = 0.0;
    p.acc[3] = 0.0;
  }
  if (!act) return;
  float* const planes = const_cast<float*>(p.pix_w[s]) + (size_t)b * S * plane + pix;
  float best = 0.f;
  int sel = -2;
  for (int i = 0; i < S; ++i) {
    const float e = planes[(size_t)i * plane];
    if (e >= 0.f && (sel < 0 || e < best)) { best = e; sel = i; }      // masked (< 0) is no candidate; ties: lowest index
  }
  if (a.automask && sel >= 0) {
    // identity errors, scaled like the map: wpix * L1 + wssim * sum_c clip((1 - SSIM_c) / 2, 0, 1)
    const float inv_n3 = p.inv_n3[s];
    const float wpix = (1.f - p.ssim_rate) * inv_n3;
    const float wssim = p.ssim_rate * inv_n3;
    const float* __restrict__ T = p.tgt_pl[s] + (size_t)b * 3 * plane;
    const float C1 = 81.f * (0.01f * 0.01f), C2 = 81.f * (0.03f * 0.03f);
    V3 tq[3][3];                         // target taps [row y-1 .. y+1][column x-1 .. x+1]
    V3 St = v3s(0.f), Stt = v3s(0.f);
    if (SSIM) {
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) tq[r][c] = sel_tap(T, plane, h, w, y - 1 + r, x - 1 + c);
      // the march's association: row sums (l + c) + r, window sums (row y-1 + row y) + row y+1
      V3 hT[3], hTT[3];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        hT[r] = (tq[r][0] + tq[r][1]) + tq[r][2];
        hTT[r] = vfma(tq[r][2], tq[r][2], vfma(tq[r][1], tq[r][1], tq[r][0] * tq[r][0]));
      }
      St = (hT[0] + hT[1]) + hT[2];
      Stt = (hTT[0] + hTT[1]) + hTT[2];
    } else {
      tq[1][1] = sel_tap(T, plane, h, w, y, x);
    }
    for (int i = 0; i < S; ++i) {
      const float* __restrict__ P = p.src_pl[s] + ((size_t)b * S + i) * 3 * plane;
      V3 pq[3][3];
      if (SSIM) {
#pragma unroll
        for (int r = 0; r < 3; ++r)
#pragma unroll
          for (int c = 0; c < 3; ++c) pq[r][c] = sel_tap(P, plane, h, w, y - 1 + r, x - 1 + c);
      } else {
        pq[1][1] = sel_tap(P, plane, h, w, y, x);
      }
      const V3 pc = pq[1][1], tc = tq[1][1];
      const float esum = fabsf(pc.a.x - tc.a.x) + fabsf(pc.a.y - tc.a.y) + fabsf(pc.b - tc.b);
      float e_id;
      if (SSIM) {
        V3 hP[3], hPP[3], hPT[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          hP[r] = (pq[r][0] + pq[r][1]) + pq[r][2];
          hPP[r] = vfma(pq[r][2], pq[r][2], vfma(pq[r][1], pq[r][1], pq[r][0] * pq[r][0]));
          hPT[r] = vfma(pq[r][2], tq[r][2], vfma(pq[r][1], tq[r][1], pq[r][0] * tq[r][0]));
        }
        const V3 Sp = (hP[0] + hP[1]) + hP[2];
        const V3 Spp = (hPP[0] + hPP[1]) + hPP[2];
        const V3 Spt = (hPT[0] + hPT[1]) + hPT[2];
        const V3 k2 = v3s(2.f), k9 = v3s(9.f), kC1 = v3s(C1), kC2 = v3s(C2);
        const V3 pp = Sp * Sp, tt = St * St, pt = Sp * St;
        const V3 n1 = vfma(k2, pt, kC1);
        const V3 n2 = vfma(k2, vfma(k9, Spt, vneg(pt)), kC2);
        const V3 d1v = (pp + tt) + kC1;
        const V3 d2v = (vfma(k9, Spp, vneg(pp)) + vfma(k9, Stt, vneg(tt))) + kC2;
        const V3 n = n1 * n2, dd = d1v * d2v;
        const V3 rd = v3(rcp_approx(dd.a.x), rcp_approx(dd.a.y), rcp_approx(dd.b));
        const V3 q = n * rd;
        const V3 raw = vfma(v3s(-0.5f), q, v3s(0.5f));
        const float sat3 = (__saturatef(raw.a.x) + __saturatef(raw.a.y)) + __saturatef(raw.b);
        e_id = wpix * esum + wssim * sat3;
      } else {
        e_id = wpix * esum;
      }
      if (best >= e_id) {                // an unwarped source matches at least as well: auto-masked
        sel = -1;
        break;
      }
    }
  }
  for (int i = 0; i < S; ++i) planes[(size_t)i * plane] = (i == sel) ? 1.f : 0.f;
  if (a.selection[s]) a.selection[s][(size_t)b * plane + pix] = (int8_t)sel;
}

}  // namespace
