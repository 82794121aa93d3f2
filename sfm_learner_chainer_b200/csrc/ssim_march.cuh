// ssim_march.cuh -- SSIM marching kernel: L1 + SSIM photometric terms (base_model.py:110-115, 126-142),
// forward and backward in one march.  Included by fused_loss.cu (shares its projection / blend helpers).
//
// A warp owns a strip of 28 interior columns (+2 halo columns each side = 32 lanes) x hseg rows and
// marches down rows y0-2 .. y1+1, lane = column.  Per row r:
//   stage A  warp the pixel (r, lane): projection, 4-tap gather, blend, image gradients dP/du, dP/dv
//   stage B  horizontal 3-sums of P, P^2, P.T, T, T^2 (neighbours through warp shuffles)
//   stage C  vertical 3-sums (register ring over the last three rows) -> SSIM at (r-1, lane), its loss
//            and the three gradient fields g_a, g_s, g_c (SURVEY A.7)
//   stage D  horizontal 3-sums of the gradient fields
//   stage E  vertical 3-sums -> dL/dP at (r-2, lane) = A(g_a) + 2P.A(g_s) + T.A(g_c) + L1 part
//   stage F  sampler / projection backward of pixel (r-2, lane) from its forward record
// The rings and the two-row delay line of forward records live in registers; the row loop is unrolled
// three times so that the ring rotation is pure renaming.  Each step runs only the stages whose row is used:
// C/D from the third step on, E/F from the fifth, no step past r = y1+1 (see RowStages).  No shared memory, no
// barrier; the only atomics are the per-task flush.  dL/dP accumulates as sum gq, sum gq*depth, sum gq*depth*y per lane
// (the lane's column x is constant along the march) and is expanded with Kinv before the flush.
#pragma once

namespace {

// Three channels as one packed pair (channels 0, 1: FFMA2 / FADD2 / FMUL2 of sm_100, one issue slot for two
// lanes) plus a scalar (channel 2).  Used for the SSIM statistics and gradient fields (tolerance-checked region; the
// individually rounded coordinate chain and the blend stay scalar).  The packed forms have the same FP32 throughput
// as scalar code; what they save is issue slots, which is what bounds this kernel.
struct V3 {
  float2 a;
  float b;
};
__device__ __forceinline__ V3 v3(float x, float y, float z) { V3 r; r.a = make_float2(x, y); r.b = z; return r; }
__device__ __forceinline__ V3 v3s(float s) { return v3(s, s, s); }
__device__ __forceinline__ V3 operator+(const V3& x, const V3& y) { V3 r; r.a = __fadd2_rn(x.a, y.a); r.b = x.b + y.b; return r; }
__device__ __forceinline__ V3 operator*(const V3& x, const V3& y) { V3 r; r.a = __fmul2_rn(x.a, y.a); r.b = x.b * y.b; return r; }
__device__ __forceinline__ V3 vfma(const V3& x, const V3& y, const V3& z) { V3 r; r.a = __ffma2_rn(x.a, y.a, z.a); r.b = fmaf(x.b, y.b, z.b); return r; }
__device__ __forceinline__ V3 vneg(const V3& x) { return v3(-x.a.x, -x.a.y, -x.b); }
__device__ __forceinline__ V3 vshfl_up(const V3& x) {
  return v3(__shfl_up_sync(0xffffffffu, x.a.x, 1), __shfl_up_sync(0xffffffffu, x.a.y, 1), __shfl_up_sync(0xffffffffu, x.b, 1));
}
__device__ __forceinline__ V3 vshfl_down(const V3& x) {
  return v3(__shfl_down_sync(0xffffffffu, x.a.x, 1), __shfl_down_sync(0xffffffffu, x.a.y, 1), __shfl_down_sync(0xffffffffu, x.b, 1));
}

struct StripTask {
  int s, b, x0, y0, y1;
};

__device__ __forceinline__ StripTask decode_strip(const SfmFusedParams& p, int t) {
  StripTask k;
  int s = 0;
#pragma unroll
  for (int q = 1; q < SFM_MAX_SCALES; ++q)
    if (q < p.ns && t >= p.tasks.task_begin[q]) s = q;
  t -= p.tasks.task_begin[s];
  k.s = s;
  const int seg = t % p.tasks.nseg[s];
  t /= p.tasks.nseg[s];
  const int strip = t % p.tasks.nstrip[s];
  k.b = t / p.tasks.nstrip[s];
  k.x0 = strip * SFM_SSIM_IW;
  k.y0 = seg * p.tasks.hseg;
  k.y1 = min(k.y0 + p.tasks.hseg, p.h[s]);
  return k;
}

// forward record of one pixel, kept for two rows until its backward runs
struct Rec {
  float Ix[3], Iy[3];     // dP_c/du, dP_c/dv (pixel units)
  float P[3], T[3];
  float q0, q1, q2, r;    // projection, 1/z (0 when out of view)
  float depth;
  float dsc;              // depth, or depth * (d disp / d x) when the disparity input is the pre-activation map
};

template <int N>
struct IC { static constexpr int value = N; };

// The stages one row step runs.  A task of h rows marches h + 4 steps, j = 0 .. h+3 on rows r = y0-2+j; step j blends
// row r (A, B), takes the SSIM of row r-1 (C, D) and the backward of row r-2 (E, F).  Rows y0-2 .. y1+1 feed the
// windows of the owned rows, the gradient fields of rows y0-1 .. y1 feed their dL/dP, so C/D are needed from step 2
// and E/F from step 4 on.  The ring slots those skipped stages would fill are overwritten before any step reads them.
// The march ends with step h+3: no step runs past row y1+1.
enum RowStages {
  ROW_AB,       // steps 0, 1
  ROW_ABCD,     // steps 2, 3
  ROW_ALL,      // steps 4 .. h+3
};

// NW = warps per CTA.  NW == 1: one warp walks the strip segment once per source.  NW == 2 (two sources, small
// batches): the two warps of a CTA walk the same segment at the same time, one source each, so a task is half as
// long and -- for the same number of resident warps -- twice as tall (half the halo rows).  gdisp stays
// deterministic: warp 1 hands its per-row term to warp 0 through shared memory (one CTA barrier per row) and warp 0
// applies both in the order of the sequential loop, with the same fused multiply-adds.
// SREC: where the two-row delay line of forward records lives.  true: shared memory (34 LDS/STS wavefronts per row,
// 168 registers, 3 warps per scheduler) -- the throughput form for grids of several waves.  false: registers (250
// registers, 2 warps per scheduler, 6 % fewer instructions and a third fewer L1 data-pipe wavefronts) -- faster whenever
// the whole grid is resident at once anyway (cfg2: 29.3 -> 26.6 us), slower when occupancy counts (cfg5: 933 -> 952 us).
// IMG (GRAD, NW == 1, SREC only): also the image gradients.  With h_a = (dL/dSt) / 2 -- the mirror image of g_a -- and
// (dL/dStt) / 9 == g_s (d2 holds Spp and Stt with the same factor), dL/dT = 2 A(h_a) + 18 T A(g_s) + 18 P A(g_c) + the
// L1 part: one more gradient field in the ring.  The task owns gtgt like gdisp (stored by the first source, then
// accumulated); dL/dP is scattered to the four taps of every in-view pixel with fp32 reductions, from the tap index
// and the two fractions the forward record carries in three more fields.
// SNIP: per-snippet terms, as in sfm_l1_march_kernel.
// PIX (NW == 1, SREC, no IMG / DEBUG): per-pixel terms.  The weight M of a pixel is loaded with its taps and is needed at
// three lags: stage A of row r (the L1 loss partial), row r-1 (lw of the SSIM loss and wl of the gradient fields: a
// one-step register carry) and row r-2 (the L1 part of dL/dP in stage F: one more field of the forward record).  Stage C
// stores the map wpix * esum + wssim * sum_c sat(raw_c) = d total / d M of the owned pixels of row r-1, whose esum is
// carried one step like its weight (p.pix_map_masked for masked pixels).  M = 1 multiplies exactly: unit weights give
// bitwise the plain step.
template <bool GRAD, bool ACCUM, bool DEBUG, bool RAW, int NW, bool SREC = true, bool IMG = false, bool SNIP = false,
          bool PIX = false>
__global__ void __launch_bounds__(32 * NW, (IMG ? SFM_SSIM_IMG_MIN_WARPS : SREC ? SFM_SSIM_MIN_WARPS : SFM_SSIM_REG_MIN_WARPS) / NW)
sfm_ssim_march_kernel(const __grid_constant__ SfmFusedParams p) {
  static_assert(!IMG || (GRAD && NW == 1 && SREC), "image gradients: GRAD, one warp per CTA, shared-memory records");
  static_assert(!PIX || (NW == 1 && SREC && !IMG && !DEBUG), "per-pixel terms: one warp per CTA, shared-memory records");
  constexpr int NREC = IMG ? 21 : PIX ? 19 : 18;        // fields of a forward record
  constexpr int NG = IMG ? 4 : 3;                       // gradient fields: g_a, g_s, g_c (, h_a)
  __shared__ float4 sP_all[NW][3];
  __shared__ float sG[(NW > 1) ? 3 * 2 * 32 : 1];       // [ring slot][gdd | dsc][lane] of warp 1's row term
  const int wi = (NW > 1) ? (int)(threadIdx.x >> 5) : 0;
  float4* const sP = sP_all[wi];
  // warp-uniform base pointers, re-read (broadcast LDS.64) where they are used: at 168 registers ptxas otherwise
  // re-derives them from the kernel parameters inside the row loop (64-bit multiplies per row, seen in the SASS)
  struct RowPtrs {
    const float* img;
    const float* tgt;
    const float* disp;
    float* gdisp;
  };
  __shared__ RowPtrs s_ptrs_all[NW];
  volatile RowPtrs* const pp = &s_ptrs_all[wi];
  // two-row delay line of forward records: [slot][field][lane], written in stage A of row r and read back by
  // the same lane in stages E/F two steps later (no synchronisation needed).  In registers these 51 values
  // pushed the kernel over its 168-register budget (17-27 local-memory spills per three rows).
  __shared__ float sRec[(GRAD && SREC) ? NW * 3 * NREC * 32 : 1];
  // IMG: gtgt of the snippet, gsrc of the pass's source (scale s), re-read like s_ptrs
  __shared__ float* s_img_ptrs[2];
  // PIX: weight and map of the pass's source (scale s), re-read like s_ptrs
  __shared__ float* s_pix_ptrs[2];
  const int lane = threadIdx.x & 31;
  float* const myrec = sRec + wi * (3 * NREC * 32) + lane;
  const StripTask t = decode_strip(p, blockIdx.x);
  const int s = t.s, b = t.b, h = p.h[s], w = p.w[s], S = p.S;
  const Geo geo = make_geo(p, s);
  const int xx = t.x0 - 2 + lane;                       // this lane's image column (may be outside)
  const bool col_in = (xx >= 0) && (xx < w);
  const bool col_own = (lane >= 2) && (lane < 2 + SFM_SSIM_IW) && (xx < w);
  float gyv = p.gy ? __ldg(p.gy) : 1.f;
  if (SNIP && p.snip_w) gyv *= __ldg(p.snip_w + b);        // per-snippet weight
  const float inv_n3 = p.inv_n3[s];
  const float wpix = gyv * (1.f - p.ssim_rate) * inv_n3;
  const float wssim = gyv * p.ssim_rate * inv_n3;
  // SSIM on raw 3x3 window SUMS (9 x the means): the 1/81 factors of numerator and denominator cancel
  const float C1 = 81.f * (0.01f * 0.01f), C2 = 81.f * (0.03f * 0.03f);
  // everything below reads what the prologue kernel wrote (pyramid, tables, the smoothness tasks' gdisp)
  cudaGridDependencySynchronize();
  cudaTriggerProgrammaticLaunchCompletion();           // lets the epilogue's CTAs become resident while this grid drains (after the
                                                       // wait: the epilogue reads the prologue's smoothness partials ahead of its own wait)
  const float* __restrict__ kinvp = p.kinv + ((size_t)b * p.ns + s) * 9;
  const float xf = (float)xx;
  const bool raw = RAW && ((p.raw_disp_mask >> s) & 1u);    // RAW: some scale takes the pre-activation disparity map
  const float kk0 = __ldg(kinvp + 0), kk1 = __ldg(kinvp + 1), kk2 = __ldg(kinvp + 2);
  const float kk3 = __ldg(kinvp + 3), kk4 = __ldg(kinvp + 4), kk5 = __ldg(kinvp + 5);
  const float kk6 = __ldg(kinvp + 6), kk7 = __ldg(kinvp + 7), kk8 = __ldg(kinvp + 8);
  // ray = Kinv.(x, y, 1): r_k = (k_k0*x + k_k1*y) + k_k2 ; the x products are row invariant
  const float rxx = __fmul_rn(kk0, xf), ryx = __fmul_rn(kk3, xf), rzx = __fmul_rn(kk6, xf);
  const int plane = h * w;
  const float* __restrict__ disp = p.disp[s] + (size_t)b * plane;
  const float* __restrict__ tgt = p.tgt_pl[s] + (size_t)b * 3 * plane;
  float* __restrict__ gdisp = GRAD ? p.gdisp[s] + (size_t)b * plane : nullptr;
  const size_t src_img = (size_t)3 * plane;
  float pix_part = 0.f, ssim_part = 0.f;
  const int r_begin = t.y0 - 2, r_end = t.y1 + 2;      // rows [r_begin, r_end) are warped
  const bool opaque_true = p.tasks.hseg != 0x7fffffff;       // always true, unknown to ptxas: basic-block fence (see step)

  for (int i = (NW > 1) ? wi : 0; i < ((NW > 1) ? wi + 1 : S); ++i) {
    __syncwarp();
    if (lane < 12) reinterpret_cast<float*>(sP)[lane] = __ldg(p.proj + (((size_t)b * S + i) * p.ns + s) * 12 + lane);
    __syncwarp();
    const float P3 = sP[0].w, P7 = sP[1].w, P11 = sP[2].w;
    float accA[3] = {0.f, 0.f, 0.f}, accB[3] = {0.f, 0.f, 0.f}, accC[3] = {0.f, 0.f, 0.f};
    const bool first = (i == 0);
    const bool writer = (NW == 1) || (wi == 0);          // the warp that loads / stores gdisp
    if (lane == 0) {
      s_ptrs_all[wi].img = p.src_pl[s] + ((size_t)b * S + i) * src_img;
      s_ptrs_all[wi].tgt = tgt;
      s_ptrs_all[wi].disp = disp;
      s_ptrs_all[wi].gdisp = gdisp;
      if (IMG) {
        s_img_ptrs[0] = p.gtgt[s] ? p.gtgt[s] + (size_t)b * 3 * plane : nullptr;
        s_img_ptrs[1] = p.gsrc[s] ? p.gsrc[s] + ((size_t)b * S + i) * src_img : nullptr;
      }
      if (PIX) {
        s_pix_ptrs[0] = p.pix_w[s] ? const_cast<float*>(p.pix_w[s]) + ((size_t)b * S + i) * plane : nullptr;
        s_pix_ptrs[1] = p.pix_map[s] ? p.pix_map[s] + ((size_t)b * S + i) * plane : nullptr;
      }
    }
    __syncwarp();
    // rings: window row sums (P, P^2, P.T, T, T^2 per channel), gradient-field row sums, forward records.  No
    // initial value: with the stage schedule of RowStages every slot is written before a step reads it.
    V3 hs[3][5], gs[3][NG];       // [ring slot][field]: (P, P^2, P.T, T, T^2) and (g_a, g_s, g_c (, h_a)) row sums, three channels each
    Rec rec[3];
    bool mask[3];                                        // all-zero mask of the row's pixel (base_model.py:96)
    float dq[3] = {1.f, 1.f, 1.f};                       // disparity / target rows fetched ahead
    float Tq[3][3];
    auto load_dT = [&](int r, float& dd, float* TT) {
      dd = 1.f;
      TT[0] = TT[1] = TT[2] = 0.f;
      if (col_in && (r >= 0) && (r < h) && (r < r_end)) {
        const unsigned o = (unsigned)(r * w + xx);
        const float* tb = pp->tgt;
        dd = __ldg(pp->disp + o);
        TT[0] = __ldg(tb + o);
        TT[1] = __ldg(tb + (o + geo.plane));
        TT[2] = __ldg(tb + (o + 2u * geo.plane));
      }
    };
    // pending rows: projected, gathers in flight, consumed by a later step.  The loop keeps one (pend[0], refilled one
    // row ahead); the head of the register-record instances keeps two, refilled two rows ahead (see the march below)
    struct Pend {
      Taps I;
      float wa, wb, wc, wd, q0, q1, q2, r, depth, dsc;
      unsigned idx;                                      // IMG: tap (v0, u0)
      float mw;                                          // PIX: per-pixel weight
    };
    Pend pend[2];
    float g_old = 0.f;
    float w_lag1 = 1.f, e_lag1 = 0.f;                    // PIX: weight and L1 sum of the row before the current one

    // refill: project row r into pending row pn (its disparity was fetched a step earlier), issue its gathers, fetch
    // row r+1's disparity / target (unless LOAD_NEXT is false) and the partial gdisp of the row whose backward runs next
    auto refill = [&](auto SLOT, Pend& pn, const int r, auto LOAD_NEXT) {
      constexpr int sl = decltype(SLOT)::value, nx = (sl + 1) % 3;
      const bool in_img = col_in && (r >= 0) && (r < h) && (r < r_end);
      float d = dq[sl], dact = 1.f;
      if (raw) d = sfm_disp_act(d, dact);      // producer-side fusion: pre-activation disparity map (warp-uniform branch)
      pn.depth = rcp_newton(d);
      if (RAW) pn.dsc = raw ? pn.depth * dact : pn.depth;
      const float yf = (float)r;
      const float rx = __fadd_rn(__fadd_rn(rxx, __fmul_rn(kk1, yf)), kk2);
      const float ry = __fadd_rn(__fadd_rn(ryx, __fmul_rn(kk4, yf)), kk5);
      const float rz = __fadd_rn(__fadd_rn(rzx, __fmul_rn(kk7, yf)), kk8);
      const float X = __fmul_rn(pn.depth, rx), Y = __fmul_rn(pn.depth, ry), Z = __fmul_rn(pn.depth, rz);
      float P[12];
      {
        const float4 a = sP[0], bb = sP[1], c = sP[2];
        P[0] = a.x; P[1] = a.y; P[2] = a.z; P[3] = a.w;
        P[4] = bb.x; P[5] = bb.y; P[6] = bb.z; P[7] = bb.w;
        P[8] = c.x; P[9] = c.y; P[10] = c.z; P[11] = c.w;
      }
      PairFwd f;
      pair_project(P, X, Y, Z, geo, f, in_img);
      pn.wa = f.wa; pn.wb = f.wb; pn.wc = f.wc; pn.wd = f.wd;
      pn.q0 = f.q0; pn.q1 = f.q1; pn.q2 = f.q2; pn.r = f.r;
      if (IMG) pn.idx = f.idx;
      gather_taps(pp->img, geo, f, pn.I);
      if (PIX) {
        float* const volatile* pq = s_pix_ptrs;
        const float* wq = pq[0];
        pn.mw = (in_img && wq) ? __ldg(wq + (unsigned)(r * w + xx)) : 1.f;
      }
      if (decltype(LOAD_NEXT)::value) load_dT(r + 1, dq[nx], Tq[nx]);
      if (GRAD && (ACCUM || !first) && writer) {
        const int rf = r - 2;
        g_old = (col_own && rf >= t.y0 && rf < t.y1) ? ld_global(pp->gdisp + (unsigned)(rf * w + xx)) : 0.f;
      }
      if (DEBUG && in_img && col_own && (r >= t.y0) && (r < t.y1) && p.dbg_u0[s]) {
        const size_t o = ((size_t)b * S + i) * plane + (size_t)r * w + xx;
        SfmCoord c;
        sfm_project(P, X, Y, Z, w, h, geo.hw, geo.hh, c);
        p.dbg_u0[s][o] = f.inb ? (int)(f.idx % (unsigned)w) : c.u0;
        p.dbg_v0[s][o] = f.inb ? (int)(f.idx / (unsigned)w) : c.v0;
        p.dbg_inb[s][o] = f.inb ? 1 : 0;
      }
    };

    // step of row r: consumes pending row pend[PQ]; AHEAD = 1 refills row r+1 into it, 2 row r+2, 0 nothing
    auto step = [&](auto PH, auto ST, auto PQ, auto AHEAD, const int r) {
      constexpr int cur = decltype(PH)::value, pv1 = (cur + 2) % 3, pv2 = (cur + 1) % 3;
      constexpr int stages = decltype(ST)::value, ahead = decltype(AHEAD)::value;
      Pend& pa = pend[decltype(PQ)::value];
      const Taps& I = pa.I;
      const int rf = r - 2;
      const bool do_f = col_own && rf >= t.y0 && rf < t.y1;
      const float g_prev = g_old;
      const float m_cur = PIX ? pa.mw : 1.f;             // weight of row r (pa is refilled below)
      float e_cur = 0.f;
      // ---------------- stage A: blend pixel (r, lane) from the taps gathered during the previous step
      Rec& rc_ = rec[cur];
      {
        const float* T = Tq[cur];
        const float w1 = __fmul_rn(pa.wa, pa.wc), w2 = __fmul_rn(pa.wb, pa.wc);
        const float w3 = __fmul_rn(pa.wa, pa.wd), w4 = __fmul_rn(pa.wb, pa.wd);
        const float P0 = sfm_blend(w1, w2, w3, w4, I.a[0], I.b[0], I.c[0], I.d[0]);
        const float P1 = sfm_blend(w1, w2, w3, w4, I.a[1], I.b[1], I.c[1], I.d[1]);
        const float P2 = sfm_blend(w1, w2, w3, w4, I.a[2], I.b[2], I.c[2], I.d[2]);
        const bool m = (P0 == 0.f) && (P1 == 0.f) && (P2 == 0.f);               // true outside the image / view
        const bool own = col_own && (r >= t.y0) && (r < t.y1);
        if (PIX) {
          e_cur = m ? 0.f : (fabsf(P0 - T[0]) + fabsf(P1 - T[1]) + fabsf(P2 - T[2]));
          pix_part += own ? e_cur * m_cur : 0.f;
        } else {
          pix_part += (own && !m) ? (fabsf(P0 - T[0]) + fabsf(P1 - T[1]) + fabsf(P2 - T[2])) : 0.f;
        }
        mask[cur] = m;
        rc_.P[0] = P0; rc_.P[1] = P1; rc_.P[2] = P2;
        rc_.T[0] = T[0]; rc_.T[1] = T[1]; rc_.T[2] = T[2];
        if (GRAD) {
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            rc_.Ix[c] = pa.wc * (I.b[c] - I.a[c]) + pa.wd * (I.d[c] - I.c[c]);
            rc_.Iy[c] = pa.wa * (I.c[c] - I.a[c]) + pa.wb * (I.d[c] - I.b[c]);
          }
          rc_.q0 = pa.q0; rc_.q1 = pa.q1; rc_.q2 = pa.q2; rc_.r = pa.r;
          rc_.depth = pa.depth;
          rc_.dsc = RAW ? pa.dsc : pa.depth;
          if (SREC) {
            float* o = myrec + cur * NREC * 32;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              o[(0 + c) * 32] = rc_.Ix[c];
              o[(3 + c) * 32] = rc_.Iy[c];
              o[(6 + c) * 32] = rc_.P[c];
              o[(9 + c) * 32] = rc_.T[c];
            }
            o[12 * 32] = pa.q0; o[13 * 32] = pa.q1; o[14 * 32] = pa.q2; o[15 * 32] = pa.r; o[16 * 32] = pa.depth;
            if (RAW) o[17 * 32] = pa.dsc;
            if (IMG) { o[18 * 32] = __uint_as_float(pa.idx); o[19 * 32] = pa.wb; o[20 * 32] = pa.wd; }
            if (PIX) o[18 * 32] = m_cur;
          }
        }
        if (DEBUG && own && p.dbg_P[s]) {
          float* o = p.dbg_P[s] + ((size_t)b * S + i) * 3 * plane + (size_t)r * w + xx;
          o[0] = P0;
          o[plane] = P1;
          o[2 * (size_t)plane] = P2;
        }
      }
      // ---------------- refill for row r + 1 (r + 2 in the head): its gathers fly while stages B..F of this step run
      if constexpr (ahead == 1) refill(IC<pv2>{}, pa, r + 1, IC<1>{});     // ring slot of row r+1 == (cur + 1) % 3
      if constexpr (ahead == 2) refill(IC<pv1>{}, pa, r + 2, IC<1>{});     // ring slot of row r+2 == (cur + 2) % 3
      // Basic-block fence.  The refill has no consumer before the next step, so ptxas' critical-path scheduler
      // otherwise sinks the projection and the four gathers to the end of the step (seen in the SASS; ncu:
      // half of all stall samples were long-scoreboard waits on the taps ~60 instructions after their issue).
      // A branch it cannot fold keeps them ahead of stages B..F, which then cover the latency.
      if (opaque_true) {
      // ---------------- stage B: row sums of P, P^2, P.T, T, T^2 over lanes-1..+1 (zero outside the image)
      {
        const V3 pv = v3(rc_.P[0], rc_.P[1], rc_.P[2]), tv = v3(rc_.T[0], rc_.T[1], rc_.T[2]);
        const V3 pl = vshfl_up(pv), prr = vshfl_down(pv), tl = vshfl_up(tv), tr = vshfl_down(tv);
        V3* h0 = hs[cur];
        h0[0] = (pl + pv) + prr;
        h0[1] = vfma(prr, prr, vfma(pv, pv, pl * pl));
        h0[2] = vfma(prr, tr, vfma(pv, tv, pl * tl));
        h0[3] = (tl + tv) + tr;
        h0[4] = vfma(tr, tr, vfma(tv, tv, tl * tl));
      }
      if constexpr (stages != ROW_AB) {
      // ---------------- stage C: SSIM at (rc = r-1, lane) from rows r-2, r-1, r
      const int rc = r - 1;
      V3 g0[NG];
      {
        const V3* h0 = hs[cur];
        const V3* h1 = hs[pv1];
        const V3* h2 = hs[pv2];
        const bool c_in = col_in && (rc >= 0) && (rc < h);
        const bool live_px = c_in && !mask[pv1];
        const bool own_c = col_own && (rc >= t.y0) && (rc < t.y1);
        const float lw = (live_px && own_c) ? (PIX ? w_lag1 : 1.f) : 0.f;
        // window sums: Sp = 9a, Spp = 9 A(P^2), Spt = 9 A(PT), St = 9 my, Stt = 9 A(T^2)
        const V3 Sp = (h2[0] + h1[0]) + h0[0];
        const V3 Spp = (h2[1] + h1[1]) + h0[1];
        const V3 Spt = (h2[2] + h1[2]) + h0[2];
        const V3 St = (h2[3] + h1[3]) + h0[3];
        const V3 Stt = (h2[4] + h1[4]) + h0[4];
        // 81 x the reference's quantities: n1 = 2 a my + c1, n2 = 2 sxy + c2, d1 = a^2 + my^2 + c1, d2 = sx + sy + c2
        const V3 k2 = v3s(2.f), k9 = v3s(9.f), kC1 = v3s(C1), kC2 = v3s(C2);
        const V3 pp = Sp * Sp, tt = St * St, pt = Sp * St;
        const V3 n1 = vfma(k2, pt, kC1);
        const V3 n2 = vfma(k2, vfma(k9, Spt, vneg(pt)), kC2);
        const V3 d1v = (pp + tt) + kC1;
        const V3 d2v = (vfma(k9, Spp, vneg(pp)) + vfma(k9, Stt, vneg(tt))) + kC2;
        const V3 n = n1 * n2, dd = d1v * d2v;
        const V3 rd = v3(rcp_approx(dd.a.x), rcp_approx(dd.a.y), rcp_approx(dd.b));
        const V3 q = n * rd;                          // SSIM
        const V3 raw = vfma(v3s(-0.5f), q, v3s(0.5f));
        const float sat3 = (__saturatef(raw.a.x) + __saturatef(raw.a.y)) + __saturatef(raw.b);
        ssim_part = fmaf(sat3, lw, ssim_part);
        if (PIX) {
          float* const volatile* pq = s_pix_ptrs;
          float* mq = pq[1];
          if (own_c && c_in && mq) st_global(mq + (unsigned)(rc * w + xx), live_px ? wpix * e_lag1 + wssim * sat3 : p.pix_map_masked);
        }
        if (GRAD) {
          // d raw / d(Sp, Spp, Spt) with n, d in the 81x units (SURVEY A.7 rescaled):
          //   g_n = dL/dn = -0.5 w / d ; g_d = dL/dd = 0.5 w n / d^2
          //   dn/dSp = 2 St (n2 - n1) ; dn/dSpt = 18 n1 ; dd/dSp = 2 Sp (d2 - d1) ; dd/dSpp = 9 d1
          // F.clip passes gradient inside [0, 1]
          const float wl = live_px ? (PIX ? -0.5f * wssim * w_lag1 : -0.5f * wssim) : 0.f;
          const V3 wv = v3((raw.a.x >= 0.f && raw.a.x <= 1.f) ? wl : 0.f, (raw.a.y >= 0.f && raw.a.y <= 1.f) ? wl : 0.f,
                           (raw.b >= 0.f && raw.b <= 1.f) ? wl : 0.f);
          const V3 g_n = wv * rd;
          const V3 g_d = vneg(g_n) * q;
          g0[0] = vfma(g_n * St, n2 + vneg(n1), (g_d * Sp) * (d2v + vneg(d1v)));   // (dL/dSp) / 2
          g0[1] = g_d * d1v;                                                       // (dL/dSpp) / 9
          g0[2] = g_n * n1;                                                        // (dL/dSpt) / 18
          if constexpr (IMG) g0[3] = vfma(g_n * Sp, n2 + vneg(n1), (g_d * St) * (d2v + vneg(d1v)));  // (dL/dSt) / 2
        }
      }
      if (GRAD) {
        // ---------------- stage D: row sums of the three gradient fields of row rc
        V3* gh0 = gs[cur];
#pragma unroll
        for (int q = 0; q < NG; ++q) gh0[q] = (vshfl_up(g0[q]) + g0[q]) + vshfl_down(g0[q]);
        if constexpr (stages != ROW_ABCD) {
        // ---------------- stages E + F: dL/dP and the warp backward for pixel (rf = r-2, lane)
        const V3* g1 = gs[pv1];
        const V3* g2 = gs[pv2];
        Rec rb = rec[pv2];
        if (SREC) {
          const float* o = myrec + pv2 * NREC * 32;
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            rb.Ix[c] = o[(0 + c) * 32];
            rb.Iy[c] = o[(3 + c) * 32];
            rb.P[c] = o[(6 + c) * 32];
            rb.T[c] = o[(9 + c) * 32];
          }
          rb.q0 = o[12 * 32]; rb.q1 = o[13 * 32]; rb.q2 = o[14 * 32]; rb.r = o[15 * 32]; rb.depth = o[16 * 32];
          rb.dsc = RAW ? o[17 * 32] : rb.depth;
        }
        const bool mf = mask[pv2];
        const float wpf = PIX ? wpix * (SREC ? myrec[pv2 * NREC * 32 + 18 * 32] : 1.f) : wpix;   // PIX: weight of row rf
        float gP[3], gT[3];
        {
          const V3 Aa = (g2[0] + g1[0]) + gh0[0];
          const V3 As = (g2[1] + g1[1]) + gh0[1];
          const V3 Ac = (g2[2] + g1[2]) + gh0[2];
          // dL/dP = sum over the 3x3 windows containing the pixel of dL/dSp + 2P dL/dSpp + T dL/dSpt
          //       = 2 Aa + 18 P As + 18 T Ac
          const V3 Pb = v3(rb.P[0], rb.P[1], rb.P[2]), Tb = v3(rb.T[0], rb.T[1], rb.T[2]);
          const V3 gsv = vfma(v3s(18.f), vfma(Tb, Ac, Pb * As), v3s(2.f) * Aa);
          const float gs3[3] = {gsv.a.x, gsv.a.y, gsv.b};
          float gt3[3] = {0.f, 0.f, 0.f};
          if constexpr (IMG) {
            // dL/dT = 2 A(h_a) + 18 T As + 18 P Ac
            const V3 Ah = (g2[3] + g1[3]) + gh0[3];
            const V3 gtv = vfma(v3s(18.f), vfma(Pb, Ac, Tb * As), v3s(2.f) * Ah);
            gt3[0] = gtv.a.x; gt3[1] = gtv.a.y; gt3[2] = gtv.b;
          }
#pragma unroll
          for (int c = 0; c < 3; ++c) {
            const float gl1 = mf ? 0.f : sfm_sign_times(rb.P[c] - rb.T[c], wpf);
            gP[c] = do_f ? gs3[c] + gl1 : 0.f;
            if (IMG) gT[c] = do_f ? gt3[c] - gl1 : 0.f;
          }
        }
        if (IMG && do_f) {
          float* const volatile* ip = s_img_ptrs;
          float* gt = ip[0];
          float* gsrc = ip[1];
          if (gt) {
            float* q = gt + (unsigned)(rf * w + xx);
            if (first) {
              q[0] = gT[0]; q[geo.plane] = gT[1]; q[2u * geo.plane] = gT[2];
            } else {
              q[0] += gT[0]; q[geo.plane] += gT[1]; q[2u * geo.plane] += gT[2];
            }
          }
          if (gsrc && rb.r != 0.f) {
            // in view: wa = 1 - wb and wc = 1 - wd exactly (wb = u - u0 is exact, and so is the difference)
            const float* o = myrec + pv2 * NREC * 32;
            const unsigned idx = __float_as_uint(o[18 * 32]);
            const float wb = o[19 * 32], wd = o[20 * 32];
            const float wa = __fsub_rn(1.f, wb), wc = __fsub_rn(1.f, wd);
            const float w1 = __fmul_rn(wa, wc), w2 = __fmul_rn(wb, wc), w3 = __fmul_rn(wa, wd), w4 = __fmul_rn(wb, wd);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
              float* qc = gsrc + (idx + (unsigned)c * geo.plane);
              atomicAdd(qc, gP[c] * w1);
              atomicAdd(qc + 1, gP[c] * w2);
              atomicAdd(qc + w, gP[c] * w3);
              atomicAdd(qc + w + 1, gP[c] * w4);
            }
          }
        }
        // sampler + projection backward (SURVEY A.6); out-of-view pixels have Ix = Iy = 0 and r = 0
        const float gu = gP[0] * rb.Ix[0] + gP[1] * rb.Ix[1] + gP[2] * rb.Ix[2];
        const float gv = gP[0] * rb.Iy[0] + gP[1] * rb.Iy[1] + gP[2] * rb.Iy[2];
        const float gq0 = gu * rb.r, gq1 = gv * rb.r;
        const float gq2 = -(gq0 * rb.q0 + gq1 * rb.q1) * rb.r;
        const float gdd = gq0 * (rb.q0 - P3) + gq1 * (rb.q1 - P7) + gq2 * (rb.q2 - P11);
        const float yfb = (float)rf;
        const float e0 = gq0 * rb.depth, e1 = gq1 * rb.depth, e2 = gq2 * rb.depth;
        accA[0] += e0; accA[1] += e1; accA[2] += e2;
        accB[0] = fmaf(e0, yfb, accB[0]); accB[1] = fmaf(e1, yfb, accB[1]); accB[2] = fmaf(e2, yfb, accB[2]);
        accC[0] += gq0; accC[1] += gq1; accC[2] += gq2;
        float* gp = pp->gdisp + (unsigned)(rf * w + xx);
        float gval = g_prev - gdd * rb.dsc;
        if (NW > 1) {
          // warp 1 -> warp 0: (gdd, dsc) of the second source for this row; warp 0 continues the sequential chain
          float* slot = sG + cur * 64 + lane;
          if (wi == 1) { slot[0] = gdd; slot[32] = rb.dsc; }
          __syncthreads();
          if (wi == 0) gval = gval - slot[0] * slot[32];
        }
        if (do_f && writer) st_global(gp, gval);
        }  // E + F
      }
      }  // C + D
      }  // opaque_true
      if (PIX) { w_lag1 = m_cur; e_lag1 = e_cur; }
    };

    // r_end - r_begin = h + 4 >= 5 steps: the four head steps, then groups of three (ring rotation = renaming) that
    // leave the loop right after the step of row r_end - 1.  The exits sit inside the loop: a peeled tail after it
    // (straight-line copies of the step) pushed the shared-memory-record instances past 168 registers.  The stage sets
    // depend only on the step, so both warps of an NW = 2 CTA meet the per-row barrier of stage F on the same steps.
    // The head's steps are short, so with one row of gathers in flight each of them waits a whole memory latency.  In
    // the register-record instances (grids resident at once: every warp is in its head at the same time) the head
    // keeps two pending rows: rows r_begin and r_begin+1 are gathered together, the head steps refill two rows ahead
    // and the last one refills nothing, which hands the loop one pending row, pend[0] (cfg2: 25.2 -> 24.7 us).  The
    // shared-memory-record instances run many waves, where other warps cover the head; there the second pending row
    // cost 2 % more instructions in the loop (ptxas' allocation) and local-memory spills in the DEBUG instances.
    load_dT(r_begin, dq[0], Tq[0]);
    if constexpr (!SREC) {
      load_dT(r_begin + 1, dq[1], Tq[1]);
      refill(IC<0>{}, pend[0], r_begin, IC<0>{});
      refill(IC<1>{}, pend[1], r_begin + 1, IC<1>{});
      step(IC<0>{}, IC<ROW_AB>{}, IC<0>{}, IC<2>{}, r_begin);
      step(IC<1>{}, IC<ROW_AB>{}, IC<1>{}, IC<2>{}, r_begin + 1);
      step(IC<2>{}, IC<ROW_ABCD>{}, IC<0>{}, IC<2>{}, r_begin + 2);
      step(IC<0>{}, IC<ROW_ABCD>{}, IC<1>{}, IC<0>{}, r_begin + 3);
    } else {
      refill(IC<0>{}, pend[0], r_begin, IC<1>{});
      step(IC<0>{}, IC<ROW_AB>{}, IC<0>{}, IC<1>{}, r_begin);
      step(IC<1>{}, IC<ROW_AB>{}, IC<0>{}, IC<1>{}, r_begin + 1);
      step(IC<2>{}, IC<ROW_ABCD>{}, IC<0>{}, IC<1>{}, r_begin + 2);
      step(IC<0>{}, IC<ROW_ABCD>{}, IC<0>{}, IC<1>{}, r_begin + 3);
    }
#pragma unroll 1
    for (int r = r_begin + 4;; r += 3) {
      step(IC<1>{}, IC<ROW_ALL>{}, IC<0>{}, IC<1>{}, r);
      if (r + 1 >= r_end) break;
      step(IC<2>{}, IC<ROW_ALL>{}, IC<0>{}, IC<1>{}, r + 1);
      if (r + 2 >= r_end) break;
      step(IC<0>{}, IC<ROW_ALL>{}, IC<0>{}, IC<1>{}, r + 2);
      if (r + 3 >= r_end) break;
    }
    // The taps of the last refill are dead once the loop is left, so ptxas sinks every step's gathers past the
    // fence and the exit test into the next step, right in front of their use (the whole gather latency exposed
    // per row: 10 % / 17 % slower at cfg2 / cfg5).  A use it cannot rule out keeps them live on the way out.
    if (!opaque_true) {
#pragma unroll
      for (int c = 0; c < 3; ++c) pix_part += ((pend[0].I.a[c] + pend[0].I.b[c]) + pend[0].I.c[c]) + pend[0].I.d[c];
    }
    // ---- flush: expand (A, B, C) to dL/dP = sum gq (x) (X, Y, Z, 1) with X = depth*((k0 x + k2) + k1 y) ...
    const bool last = (NW > 1) || (i == S - 1);
    if (GRAD || last) {
      float acc[12];
      if (GRAD) {
        const float cx = rxx + kk2, cy = ryx + kk5, cz = rzx + kk8;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          acc[k * 4 + 0] = cx * accA[k] + kk1 * accB[k];
          acc[k * 4 + 1] = cy * accA[k] + kk4 * accB[k];
          acc[k * 4 + 2] = cz * accA[k] + kk7 * accB[k];
          acc[k * 4 + 3] = accC[k];
        }
      }
      flush_dP<SNIP>(p, acc, b, i, s, lane, last ? pix_part * inv_n3 : 0.f, last ? ssim_part * inv_n3 : 0.f, 0.f, 0, 3, -1, GRAD);
    }
  }
}

}  // namespace
