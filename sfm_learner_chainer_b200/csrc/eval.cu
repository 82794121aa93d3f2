// eval.cu -- inference-side depth evaluation of one batch on the device (SURVEY section 8(f) rank 4):
//   evaluate.py:94-103     pred = F.resize_images(pred_depth, gt.shape[1:]); F.clip(pred, min_depth, max_depth)[:, 0];
//                          pred[mask], gt[mask]; pred *= median(gt) / median(pred)
//   kitti_eval/depth_util.py:6-22   abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3
// The reference copies prediction, mask and ground truth to the host and runs numpy there; here the batch stays on
// the device and only the seven numbers leave it.  Pipeline (all on the caller's stream, no host synchronisation):
//   1. resize (Chainer's align-corners bilinear, float64 coordinates / weights as in prep.cu) + clip -> scratch;
//      histogram of the upper 16 bits of the masked ground-truth and prediction bit patterns (positive floats order
//      like their bit patterns), masked count
//   2. one CTA scans the histograms for the bins holding the two middle ranks (n-1)/2 and n/2 (np.median)
//   3. histogram of the lower 16 bits inside those bins; 4. one CTA reads off the exact middle values ->
//      medians -> scale;  5. metric sums in fp64;  6. the seven numbers
// The medians are exact (radix select, no approximation), so the scale factor is bit-identical to numpy's.
#include "common.cuh"
#include "kernels.h"

namespace {

struct EvalState {
  unsigned long long n;          // masked pixels
  unsigned bin[2][2];            // [gt|pred][lower|upper middle rank] -> upper-16-bit bin
  unsigned long long rank[2][2]; // rank inside that bin
  float scale;
  float med[2];
  double sums[7];
};

struct EvalLayout {
  size_t off_pred, off_hi, off_lo, off_state, total;
};

inline EvalLayout eval_layout(int B, int Hg, int Wg) {
  EvalLayout L;
  size_t off = 0;
  L.off_pred = off; off = sfm_align_up(off + (size_t)B * Hg * Wg * sizeof(float), 256);
  L.off_hi = off; off = sfm_align_up(off + 2 * 65536 * sizeof(unsigned), 256);
  L.off_lo = off; off = sfm_align_up(off + 4 * 65536 * sizeof(unsigned), 256);
  L.off_state = off; off = sfm_align_up(off + sizeof(EvalState), 256);
  L.total = off;
  return L;
}

__global__ void __launch_bounds__(256) eval_resize_hist_kernel(const float* __restrict__ pred_in, const float* __restrict__ gt,
                                                               const uint8_t* __restrict__ mask, float* __restrict__ pred_out,
                                                               unsigned* __restrict__ hist_hi, EvalState* st, int B, int h, int w,
                                                               int Hg, int Wg, float lo, float hi) {
  const long long total = (long long)B * Hg * Wg;
  const double stepx = (Wg > 1) ? __ddiv_rn((double)(w - 1), (double)(Wg - 1)) : 0.0;
  const double stepy = (Hg > 1) ? __ddiv_rn((double)(h - 1), (double)(Hg - 1)) : 0.0;
  unsigned cnt = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / ((long long)Hg * Wg));
    const int r = (int)(i - (long long)b * Hg * Wg);
    const int y = r / Wg, x = r - y * Wg;
    const double u = (x == Wg - 1 && Wg > 1) ? (double)(w - 1) : __dmul_rn((double)x, stepx);
    const double v = (y == Hg - 1 && Hg > 1) ? (double)(h - 1) : __dmul_rn((double)y, stepy);
    const int u0 = min(max((int)floor(u), 0), w - 2), v0 = min(max((int)floor(v), 0), h - 2);
    const double ua = __dsub_rn((double)(u0 + 1), u), ub = __dsub_rn(u, (double)u0);
    const double va = __dsub_rn((double)(v0 + 1), v), vb = __dsub_rn(v, (double)v0);
    const float w1 = (float)__dmul_rn(va, ua), w2 = (float)__dmul_rn(va, ub);
    const float w3 = (float)__dmul_rn(vb, ua), w4 = (float)__dmul_rn(vb, ub);
    const float* __restrict__ t = pred_in + (size_t)b * h * w + (size_t)v0 * w + u0;
    float p = sfm_blend(w1, w2, w3, w4, __ldg(t), __ldg(t + 1), __ldg(t + w), __ldg(t + w + 1));
    p = fminf(fmaxf(p, lo), hi);                                     // F.clip
    pred_out[i] = p;
    if (mask[i]) {
      ++cnt;
      atomicAdd(hist_hi + (__float_as_uint(__ldg(gt + i)) >> 16), 1u);
      atomicAdd(hist_hi + 65536 + (__float_as_uint(p) >> 16), 1u);
    }
  }
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&st->n, (unsigned long long)cnt);
}

// One CTA of 1024 threads: for each of the (up to 4) histograms locate the bin holding a rank and the rank inside it.
// hist: 65536 bins; thread t owns bins [64 t, 64 t + 64).
__device__ void locate(const unsigned* __restrict__ hist, unsigned long long rank, unsigned& bin_out, unsigned long long& rest_out,
                       unsigned long long* s_scan) {
  const int t = threadIdx.x;
  unsigned long long local = 0;
  for (int k = 0; k < 64; ++k) local += hist[t * 64 + k];
  s_scan[t] = local;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {            // inclusive Hillis-Steele scan
    const unsigned long long v = (t >= off) ? s_scan[t - off] : 0ull;
    __syncthreads();
    s_scan[t] += v;
    __syncthreads();
  }
  const unsigned long long before = s_scan[t] - local;
  if (rank >= before && rank < before + local) {
    unsigned long long acc = before;
    for (int k = 0; k < 64; ++k) {
      const unsigned c = hist[t * 64 + k];
      if (rank < acc + c) { bin_out = (unsigned)(t * 64 + k); rest_out = rank - acc; break; }
      acc += c;
    }
  }
  __syncthreads();
}

__global__ void __launch_bounds__(1024) eval_select_hi_kernel(const unsigned* __restrict__ hist_hi, EvalState* st) {
  __shared__ unsigned long long s_scan[1024];
  const unsigned long long n = st->n;
  if (n == 0) return;
  for (int a = 0; a < 2; ++a)
    for (int m = 0; m < 2; ++m) locate(hist_hi + a * 65536, m == 0 ? (n - 1) / 2 : n / 2, st->bin[a][m], st->rank[a][m], s_scan);
}

__global__ void __launch_bounds__(256) eval_hist_lo_kernel(const float* __restrict__ gt, const float* __restrict__ pred,
                                                           const uint8_t* __restrict__ mask, unsigned* __restrict__ hist_lo,
                                                           const EvalState* __restrict__ st, long long total) {
  const unsigned b00 = st->bin[0][0], b01 = st->bin[0][1], b10 = st->bin[1][0], b11 = st->bin[1][1];
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (!mask[i]) continue;
    const unsigned g = __float_as_uint(__ldg(gt + i)), p = __float_as_uint(__ldg(pred + i));
    if ((g >> 16) == b00) atomicAdd(hist_lo + 0 * 65536 + (g & 0xffffu), 1u);
    if ((g >> 16) == b01) atomicAdd(hist_lo + 1 * 65536 + (g & 0xffffu), 1u);
    if ((p >> 16) == b10) atomicAdd(hist_lo + 2 * 65536 + (p & 0xffffu), 1u);
    if ((p >> 16) == b11) atomicAdd(hist_lo + 3 * 65536 + (p & 0xffffu), 1u);
  }
}

__global__ void __launch_bounds__(1024) eval_select_lo_kernel(const unsigned* __restrict__ hist_lo, EvalState* st) {
  __shared__ unsigned long long s_scan[1024];
  __shared__ unsigned s_bin[2][2];
  __shared__ unsigned long long s_rest[2][2];
  if (st->n == 0) return;
  for (int a = 0; a < 2; ++a)
    for (int m = 0; m < 2; ++m) locate(hist_lo + (a * 2 + m) * 65536, st->rank[a][m], s_bin[a][m], s_rest[a][m], s_scan);
  if (threadIdx.x == 0) {
    for (int a = 0; a < 2; ++a) {
      const float lo = __uint_as_float((st->bin[a][0] << 16) | s_bin[a][0]);
      const float hi = __uint_as_float((st->bin[a][1] << 16) | s_bin[a][1]);
      st->med[a] = __fmul_rn(__fadd_rn(lo, hi), 0.5f);            // np.median: mean of the two middle elements
    }
    st->scale = __fdiv_rn(st->med[0], st->med[1]);                // evaluate.py:101
  }
}

__global__ void __launch_bounds__(256) eval_metrics_kernel(const float* __restrict__ gt, const float* __restrict__ pred,
                                                           const uint8_t* __restrict__ mask, EvalState* st, long long total) {
  const float scale = st->scale;
  double s[7] = {0, 0, 0, 0, 0, 0, 0};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    if (!mask[i]) continue;
    const float g = __ldg(gt + i), p = __fmul_rn(__ldg(pred + i), scale);          // pred_depth *= scale_factor
    const float th = fmaxf(__fdiv_rn(g, p), __fdiv_rn(p, g));                      // depth_util.py:7
    const float d = __fsub_rn(g, p), d2 = __fmul_rn(d, d);
    const float dl = __fsub_rn(logf(g), logf(p));
    s[0] += (double)__fdiv_rn(fabsf(d), g);        // abs_rel
    s[1] += (double)__fdiv_rn(d2, g);              // sq_rel
    s[2] += (double)d2;                            // rmse^2
    s[3] += (double)__fmul_rn(dl, dl);             // rmse_log^2
    s[4] += th < 1.25f ? 1.0 : 0.0;
    s[5] += th < 1.5625f ? 1.0 : 0.0;
    s[6] += th < 1.953125f ? 1.0 : 0.0;
  }
  __shared__ double part[8][7];
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    double v = s[k];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 7) {
    double v = 0;
    for (int k = 0; k < 8; ++k) v += part[k][threadIdx.x];
    if (v != 0.0) atomicAdd(&st->sums[threadIdx.x], v);
  }
}

__global__ void eval_finish_kernel(const EvalState* __restrict__ st, float* __restrict__ out) {
  const double n = (double)st->n;
  // order of depth_util.py:22: abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3
  out[0] = (float)(st->sums[0] / n);
  out[1] = (float)(st->sums[1] / n);
  out[2] = (float)sqrt(st->sums[2] / n);
  out[3] = (float)sqrt(st->sums[3] / n);
  out[4] = (float)(st->sums[4] / n);
  out[5] = (float)(st->sums[5] / n);
  out[6] = (float)(st->sums[6] / n);
  out[7] = st->scale;
}

}  // namespace

size_t sfm_eval_scratch_bytes_impl(int B, int Hg, int Wg) { return eval_layout(B, Hg, Wg).total; }

int sfm_launch_eval_depth(int B, int h, int w, int Hg, int Wg, const float* pred, const float* gt, const uint8_t* mask, float lo,
                          float hi, float* out, void* scratch, cudaStream_t stream) {
  const EvalLayout L = eval_layout(B, Hg, Wg);
  char* ws = (char*)scratch;
  float* pred_full = (float*)(ws + L.off_pred);
  unsigned* hist_hi = (unsigned*)(ws + L.off_hi);
  unsigned* hist_lo = (unsigned*)(ws + L.off_lo);
  EvalState* st = (EvalState*)(ws + L.off_state);
  SFM_CUDA_CHECK(cudaMemsetAsync(ws + L.off_hi, 0, L.total - L.off_hi, stream));
  const long long total = (long long)B * Hg * Wg;
  const int blocks = (int)((total + 255) / 256 > SFM_REF_SMS * 8 ? SFM_REF_SMS * 8 : (total + 255) / 256);
  eval_resize_hist_kernel<<<blocks, 256, 0, stream>>>(pred, gt, mask, pred_full, hist_hi, st, B, h, w, Hg, Wg, lo, hi);
  eval_select_hi_kernel<<<1, 1024, 0, stream>>>(hist_hi, st);
  eval_hist_lo_kernel<<<blocks, 256, 0, stream>>>(gt, pred_full, mask, hist_lo, st, total);
  eval_select_lo_kernel<<<1, 1024, 0, stream>>>(hist_lo, st);
  eval_metrics_kernel<<<blocks, 256, 0, stream>>>(gt, pred_full, mask, st, total);
  eval_finish_kernel<<<1, 1, 0, stream>>>(st, out);
  SFM_CUDA_CHECK(cudaGetLastError());
  return 0;
}
