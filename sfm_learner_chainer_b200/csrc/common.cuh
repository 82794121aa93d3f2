// common.cuh -- shared host/device helpers of libsfmloss (sm_100a).
//
// The coordinate chain below is the "spec arithmetic" shared with oracle/sfm_oracle.py: every
// operation is individually rounded fp32 (__fmul_rn/__fadd_rn/__fdiv_rn are never contracted into
// FMAs), so floor indices and in-bounds masks are bit-identical to the numpy restatement of
// models/transform.py:94-133 and F.spatial_transformer_sampler (transform.py:189).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>

#include "sfmloss.h"

#define SFM_PI_F 3.14159274101257324f  // float(np.pi): F.clip(r, -np.pi, np.pi) on an fp32 array, transform.py:23

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
void sfm_set_error(const char* fmt, ...);
#define SFM_CUDA_CHECK(expr)                                                                   \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      sfm_set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return (int)_e;                                                                          \
    }                                                                                          \
  } while (0)

// ---------------------------------------------------------------------------------------------
// workspace layout (host + device agree through this struct)
// ---------------------------------------------------------------------------------------------
struct SfmWsLayout {
  // Image pyramid, scales >= 1 only: planar fp32 exactly like the caller's tensors ([img][3][h][w], no padding).
  // Scale 0 is the identity of F.resize_images and is read straight from the caller's tgt / src tensors.
  size_t off_tgt[SFM_MAX_SCALES];  // float [B][3][h][w]
  size_t off_src[SFM_MAX_SCALES];  // float [B*S][3][h][w]
  size_t off_proj;                 // float  [B][S][ns][12]  3x4 projection K4.T
  size_t off_kinv;                 // float  [B][ns][9]
  size_t off_acc;                  // double [4 + B*S*ns*12] loss sums (pixel, smooth, exp, ssim) + dL/dP per scale
  size_t off_posevec;              // float  [B][S][6]   6-DoF vectors reduced from the raw `poseout` map (raw_pose_hw > 0)
  size_t off_smpart;               // float  [tasks / 8] loss partials of the smoothness CTAs of the prologue kernel
  size_t acc_doubles;
  size_t total;
};

#ifdef __CUDACC__
#define SFM_HD __host__ __device__
#else
#define SFM_HD
#endif

static inline size_t sfm_align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// SM count of a B200.  The fixed reference of the decisions that must not depend on the device the code runs on (the
// workspace layout) and of the ones tuned for it without a query (the prologue's band rule, grid caps).
constexpr int SFM_REF_SMS = 148;

// Decomposition of the second-order smoothness term into warp tasks (strips of SFM_SMOOTH_IW interior columns x hseg
// rows of every (snippet, scale)); shared by the planner (plan.cu) and the workspace layout (one loss-partial slot
// per 8 tasks).  Segment height: enough warps to cover the chip a few times, few enough that the 4 halo rows stay cheap.
#define SFM_SMOOTH_IW 28
static inline int sfm_smooth_plan(int B, int ns, int H, int W, int* hseg_out) {
  int hseg = 64;
  long long n = 0;
  for (;;) {
    n = 0;
    for (int s = 0; s < ns; ++s) n += (long long)B * (((W >> s) + SFM_SMOOTH_IW - 1) / SFM_SMOOTH_IW) * (((H >> s) + hseg - 1) / hseg);
    if (n >= SFM_REF_SMS * 4 * 8 || hseg <= 8) break;
    hseg >>= 1;
  }
  if (hseg_out) *hseg_out = hseg;
  return (int)n;
}

static inline void sfm_ws_layout(const SfmDesc* d, SfmWsLayout* L) {
  size_t off = 0;
  for (int s = 0; s < SFM_MAX_SCALES; ++s) {
    L->off_tgt[s] = L->off_src[s] = 0;
  }
  for (int s = 1; s < d->n_scales; ++s) {
    const int h = d->H >> s, w = d->W >> s;
    L->off_tgt[s] = off;
    off = sfm_align_up(off + (size_t)d->B * 3 * h * w * sizeof(float), 256);
    L->off_src[s] = off;
    off = sfm_align_up(off + (size_t)d->B * d->S * 3 * h * w * sizeof(float), 256);
  }
  L->off_proj = off;
  off = sfm_align_up(off + (size_t)d->B * d->S * d->n_scales * 12 * sizeof(float), 256);
  L->off_kinv = off;
  off = sfm_align_up(off + (size_t)d->B * d->n_scales * 9 * sizeof(float), 256);
  L->acc_doubles = 4 + (size_t)d->B * d->S * d->n_scales * 12;
  L->off_acc = off;
  off += L->acc_doubles * sizeof(double);
  off = sfm_align_up(off, 256);
  L->off_posevec = off;
  off = sfm_align_up(off + (size_t)d->B * d->S * 6 * sizeof(float), 256);
  L->off_smpart = off;
  off = sfm_align_up(off + (size_t)((sfm_smooth_plan(d->B, d->n_scales, d->H, d->W, nullptr) + 7) / 8) * sizeof(float), 256);
  L->total = off;
}

int sfm_validate_desc(const SfmDesc* d);

// ---------------------------------------------------------------------------------------------
// device math shared by the kernels
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// C = A.B (3x3, row major), canonical order ((a0*b0 + a1*b1) + a2*b2), no FMA (oracle `_mm`).
__device__ __forceinline__ void sfm_mm3(const float* A, const float* B, float* C) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c)
      C[r * 3 + c] = __fadd_rn(__fadd_rn(__fmul_rn(A[r * 3 + 0], B[0 * 3 + c]), __fmul_rn(A[r * 3 + 1], B[1 * 3 + c])),
                               __fmul_rn(A[r * 3 + 2], B[2 * 3 + c]));
}

// euler angles -> sin/cos, clipped to [-pi, pi] (transform.py:23-25); evaluated in fp64, rounded to fp32.
__device__ __forceinline__ void sfm_euler_sincos(const float* r, float* c, float* s) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float rc = fminf(fmaxf(r[k], -SFM_PI_F), SFM_PI_F);
    double sd, cd;
    sincos((double)rc, &sd, &cd);
    c[k] = (float)cd;
    s[k] = (float)sd;
  }
}

__device__ __forceinline__ void sfm_rot_mats(const float* c, const float* s, float* X, float* Y, float* Z) {
  Z[0] = c[2]; Z[1] = -s[2]; Z[2] = 0.f; Z[3] = s[2]; Z[4] = c[2]; Z[5] = 0.f; Z[6] = 0.f; Z[7] = 0.f; Z[8] = 1.f;
  Y[0] = c[1]; Y[1] = 0.f; Y[2] = s[1]; Y[3] = 0.f; Y[4] = 1.f; Y[5] = 0.f; Y[6] = -s[1]; Y[7] = 0.f; Y[8] = c[1];
  X[0] = 1.f; X[1] = 0.f; X[2] = 0.f; X[3] = 0.f; X[4] = c[0]; X[5] = -s[0]; X[6] = 0.f; X[7] = s[0]; X[8] = c[0];
}

// proj (3x4) = K . [R | t]   with R = (Rx.Ry).Rz    (transform.py:27-39, 52-58, 86-88)
__device__ __forceinline__ void sfm_build_proj(const float* pose, const float* K, float* P) {
  float c[3], s[3], X[9], Y[9], Z[9], XY[9], R[9];
  sfm_euler_sincos(pose, c, s);
  sfm_rot_mats(c, s, X, Y, Z);
  sfm_mm3(X, Y, XY);
  sfm_mm3(XY, Z, R);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float t0 = (j < 3) ? R[0 * 3 + j] : pose[3];
      float t1 = (j < 3) ? R[1 * 3 + j] : pose[4];
      float t2 = (j < 3) ? R[2 * 3 + j] : pose[5];
      P[r * 4 + j] =
          __fadd_rn(__fadd_rn(__fmul_rn(K[r * 3 + 0], t0), __fmul_rn(K[r * 3 + 1], t1)), __fmul_rn(K[r * 3 + 2], t2));
    }
  }
}

// F.batch_inv(K) (transform.py:105): closed-form adjugate in fp64, fixed order, rounded to fp32
// (oracle `batch_inv3`).
__device__ __forceinline__ void sfm_inv3(const float* K, float* inv) {
  const double a = K[0], b = K[1], c = K[2], d = K[3], e = K[4], f = K[5], g = K[6], h = K[7], i = K[8];
  const double A = __dsub_rn(__dmul_rn(e, i), __dmul_rn(f, h));
  const double Bc = -__dsub_rn(__dmul_rn(d, i), __dmul_rn(f, g));
  const double C = __dsub_rn(__dmul_rn(d, h), __dmul_rn(e, g));
  const double det = __dadd_rn(__dadd_rn(__dmul_rn(a, A), __dmul_rn(b, Bc)), __dmul_rn(c, C));
  inv[0] = (float)__ddiv_rn(A, det);
  inv[1] = (float)__ddiv_rn(-__dsub_rn(__dmul_rn(b, i), __dmul_rn(c, h)), det);
  inv[2] = (float)__ddiv_rn(__dsub_rn(__dmul_rn(b, f), __dmul_rn(c, e)), det);
  inv[3] = (float)__ddiv_rn(Bc, det);
  inv[4] = (float)__ddiv_rn(__dsub_rn(__dmul_rn(a, i), __dmul_rn(c, g)), det);
  inv[5] = (float)__ddiv_rn(-__dsub_rn(__dmul_rn(a, f), __dmul_rn(c, d)), det);
  inv[6] = (float)__ddiv_rn(C, det);
  inv[7] = (float)__ddiv_rn(-__dsub_rn(__dmul_rn(a, h), __dmul_rn(b, g)), det);
  inv[8] = (float)__ddiv_rn(__dsub_rn(__dmul_rn(a, e), __dmul_rn(b, d)), det);
}

// ray = Kinv.(x, y, 1):  r_k = (k_k0*x + k_k1*y) + k_k2      (pixel2cam, transform.py:105-106)
__device__ __forceinline__ void sfm_ray(const float* kinv, float xf, float yf, float& rx, float& ry, float& rz) {
  rx = __fadd_rn(__fadd_rn(__fmul_rn(kinv[0], xf), __fmul_rn(kinv[1], yf)), kinv[2]);
  ry = __fadd_rn(__fadd_rn(__fmul_rn(kinv[3], xf), __fmul_rn(kinv[4], yf)), kinv[5]);
  rz = __fadd_rn(__fadd_rn(__fmul_rn(kinv[6], xf), __fmul_rn(kinv[7], yf)), kinv[8]);
}

// ---- producer-side fusions (SfmDesc.raw_disp_scales / raw_pose_hw)
// disp = DISP_SCALING * F.sigmoid(x) + MIN_DISP (disp_net.py:7-8,104).  Chainer's sigmoid is
// tanh(x * 0.5) * 0.5 + 0.5 (CPU: numpy.tanh, GPU: the same expression in an elementwise CUDA kernel, i.e.
// this tanhf); the scaling and the offset are separate elementwise ops, each rounded.  dact = d disp / d x
// = 10 y (1 - y)  (Sigmoid.backward: gy * y * (1 - y)).
__device__ __forceinline__ float sfm_disp_act(float x, float& dact) {
  const float y = __fadd_rn(__fmul_rn(tanhf(__fmul_rn(x, 0.5f)), 0.5f), 0.5f);
  dact = 10.f * y * (1.f - y);
  return __fadd_rn(__fmul_rn(10.f, y), 0.01f);
}
// fp32 sum of n <= 128 values in numpy's pairwise order (numpy/core/src/umath/loops_utils.h.src, pairwise_sum:
// sequential for n < 8, otherwise eight running partial sums combined as ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) and
// the tail added sequentially) -- the order F.mean(h, (2, 3)) uses on the contiguous (h', w') block of one
// channel (pose_net.py:52).
__device__ __forceinline__ float sfm_np_sum(const float* __restrict__ a, int n) {
  if (n < 8) {
    float r = 0.f;                    // numpy seeds the reduction with the first element; 0 + a0 == a0 (also -0: sign irrelevant here)
    for (int i = 0; i < n; ++i) r = __fadd_rn(r, a[i]);
    return r;
  }
  float r[8];
  for (int k = 0; k < 8; ++k) r[k] = a[k];
  int i = 8;
  for (; i < n - (n % 8); i += 8)
    for (int k = 0; k < 8; ++k) r[k] = __fadd_rn(r[k], a[i + k]);
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])), __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __fadd_rn(res, a[i]);
  return res;
}
// pose component = 0.01 * mean(x[0..n))   (pose_net.py:52: float32(0.01) * (sum / n))
__device__ __forceinline__ float sfm_pose_component(const float* __restrict__ x, int n) {
  return __fmul_rn(0.01f, __fdiv_rn(sfm_np_sum(x, n), (float)n));
}

// Everything the sampler needs about one (target pixel, source) pair.
struct SfmCoord {
  float q0, q1, z;   // unnormalised projection (cam2pixel, transform.py:122-123)
  float fx, fy;      // 1 inside, 2 outside: the x2 rule's constant factor on the grid gradient (:128-131)
  int u0, v0;        // floor indices (integer work: bit-exact vs the oracle)
  float wa, wb, wc, wd;  // u1-u, u-u0, v1-v, v-v0
  bool inb;          // strictly inside (-1,1)^2
  bool v00, v01, v10, v11;  // tap validity under zero padding
  bool any;
};

// cam2pixel (transform.py:111-133) followed by the sampler's coordinate mapping
// u = ((xn+1)*(w-1))/2 (F.spatial_transformer_sampler, align corners, zero padding).
__device__ __forceinline__ void sfm_project(const float* P, float X, float Y, float Z, int w, int h, float hw,
                                            float hh, SfmCoord& c) {
  const float q0 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P[0], X), __fmul_rn(P[1], Y)), __fmul_rn(P[2], Z)), P[3]);
  const float q1 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P[4], X), __fmul_rn(P[5], Y)), __fmul_rn(P[6], Z)), P[7]);
  const float q2 = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(P[8], X), __fmul_rn(P[9], Y)), __fmul_rn(P[10], Z)), P[11]);
  const float z = __fadd_rn(q2, 1e-10f);
  float xn = __fsub_rn(__fdiv_rn(__fdiv_rn(q0, z), hw), 1.f);
  float yn = __fsub_rn(__fdiv_rn(__fdiv_rn(q1, z), hh), 1.f);
  const bool inx = (xn > -1.f) && (xn < 1.f);
  const bool iny = (yn > -1.f) && (yn < 1.f);
  if (!inx) xn = __fmul_rn(xn, 2.f);
  if (!iny) yn = __fmul_rn(yn, 2.f);
  const float u = __fmul_rn(__fmul_rn(__fadd_rn(xn, 1.f), (float)(w - 1)), 0.5f);
  const float v = __fmul_rn(__fmul_rn(__fadd_rn(yn, 1.f), (float)(h - 1)), 0.5f);
  float u0f = floorf(u), v0f = floorf(v);
  // clamp before the int conversion so inf/NaN/huge stay defined: anything outside [-2, n+1] has no valid tap
  const float u0c = (u0f >= -2.f) ? fminf(u0f, (float)(w + 1)) : -2.f;
  const float v0c = (v0f >= -2.f) ? fminf(v0f, (float)(h + 1)) : -2.f;
  c.u0 = (int)u0c;
  c.v0 = (int)v0c;
  c.wa = __fsub_rn(__fadd_rn(u0f, 1.f), u);
  c.wb = __fsub_rn(u, u0f);
  c.wc = __fsub_rn(__fadd_rn(v0f, 1.f), v);
  c.wd = __fsub_rn(v, v0f);
  const bool vu0 = (c.u0 >= 0) && (c.u0 <= w - 1), vu1 = (c.u0 + 1 >= 0) && (c.u0 + 1 <= w - 1);
  const bool vv0 = (c.v0 >= 0) && (c.v0 <= h - 1), vv1 = (c.v0 + 1 >= 0) && (c.v0 + 1 <= h - 1);
  c.v00 = vv0 && vu0; c.v01 = vv0 && vu1; c.v10 = vv1 && vu0; c.v11 = vv1 && vu1;
  c.any = (vv0 || vv1) && (vu0 || vu1);
  c.q0 = q0; c.q1 = q1; c.z = z;
  c.fx = inx ? 1.f : 2.f;
  c.fy = iny ? 1.f : 2.f;
  c.inb = inx && iny;
}

// P_c = ((w1*I00 + w2*I01) + w3*I10) + w4*I11, products and sums individually rounded.
__device__ __forceinline__ float sfm_blend(float w1, float w2, float w3, float w4, float a, float b, float c, float d) {
  return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(w1, a), __fmul_rn(w2, b)), __fmul_rn(w3, c)), __fmul_rn(w4, d));
}

// sign(v) * c for either sign of c, 0 when v == 0
__device__ __forceinline__ float sfm_sign_times(float v, float c) {
  const float t = __int_as_float((__float_as_int(v) & 0x80000000) ^ __float_as_int(c));
  return (v == 0.f) ? 0.f : t;
}

__device__ __forceinline__ float sfm_warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// dL/dpose (6) from dL/dT (3x4, fp64) through T = [R|t], R = (Rx.Ry).Rz   (SURVEY A.6)
__device__ __forceinline__ void sfm_pose_backward_cs(const float* pose, const float* cf, const float* sf, const double* dT,
                                                     float* gpose);
__device__ __forceinline__ void sfm_pose_backward(const float* pose, const double* dT, float* gpose) {
  float cf[3], sf[3];
  sfm_euler_sincos(pose, cf, sf);
  sfm_pose_backward_cs(pose, cf, sf, dT, gpose);
}
// same with the sin/cos of the clipped angles supplied by the caller
__device__ __forceinline__ void sfm_pose_backward_cs(const float* pose, const float* cf, const float* sf, const double* dT,
                                                     float* gpose) {
  float Xf[9], Yf[9], Zf[9];
  sfm_rot_mats(cf, sf, Xf, Yf, Zf);
  double X[9], Y[9], Z[9], A[9], GR[9], GA[9], GRz[9], GRx[9], GRy[9];
  for (int k = 0; k < 9; ++k) { X[k] = Xf[k]; Y[k] = Yf[k]; Z[k] = Zf[k]; }
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      GR[r * 3 + c] = dT[r * 4 + c];
      double a = 0;
      for (int k = 0; k < 3; ++k) a += X[r * 3 + k] * Y[k * 3 + c];
      A[r * 3 + c] = a;
    }
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      double gz = 0, ga = 0;
      for (int k = 0; k < 3; ++k) {
        gz += A[k * 3 + r] * GR[k * 3 + c];   // A^T . G_R
        ga += GR[r * 3 + k] * Z[c * 3 + k];   // G_R . Rz^T
      }
      GRz[r * 3 + c] = gz;
      GA[r * 3 + c] = ga;
    }
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) {
      double gx = 0, gy = 0;
      for (int k = 0; k < 3; ++k) {
        gx += GA[r * 3 + k] * Y[c * 3 + k];   // G_A . Ry^T
        gy += X[k * 3 + r] * GA[k * 3 + c];   // Rx^T . G_A
      }
      GRx[r * 3 + c] = gx;
      GRy[r * 3 + c] = gy;
    }
  const double c0 = cf[0], s0 = sf[0], c1 = cf[1], s1 = sf[1], c2 = cf[2], s2 = sf[2];
  double g0 = GRx[4] * (-s0) + GRx[5] * (-c0) + GRx[7] * c0 + GRx[8] * (-s0);
  double g1 = GRy[0] * (-s1) + GRy[2] * c1 + GRy[6] * (-c1) + GRy[8] * (-s1);
  double g2 = GRz[0] * (-s2) + GRz[1] * (-c2) + GRz[3] * c2 + GRz[4] * (-s2);
  // F.clip backward: gradient passes where -pi <= r <= pi
  gpose[0] = (pose[0] >= -SFM_PI_F && pose[0] <= SFM_PI_F) ? (float)g0 : 0.f;
  gpose[1] = (pose[1] >= -SFM_PI_F && pose[1] <= SFM_PI_F) ? (float)g1 : 0.f;
  gpose[2] = (pose[2] >= -SFM_PI_F && pose[2] <= SFM_PI_F) ? (float)g2 : 0.f;
  gpose[3] = (float)dT[3];
  gpose[4] = (float)dT[7];
  gpose[5] = (float)dT[11];
}

#endif  // __CUDACC__
