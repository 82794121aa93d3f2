"""CPU oracle for the SfM-Learner view-synthesis loss path.

TEST INFRASTRUCTURE -- NOT PRODUCT CODE.  Only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl
reference`` legs may import this module, and only as the checker / the timed
CPU baseline.  The product path (``sfm_learner_chainer_b200``) never imports it.

What this is
------------
A numpy restatement of the reference's algorithm for the hot path, written
function by function after the reference (citations are relative to
``/root/reference``):

* ``models/transform.py:11-40``   euler2mat
* ``models/transform.py:43-59``   pose_vec2mat
* ``models/transform.py:64-91``   proj_tgt_to_src
* ``models/transform.py:94-109``  pixel2cam
* ``models/transform.py:111-133`` cam2pixel
* ``models/transform.py:137-154`` generate_2dmeshgrid
* ``models/transform.py:156-193`` projective_inverse_warp
* ``models/spational_transformer_sampler_interp.py:32-149`` (secondary sampler)
* ``models/base_model.py:48-124`` SFMLearner.__call__ loss loop
* ``models/base_model.py:126-142`` compute_ssim
* ``models/base_model.py:157-167`` compute_exp_reg_loss
* ``models/base_model.py:169-185`` compute_smooth_loss
* ``models/base_model.py:144-155`` compute_disp_smooth (edge-aware alternative, commented out at :78-80)
* ``models/disp_net.py:7-8,104``  disparity activation  (seam, SURVEY 8(f) rank 1)
* ``models/pose_net.py:52-53``    pose scaling / spatial mean (seam)

The arithmetic of the reference lives in a third-party dependency that is NOT
under ``/root/reference`` and NOT installable here: ``chainer==4.0.0b1`` /
``cupy==4.0.0b1`` (``requirements.txt:1,3``).  The Chainer ops the path calls
(``F.spatial_transformer_sampler``, ``F.resize_images``,
``F.average_pooling_2d``, ``F.batch_matmul``, ``F.batch_inv``, ``F.sigmoid``,
``F.sigmoid_cross_entropy``, ``F.clip`` ...) are restated here from their
published algorithm.

Pinning status
--------------
The reference ships no tests, golden vectors or fixtures, and Chainer cannot be
imported, so the *third-party op semantics* are "parity unpinned".  What IS
pinned: the reference's own source files (``models/transform.py``,
``models/base_model.py``, ``models/spational_transformer_sampler_interp.py``)
are executed UNMODIFIED under ``oracle/chainer_shim`` (a torch-CPU-backed stand
in for the absent Chainer) by ``tests/golden/make_golden.py``; the fixtures it
wrote are compared with this oracle in ``tests/test_oracle_golden.py``.

Canonical ("spec") arithmetic
-----------------------------
Bit-exact integer work (floor indices, in-bounds masks) between this oracle and
the CUDA kernels needs one agreed sequence of individually rounded fp32
operations for the coordinate chain; numpy ufuncs round every operation
separately (no FMA contraction) and the kernels use ``__fmul_rn/__fadd_rn/
__fdiv_rn``.  The sequence is written out in `pixel2cam`, `cam2pixel` and
`spatial_transformer_sampler` below.  Small matrix products use `_mm`
(left-to-right sum of individually rounded products) instead of BLAS.
sin/cos and the 3x3 inverse are evaluated in float64 and rounded to the
working dtype.

Everything is dtype generic: run with float32 for the canonical restatement or
float64 for a "true math" cross-check.
"""
import math

import numpy as np

N_SCALES = 4
SSIM_C1 = 0.01 ** 2
SSIM_C2 = 0.03 ** 2


# --------------------------------------------------------------------------
# small helpers
# --------------------------------------------------------------------------
def _mm(A, B):
    """Batched small matmul, canonical order: ((a0*b0 + a1*b1) + a2*b2) + ...
    Replaces F.batch_matmul (transform.py:39,88,105,122)."""
    k = A.shape[-1]
    acc = A[..., :, 0, None] * B[..., None, 0, :]
    for j in range(1, k):
        acc = acc + A[..., :, j, None] * B[..., None, j, :]
    return acc


def _sigmoid(x):
    """Chainer's F.sigmoid CPU formula: tanh(x/2)/2 + 1/2 (base_model.py:107)."""
    half = x.dtype.type(0.5)
    return np.tanh(x * half) * half + half


def _softplus_neg(x):
    """sigmoid_cross_entropy(x, t=1, reduce='no') = softplus(-x)
    = -(x*(1 - (x>=0)) - log1p(exp(-|x|)))   (base_model.py:157-167)."""
    return -(x * (1 - (x >= 0)).astype(x.dtype) - np.log1p(np.exp(-np.abs(x))))


def scale_shape(H, W, s):
    return H // (2 ** s), W // (2 ** s)


# --------------------------------------------------------------------------
# geometry  (models/transform.py)
# --------------------------------------------------------------------------
def euler_sincos(r):
    """clip to [-pi, pi] (transform.py:23) and sin/cos (transform.py:24-25).
    Canonical: evaluated in float64, rounded to the working dtype."""
    dt = r.dtype
    lo, hi = dt.type(-np.pi), dt.type(np.pi)
    rc = np.clip(r, lo, hi)
    c = np.cos(rc.astype(np.float64)).astype(dt)
    s = np.sin(rc.astype(np.float64)).astype(dt)
    return rc, c, s


def _rot_mats(c, s):
    N = c.shape[0]
    dt = c.dtype
    z = np.zeros(N, dt)
    o = np.ones(N, dt)
    zmat = np.stack([c[:, 2], -s[:, 2], z,
                     s[:, 2], c[:, 2], z,
                     z, z, o], axis=1).reshape(N, 3, 3)
    ymat = np.stack([c[:, 1], z, s[:, 1],
                     z, o, z,
                     -s[:, 1], z, c[:, 1]], axis=1).reshape(N, 3, 3)
    xmat = np.stack([o, z, z,
                     z, c[:, 0], -s[:, 0],
                     z, s[:, 0], c[:, 0]], axis=1).reshape(N, 3, 3)
    return xmat, ymat, zmat


def euler2mat(r):
    """transform.py:11-40.  R = (Rx . Ry) . Rz, association as written (:39)."""
    _, c, s = euler_sincos(r)
    xmat, ymat, zmat = _rot_mats(c, s)
    return _mm(_mm(xmat, ymat), zmat)


def pose_vec2mat(vec):
    """transform.py:43-59.  vec = [rx, ry, rz, tx, ty, tz] -> (N,4,4)."""
    N = vec.shape[0]
    dt = vec.dtype
    R = euler2mat(vec[:, :3])
    T = np.zeros((N, 4, 4), dt)
    T[:, :3, :3] = R
    T[:, :3, 3] = vec[:, 3:]
    T[:, 3, 3] = 1
    return T


def proj_tgt_to_src(vec, K):
    """transform.py:64-91.  P = K4 . T, K4 = [[K,0],[0 0 0 1]] -> (N,4,4)."""
    N = vec.shape[0]
    dt = vec.dtype
    K4 = np.zeros((N, 4, 4), dt)
    K4[:, :3, :3] = K
    K4[:, 3, 3] = 1
    return _mm(K4, pose_vec2mat(vec))


def batch_inv3(K):
    """F.batch_inv(K) (transform.py:105).  Canonical: closed-form adjugate
    evaluated in float64 in the fixed order below, rounded to K.dtype."""
    K64 = K.astype(np.float64)
    a, b, c = K64[:, 0, 0], K64[:, 0, 1], K64[:, 0, 2]
    d, e, f = K64[:, 1, 0], K64[:, 1, 1], K64[:, 1, 2]
    g, h, i = K64[:, 2, 0], K64[:, 2, 1], K64[:, 2, 2]
    A = e * i - f * h
    Bc = -(d * i - f * g)
    C = d * h - e * g
    det = (a * A + b * Bc) + c * C
    inv = np.empty_like(K64)
    inv[:, 0, 0] = A / det
    inv[:, 0, 1] = -(b * i - c * h) / det
    inv[:, 0, 2] = (b * f - c * e) / det
    inv[:, 1, 0] = Bc / det
    inv[:, 1, 1] = (a * i - c * g) / det
    inv[:, 1, 2] = -(a * f - c * d) / det
    inv[:, 2, 0] = C / det
    inv[:, 2, 1] = -(a * h - b * g) / det
    inv[:, 2, 2] = (a * e - b * d) / det
    return inv.astype(K.dtype)


def generate_2dmeshgrid(h, w, dt):
    """transform.py:137-154: rows x, y, 1; x fastest.  Returns xs, ys (h*w,)."""
    ys, xs = np.meshgrid(np.arange(h, dtype=dt), np.arange(w, dtype=dt),
                         indexing='ij')
    return xs.reshape(-1), ys.reshape(-1)


def pixel2cam(depth, Kinv, h, w):
    """transform.py:94-109.  depth (N,h*w), Kinv (N,3,3).
    ray = Kinv . (x, y, 1):  r_k = (k_k0*x + k_k1*y) + k_k2 ; cam = depth*ray.
    Returns ray (N,3,hw) and cam (N,3,hw) (the appended ones row is implicit)."""
    xs, ys = generate_2dmeshgrid(h, w, depth.dtype)
    k = Kinv
    ray = np.stack([(k[:, r, 0, None] * xs[None] + k[:, r, 1, None] * ys[None])
                    + k[:, r, 2, None] for r in range(3)], axis=1)
    cam = depth[:, None, :] * ray
    return ray, cam


def cam2pixel(cam, proj, h, w):
    """transform.py:111-133.  q_k = ((P_k0*X + P_k1*Y) + P_k2*Z) + P_k3 ;
    z = q2 + 1e-10 ; xn = (q0/z)/((w-1)/2) - 1 ; yn likewise ; coordinates
    not strictly inside (-1,1) are multiplied by 2 (:128-131).
    Returns dict with q (N,3,hw), z, xn, yn (after the x2), inx, iny."""
    dt = cam.dtype
    P = proj
    X, Y, Z = cam[:, 0], cam[:, 1], cam[:, 2]
    q = np.stack([((P[:, r, 0, None] * X + P[:, r, 1, None] * Y)
                   + P[:, r, 2, None] * Z) + P[:, r, 3, None]
                  for r in range(3)], axis=1)
    z = q[:, 2] + dt.type(1e-10)
    hw = dt.type((w - 1) / 2.)
    hh = dt.type((h - 1) / 2.)
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        xn = (q[:, 0] / z) / hw - dt.type(1)
        yn = (q[:, 1] / z) / hh - dt.type(1)
        inx = (xn > -1) & (xn < 1)
        iny = (yn > -1) & (yn < 1)
        xn = np.where(inx, xn, xn * dt.type(2))
        yn = np.where(iny, yn, yn * dt.type(2))
    return dict(q=q, z=z, xn=xn, yn=yn, inx=inx, iny=iny, hw=hw, hh=hh)


# --------------------------------------------------------------------------
# samplers
# --------------------------------------------------------------------------
def _taps(img, u, v):
    """Zero-padded 2x2 neighbourhood gather.  img (N,C,h,w); u,v (N,hw) in
    pixel units.  Returns u0,v0 (int32), validity, the four (N,C,hw) taps and
    the 1-D weight factors."""
    N, C, h, w = img.shape
    dt = img.dtype
    with np.errstate(invalid='ignore'):
        u0f = np.floor(u)
        v0f = np.floor(v)
        # clip before the int cast so +-inf/huge coordinates stay defined
        u0 = np.clip(np.nan_to_num(u0f, nan=-2.0), -2, w + 1).astype(np.int32)
        v0 = np.clip(np.nan_to_num(v0f, nan=-2.0), -2, h + 1).astype(np.int32)
    u1 = u0 + 1
    v1 = v0 + 1
    wa = (u0f + dt.type(1)) - u      # u1 - u
    wb = u - u0f                     # u - u0
    wc = (v0f + dt.type(1)) - v
    wd = v - v0f
    vu0 = (u0 >= 0) & (u0 <= w - 1)
    vu1 = (u1 >= 0) & (u1 <= w - 1)
    vv0 = (v0 >= 0) & (v0 <= h - 1)
    vv1 = (v1 >= 0) & (v1 <= h - 1)
    bi = np.arange(N)[:, None]

    def tap(vi, ui, ok):
        g = img[bi, :, np.clip(vi, 0, h - 1), np.clip(ui, 0, w - 1)]  # (N,hw,C)
        g = np.where(ok[..., None], g, dt.type(0))
        return g.transpose(0, 2, 1)

    I00 = tap(v0, u0, vv0 & vu0)
    I01 = tap(v0, u1, vv0 & vu1)
    I10 = tap(v1, u0, vv1 & vu0)
    I11 = tap(v1, u1, vv1 & vu1)
    return dict(u0=u0, v0=v0, wa=wa, wb=wb, wc=wc, wd=wd,
                I00=I00, I01=I01, I10=I10, I11=I11,
                any_valid=(vv0 | vv1) & (vu0 | vu1))


def spatial_transformer_sampler(img, xn, yn):
    """F.spatial_transformer_sampler (call site transform.py:189): normalised
    coordinates, align-corners, bilinear, ZERO padding.
    u = ((xn+1)*(w-1))/2 ; P = ((w1*I00 + w2*I01) + w3*I10) + w4*I11.
    img (N,C,h,w); xn, yn (N,hw).  Returns P (N,C,hw) and the tap record."""
    N, C, h, w = img.shape
    dt = img.dtype
    with np.errstate(invalid='ignore', over='ignore'):
        u = ((xn + dt.type(1)) * dt.type(w - 1)) / dt.type(2)
        v = ((yn + dt.type(1)) * dt.type(h - 1)) / dt.type(2)
        t = _taps(img, u, v)
        w1 = (t['wa'] * t['wc'])[:, None]
        w2 = (t['wb'] * t['wc'])[:, None]
        w3 = (t['wa'] * t['wd'])[:, None]
        w4 = (t['wb'] * t['wd'])[:, None]
        P = ((w1 * t['I00'] + w2 * t['I01']) + w3 * t['I10']) + w4 * t['I11']
        # pixels whose every tap is in the zero pad are exactly 0
        P = np.where(t['any_valid'][:, None], P, dt.type(0))
    t['u'] = u
    t['v'] = v
    return P, t


def spatial_transformer_sampler_grad(t, gy, h, w):
    """Backward of the sampler w.r.t. the normalised grid (A.2):
    g_xn = sum_c gy_c [wc (I01-I00) + wd (I11-I10)] * (w-1)/2."""
    dt = gy.dtype
    du = t['wc'][:, None] * (t['I01'] - t['I00']) + t['wd'][:, None] * (t['I11'] - t['I10'])
    dv = t['wa'][:, None] * (t['I10'] - t['I00']) + t['wb'][:, None] * (t['I11'] - t['I01'])
    gu = np.sum(gy * du, axis=1)
    gv = np.sum(gy * dv, axis=1)
    gu = np.where(t['any_valid'], gu, dt.type(0))
    gv = np.where(t['any_valid'], gv, dt.type(0))
    return gu * dt.type((w - 1) / 2.), gv * dt.type((h - 1) / 2.)


def sampler_image_adjoint(t, gP, h, w):
    """Gradient of the sampler w.r.t. its image (float64): every pixel scatters gP_c * w_k to its valid taps; a
    pixel with no valid tap (out of view by the x2 rule) contributes nothing.  t: the tap record of the forward,
    gP (N,3,hw) -> (N,3,h*w)."""
    N = gP.shape[0]
    u0, v0 = t['u0'].astype(np.int64), t['v0'].astype(np.int64)
    wa, wb = t['wa'].astype(np.float64), t['wb'].astype(np.float64)
    wc, wd = t['wc'].astype(np.float64), t['wd'].astype(np.float64)
    out = np.zeros((N, 3, h * w), np.float64)
    bi = np.broadcast_to(np.arange(N)[:, None], u0.shape)
    for du, dv, wk in ((0, 0, wa * wc), (1, 0, wb * wc), (0, 1, wa * wd), (1, 1, wb * wd)):
        uu, vv = u0 + du, v0 + dv
        ok = t['any_valid'] & (uu >= 0) & (uu <= w - 1) & (vv >= 0) & (vv <= h - 1)
        wk = wk.astype(t['wa'].dtype).astype(np.float64)      # the forward rounds the weight products to the image dtype
        idx = np.where(ok, vv * w + uu, 0)
        for c in range(3):
            np.add.at(out[:, c], (bi, idx), np.where(ok, wk * gP[:, c], 0.0))
    return out


def sampler_interp_forward(x, grid):
    """models/spational_transformer_sampler_interp.py:32-78 -- the repo-local
    sampler (unused by the live path): grid in PIXEL units, indices clamped to
    the image, weights taken from the clamped indices."""
    B, C, H, W = x.shape
    u = grid[:, 0].reshape(-1)
    v = grid[:, 1].reshape(-1)
    u0 = np.floor(u)
    u1 = u0 + 1
    v0 = np.floor(v)
    v1 = v0 + 1
    u0 = u0.clip(0, W - 1)
    v0 = v0.clip(0, H - 1)
    u1 = u1.clip(0, W - 1)
    v1 = v1.clip(0, H - 1)
    wt_x0 = u1 - u
    wt_x1 = u - u0
    wt_y0 = v1 - v
    wt_y1 = v - v0
    w1 = (wt_x0 * wt_y0).astype(x.dtype)
    w2 = (wt_x1 * wt_y0).astype(x.dtype)
    w3 = (wt_x0 * wt_y1).astype(x.dtype)
    w4 = (wt_x1 * wt_y1).astype(x.dtype)
    u0 = u0.astype(np.int32)
    v0 = v0.astype(np.int32)
    u1 = u1.astype(np.int32)
    v1 = v1.astype(np.int32)
    oH, oW = grid.shape[2:]
    bi = np.repeat(np.arange(B), oH * oW)
    y = w1[:, None] * x[bi, :, v0, u0]
    y = y + w2[:, None] * x[bi, :, v0, u1]
    y = y + w3[:, None] * x[bi, :, v1, u0]
    y = y + w4[:, None] * x[bi, :, v1, u1]
    return y.reshape(B, oH, oW, C).transpose(0, 3, 1, 2)


def sampler_interp_backward(x, grid, gy):
    """models/spational_transformer_sampler_interp.py:86-149: ggrid in pixel
    units, gx = zeros (:148)."""
    B, C, H, W = x.shape
    oH, oW = grid.shape[2:]
    u = grid[:, 0].reshape(-1)
    v = grid[:, 1].reshape(-1)
    u0 = np.floor(u)
    u1 = u0 + 1
    v0 = np.floor(v)
    v1 = v0 + 1
    u0 = u0.clip(0, W - 1)
    v0 = v0.clip(0, H - 1)
    u1 = u1.clip(0, W - 1)
    v1 = v1.clip(0, H - 1)
    wt_x0 = (u1 - u).astype(gy.dtype)
    wt_x1 = (u - u0).astype(gy.dtype)
    wt_y0 = (v1 - v).astype(gy.dtype)
    wt_y1 = (v - v0).astype(gy.dtype)
    u0 = u0.astype(np.int32)
    v0 = v0.astype(np.int32)
    u1 = u1.astype(np.int32)
    v1 = v1.astype(np.int32)
    bi = np.repeat(np.arange(B), oH * oW)
    x1 = x[bi, :, v0, u0]
    x2 = x[bi, :, v0, u1]
    x3 = x[bi, :, v1, u0]
    x4 = x[bi, :, v1, u1]
    gu = -wt_y0[:, None] * x1
    gu = gu + wt_y0[:, None] * x2
    gu = gu - wt_y1[:, None] * x3
    gu = gu + wt_y1[:, None] * x4
    gv = -wt_x0[:, None] * x1
    gv = gv - wt_x1[:, None] * x2
    gv = gv + wt_x0[:, None] * x3
    gv = gv + wt_x1[:, None] * x4
    gu = gu.reshape(B, oH, oW, C).transpose(0, 3, 1, 2) * gy
    gv = gv.reshape(B, oH, oW, C).transpose(0, 3, 1, 2) * gy
    ggrid = np.concatenate((gu.sum(1)[:, None], gv.sum(1)[:, None]), axis=1)
    return np.zeros_like(x), ggrid


# --------------------------------------------------------------------------
# pyramid  (F.resize_images, call sites base_model.py:71-72)
# --------------------------------------------------------------------------
def resize_axis_tables(n_in, n_out):
    """float64 linspace coordinates -> (i0, w0=(i1-u), w1=(u-i0)) per output
    index, exactly as Chainer's resize_images computes them."""
    if n_out > 1:
        step = float(n_in - 1) / float(n_out - 1)
        u = np.arange(n_out, dtype=np.float64) * step
        u[-1] = float(n_in - 1)
    else:
        u = np.zeros(1, np.float64)
    i0 = np.clip(np.floor(u).astype(np.int32), 0, n_in - 2)
    i1 = i0 + 1
    return i0, (i1 - u), (u - i0)


def resize_images(x, out_shape):
    """Align-corners bilinear from full resolution; weights are float64
    products cast to x.dtype; y = ((w1*a + w2*b) + w3*c) + w4*d."""
    B, C, H, W = x.shape
    oh, ow = out_shape
    u0, ua, ub = resize_axis_tables(W, ow)
    v0, va, vb = resize_axis_tables(H, oh)
    w1 = (va[:, None] * ua[None, :]).astype(x.dtype)
    w2 = (va[:, None] * ub[None, :]).astype(x.dtype)
    w3 = (vb[:, None] * ua[None, :]).astype(x.dtype)
    w4 = (vb[:, None] * ub[None, :]).astype(x.dtype)
    V0, U0 = v0[:, None], u0[None, :]
    return ((w1 * x[:, :, V0, U0] + w2 * x[:, :, V0, U0 + 1])
            + w3 * x[:, :, V0 + 1, U0]) + w4 * x[:, :, V0 + 1, U0 + 1]


def resize_images_adjoint(gy, in_shape, dtype=np.float32):
    """Adjoint of resize_images (float64): gy (B,C,oh,ow) -> (B,C,H,W).  The tap weights are the forward's, float64
    products rounded to `dtype`.  The identity when the sizes agree (scale 0)."""
    B, C, oh, ow = gy.shape
    H, W = in_shape
    if (oh, ow) == (H, W):
        return gy.astype(np.float64)
    u0, ua, ub = resize_axis_tables(W, ow)
    v0, va, vb = resize_axis_tables(H, oh)
    gx = np.zeros((B, C, H, W), np.float64)
    V0, U0 = np.broadcast_arrays(v0[:, None], u0[None, :])
    for wv, wu, dv, du in ((va, ua, 0, 0), (va, ub, 0, 1), (vb, ua, 1, 0), (vb, ub, 1, 1)):
        wk = (wv[:, None] * wu[None, :]).astype(dtype).astype(np.float64)
        np.add.at(gx.transpose(2, 3, 0, 1), (V0 + dv, U0 + du), (wk * gy).transpose(2, 3, 0, 1))
    return gx


# --------------------------------------------------------------------------
# loss terms (models/base_model.py)
# --------------------------------------------------------------------------
def avg_pool3(x):
    """F.average_pooling_2d(x, 3, 1, 1): zero pad, always divide by 9.
    Canonical order: row-major running sum of the 9 taps, then /9."""
    h, w = x.shape[-2:]
    pad = [(0, 0)] * (x.ndim - 2) + [(1, 1), (1, 1)]
    xp = np.pad(x, pad, mode='constant')
    acc = None
    for dy in range(3):
        for dx in range(3):
            t = xp[..., dy:dy + h, dx:dx + w]
            acc = t if acc is None else acc + t
    return acc / x.dtype.type(9)


def ssim_terms(P, T):
    """base_model.py:126-142 -- returns every intermediate the backward needs."""
    dt = P.dtype
    c1, c2 = dt.type(SSIM_C1), dt.type(SSIM_C2)
    a = avg_pool3(P)
    my = avg_pool3(T)
    sx = avg_pool3(P * P) - a * a
    sy = avg_pool3(T * T) - my * my
    sxy = avg_pool3(P * T) - a * my
    n1 = dt.type(2) * a * my + c1
    n2 = dt.type(2) * sxy + c2
    d1 = a * a + my * my + c1
    d2 = sx + sy + c2
    n = n1 * n2
    d = d1 * d2
    raw = (dt.type(1) - n / d) / dt.type(2)
    return dict(a=a, my=my, n1=n1, n2=n2, d1=d1, d2=d2, n=n, d=d, raw=raw)


def compute_ssim(P, T):
    return np.clip(ssim_terms(P, T)['raw'], 0, 1)


def smooth_terms(D):
    """base_model.py:169-185 on disp (B,1,h,w)."""
    dx = D[..., :, 1:] - D[..., :, :-1]
    dy = D[..., 1:, :] - D[..., :-1, :]
    dx2 = dx[..., :, 1:] - dx[..., :, :-1]
    dxdy = dx[..., 1:, :] - dx[..., :-1, :]
    dydx = dy[..., :, 1:] - dy[..., :, :-1]
    dy2 = dy[..., 1:, :] - dy[..., :-1, :]
    return dx2, dxdy, dydx, dy2


def _fsum(x):
    return float(np.sum(x, dtype=np.float64))


# --------------------------------------------------------------------------
# stage API used by stage-isolated parity tests
# --------------------------------------------------------------------------
def projective_inverse_warp(imgs, depth, poses, K, proj=None, Kinv=None):
    """transform.py:156-193.  imgs (N,3,h,w), depth (N,h*w) [the reference
    passes it broadcast to 3 rows], poses (N,6), K (N,3,3).
    Returns P (N,3,h,w) and a record of intermediates (u0, v0, in-bounds ...)."""
    N, _, h, w = imgs.shape
    if proj is None:
        proj = proj_tgt_to_src(poses, K)
    if Kinv is None:
        Kinv = batch_inv3(K)
    ray, cam = pixel2cam(depth, Kinv, h, w)
    g = cam2pixel(cam, proj, h, w)
    P, t = spatial_transformer_sampler(imgs, g['xn'], g['yn'])
    rec = dict(ray=ray, cam=cam, grid=g, taps=t, proj=proj, Kinv=Kinv)
    return P.reshape(N, 3, h, w), rec


# --------------------------------------------------------------------------
# the full loss path, forward + analytic backward
# --------------------------------------------------------------------------
def disp_smooth_terms(img, D):
    """compute_disp_smooth (base_model.py:144-155): first differences of the disparity weighted by
    exp(-|channel-mean image gradient|).  img (B,3,h,w), D (B,1,h,w) -> (d_dx, e_x, d_dy, e_y)."""
    t = D.dtype.type
    d_dy = D[:, :, 1:] - D[:, :, :-1]
    d_dx = D[:, :, :, 1:] - D[:, :, :, :-1]
    i_dy = (img[:, :, 1:] - img[:, :, :-1]).mean(axis=1, keepdims=True, dtype=D.dtype)
    i_dx = (img[:, :, :, 1:] - img[:, :, :, :-1]).mean(axis=1, keepdims=True, dtype=D.dtype)
    return d_dx, np.exp(-np.abs(i_dx)).astype(D.dtype), d_dy, np.exp(-np.abs(i_dy)).astype(D.dtype)


class LossConfig(object):
    def __init__(self, smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0,
                 n_scales=N_SCALES, B_global=None, edge_aware_smooth=False):
        # edge_aware_smooth: the smoothness term is compute_disp_smooth(curr_tgt_img, pred_disps[ns]) -- the
        # alternative the reference keeps commented out at base_model.py:78-80 -- instead of compute_smooth_loss
        self.edge_aware_smooth = edge_aware_smooth
        self.smooth_reg = smooth_reg
        self.exp_reg = exp_reg
        self.ssim_rate = ssim_rate
        self.n_scales = n_scales
        self.B_global = B_global


def _pose_backward(vec, K_scales, dP_scales):
    """Chain dL/dP_s (N,3,4) per scale back to the 6-DoF vector (A.6)."""
    dt = vec.dtype
    N = vec.shape[0]
    dT = np.zeros((N, 3, 4), np.float64)
    for K, dP in zip(K_scales, dP_scales):
        dT += np.einsum('nkr,nkj->nrj', K.astype(np.float64), dP)
    rc, c, s = euler_sincos(vec[:, :3])
    xmat, ymat, zmat = [m.astype(np.float64) for m in _rot_mats(c, s)]
    c = c.astype(np.float64)
    s = s.astype(np.float64)
    G_R = dT[:, :, :3]
    A = xmat @ ymat
    G_Rz = A.transpose(0, 2, 1) @ G_R
    G_A = G_R @ zmat.transpose(0, 2, 1)
    G_Rx = G_A @ ymat.transpose(0, 2, 1)
    G_Ry = xmat.transpose(0, 2, 1) @ G_A
    z = np.zeros(N)
    dRx = np.stack([z, z, z, z, -s[:, 0], -c[:, 0], z, c[:, 0], -s[:, 0]], 1).reshape(N, 3, 3)
    dRy = np.stack([-s[:, 1], z, c[:, 1], z, z, z, -c[:, 1], z, -s[:, 1]], 1).reshape(N, 3, 3)
    dRz = np.stack([-s[:, 2], -c[:, 2], z, c[:, 2], -s[:, 2], z, z, z, z], 1).reshape(N, 3, 3)
    g = np.zeros((N, 6), np.float64)
    g[:, 0] = np.sum(G_Rx * dRx, axis=(1, 2))
    g[:, 1] = np.sum(G_Ry * dRy, axis=(1, 2))
    g[:, 2] = np.sum(G_Rz * dRz, axis=(1, 2))
    r = vec[:, :3]
    inside = (r >= dt.type(-np.pi)) & (r <= dt.type(np.pi))   # F.clip backward
    g[:, :3] *= inside
    g[:, 3:] = dT[:, :, 3]
    return g.astype(dt), dT


def intrinsics_grad(intrinsics, poses, dP):
    """d total / d intrinsics from the dL/dP cells -> (B,n_scales,3,3) float64.  intrinsics (B,n_scales,3,3), poses
    (B,S,6) as the loss used them, dP (B,S,n_scales,3,4).

    K enters the projection P = K4 . [R|t] (transform.py:86-88) and pixel2cam's batch_inv(K) (:105).  Per pixel
    q = K (R c + t) with c = depth K^-1 pix, so with the cells dL/dP = [A_i | g_i] (A_i = sum gq (x) c, g_i = sum gq):

        dL/dK_s = sum_i [ A_i R_i^T + g_i t_i^T - K_s^-T R_i^T K_s^T A_i ]

    R_i = (Rx . Ry) . Rz of the clipped angles with sin / cos rounded to the working dtype and t_i unclipped, as
    `_pose_backward` has them; K^-1 and the sum in float64."""
    B, S, ns = dP.shape[:3]
    K = intrinsics.astype(np.float64)
    Ki = np.linalg.inv(K)
    out = np.zeros((B, ns, 3, 3), np.float64)
    for i in range(S):
        _, c, s = euler_sincos(poses[:, i, :3])
        xm, ym, zm = [m.astype(np.float64) for m in _rot_mats(c, s)]
        R = ((xm @ ym) @ zm)[:, None]                                    # (B,1,3,3)
        t = poses[:, i, 3:].astype(np.float64)[:, None]                  # (B,1,3)
        A, g = dP[:, i, :, :, :3], dP[:, i, :, :, 3]
        RT = np.swapaxes(R, -1, -2)
        out += A @ RT + g[..., :, None] * t[..., None, :]
        out -= np.swapaxes(Ki, -1, -2) @ RT @ np.swapaxes(K, -1, -2) @ A
    return out


def sfm_loss(tgt, src, intrinsics, disps, poses, logits, cfg,
             want_grads=True, proj_override=None, kinv_override=None,
             want_debug=False, want_image_grads=False, want_intrinsics_grad=False):
    """SFMLearner.__call__ loss loop (base_model.py:57-124) + its backward.

    tgt (B,3,H,W); src (B,S,3,H,W); intrinsics (B,n_scales,3,3);
    disps: list of (B,1,h_s,w_s); poses (B,S,6); logits: list of (B,S,h_s,w_s)
    or None.  Returns (losses dict, grads dict or None, debug dict).
    `cfg.B_global` (default B) is the batch size every F.mean divides by, so a
    shard of a larger batch yields partial sums that add up to the full loss.

    Opt-in gradients (both need `want_grads`), added to the grads dict in float64:
    * want_image_grads: gtgt (B,3,H,W) and gsrc (B,S,3,H,W).  The images are
      treated as differentiable throughout (the reference's `.data` on the
      pyramid, base_model.py:71-72, and on mu_y / sigma_y, :131, :134, are
      lifted), so they are the derivative of the reported total; the all-zero
      mask (:96) is piecewise constant.  Not with the edge-aware smoothness term.
    * want_intrinsics_grad: dP (B,S,n_scales,3,4), the dL/dP cells the pose
      chain starts from, and gintrinsics (B,n_scales,3,3) (`intrinsics_grad`).
    """
    if (want_image_grads or want_intrinsics_grad) and not want_grads:
        raise ValueError('image and intrinsics gradients need want_grads')
    if want_image_grads and cfg.smooth_reg and cfg.edge_aware_smooth:
        raise ValueError('image gradients through the edge-aware smoothness term are not supported')
    dt = tgt.dtype
    B, S, _, H, W = src.shape
    Bg = cfg.B_global if cfg.B_global else B
    ns_total = cfg.n_scales
    stacked = src.reshape(B, 3 * S, H, W)
    pixel_loss = smooth_loss = exp_loss = ssim_loss = 0.0
    use_exp = bool(cfg.exp_reg)
    use_ssim = (not use_exp) and bool(cfg.ssim_rate)
    use_smooth = bool(cfg.smooth_reg)
    ssim_rate = cfg.ssim_rate if cfg.ssim_rate else 0.0
    gdisp = [np.zeros(d.shape, np.float64) for d in disps]
    glogits = [np.zeros(l.shape, np.float64) for l in logits] if (use_exp and logits is not None) else None
    dP_all = [[None] * ns_total for _ in range(S)]
    if want_image_grads:
        gtgt = np.zeros(tgt.shape, np.float64)
        gsrc = np.zeros(src.shape, np.float64)
    debug = dict(P=[], u0=[], v0=[], inb=[], tgt_pyr=[], src_pyr=[])

    for ns in range(ns_total):
        h, w = scale_shape(H, W, ns)
        hw_n = h * w
        cur_tgt = resize_images(tgt, (h, w))
        cur_src = resize_images(stacked, (h, w))
        if want_debug:
            debug['tgt_pyr'].append(cur_tgt)
            debug['src_pyr'].append(cur_src.reshape(B, S, 3, h, w))
        D = disps[ns]
        # ---- edge-aware smoothness (base_model.py:78-80 as written in the comment, 144-155)
        if use_smooth and cfg.edge_aware_smooth:
            wgt = cfg.smooth_reg / (2 ** ns)
            d_dx, e_x, d_dy, e_y = disp_smooth_terms(cur_tgt, D)
            n_x, n_y = Bg * h * (w - 1), Bg * (h - 1) * w
            smooth_loss += wgt * (_fsum(np.abs(d_dx) * e_x) / n_x + _fsum(np.abs(d_dy) * e_y) / n_y)
            if want_grads:
                g = gdisp[ns][:, 0]
                sx = np.sign(d_dx[:, 0]).astype(np.float64) * e_x[:, 0] * (wgt / n_x)
                g[:, :, 1:] += sx
                g[:, :, :-1] -= sx
                sy = np.sign(d_dy[:, 0]).astype(np.float64) * e_y[:, 0] * (wgt / n_y)
                g[:, 1:, :] += sy
                g[:, :-1, :] -= sy
        # ---- smoothness (base_model.py:75-77, 169-185)
        elif use_smooth:
            wgt = cfg.smooth_reg / (2 ** ns)
            dx2, dxdy, dydx, dy2 = smooth_terms(D)
            n_dx2 = Bg * h * (w - 2)
            n_mix = Bg * (h - 1) * (w - 1)
            n_dy2 = Bg * (h - 2) * w
            smooth_loss += wgt * (_fsum(np.abs(dx2)) / n_dx2 + _fsum(np.abs(dxdy)) / n_mix
                                  + _fsum(np.abs(dydx)) / n_mix + _fsum(np.abs(dy2)) / n_dy2)
            if want_grads:
                g = gdisp[ns][:, 0]
                s = np.sign(dx2[:, 0]).astype(np.float64) * (wgt / n_dx2)
                g[:, :, :-2] += s
                g[:, :, 1:-1] -= 2 * s
                g[:, :, 2:] += s
                s = np.sign(dy2[:, 0]).astype(np.float64) * (wgt / n_dy2)
                g[:, :-2, :] += s
                g[:, 1:-1, :] -= 2 * s
                g[:, 2:, :] += s
                for m in (dxdy, dydx):
                    s = np.sign(m[:, 0]).astype(np.float64) * (wgt / n_mix)
                    g[:, 1:, 1:] += s
                    g[:, 1:, :-1] -= s
                    g[:, :-1, 1:] -= s
                    g[:, :-1, :-1] += s
        # ---- depth (base_model.py:60, 81-84)
        disp_flat = D.reshape(B, hw_n)
        depth = dt.type(1) / disp_flat
        K = intrinsics[:, ns]
        Kinv = kinv_override[:, ns] if kinv_override is not None else batch_inv3(K)
        ray, cam = pixel2cam(depth, Kinv, h, w)
        g_depth = np.zeros((B, hw_n), np.float64)
        if want_image_grads:
            gT = np.zeros((B, 3, h, w), np.float64)
            gS = np.zeros((B, S, 3, h, w), np.float64)
        dbgP, dbgu, dbgv, dbgi = [], [], [], []
        for i in range(S):
            img = cur_src[:, 3 * i:3 * i + 3]
            if proj_override is not None:
                proj = proj_override[:, i, ns]
            else:
                proj = proj_tgt_to_src(poses[:, i], K)
            gr = cam2pixel(cam, proj, h, w)
            Pf, t = spatial_transformer_sampler(img, gr['xn'], gr['yn'])
            P = Pf.reshape(B, 3, h, w)
            if want_debug:
                dbgP.append(P)
                dbgu.append(t['u0'].reshape(B, h, w))
                dbgv.append(t['v0'].reshape(B, h, w))
                dbgi.append((gr['inx'] & gr['iny']).reshape(B, h, w))
            diff = P - cur_tgt
            err = np.abs(diff)
            m = np.all(P == 0, axis=1, keepdims=True)          # base_model.py:96
            err = np.where(m, dt.type(0), err)
            n_pix3 = Bg * 3 * h * w
            gP = np.zeros(P.shape, np.float64)
            sgn = np.where(m, 0.0, np.sign(diff)).astype(np.float64)
            if use_exp:
                l = logits[ns][:, i:i + 1]
                sg = _sigmoid(l)
                exp_loss += cfg.exp_reg * _fsum(_softplus_neg(l)) / (Bg * h * w)
                pixel_loss += _fsum(err * sg) / n_pix3
                if want_grads:
                    sg64 = sg.astype(np.float64)
                    gP += sgn * sg64 * ((1 - ssim_rate) / n_pix3)
                    e_sum = np.sum(err.astype(np.float64), axis=1, keepdims=True)
                    glogits[ns][:, i:i + 1] += ((1 - ssim_rate) * e_sum * sg64 * (1 - sg64) / n_pix3
                                                - cfg.exp_reg * (1 - sg64) / (Bg * h * w))
            else:
                pixel_loss += _fsum(err) / n_pix3
                if want_grads:
                    gP += sgn * ((1 - ssim_rate) / n_pix3)
            if want_image_grads:
                gT -= gP                                        # the L1 part: d|P - T| / dT = -d|P - T| / dP
            if use_ssim:
                st = ssim_terms(P, cur_tgt)
                e = np.clip(st['raw'], 0, 1) * (1 - m)
                ssim_loss += _fsum(e) / n_pix3
                if want_grads:
                    raw = st['raw'].astype(np.float64)
                    a, my = st['a'].astype(np.float64), st['my'].astype(np.float64)
                    n1, n2 = st['n1'].astype(np.float64), st['n2'].astype(np.float64)
                    d1, d2 = st['d1'].astype(np.float64), st['d2'].astype(np.float64)
                    n, d = st['n'].astype(np.float64), st['d'].astype(np.float64)
                    g_e = (ssim_rate / n_pix3) * (1 - m) * ((raw >= 0) & (raw <= 1))
                    g_n = -g_e / (2 * d)
                    g_d = g_e * n / (2 * d * d)
                    g_a = g_n * (2 * my * n2 - 2 * my * n1) + g_d * (2 * a * d2 - 2 * a * d1)
                    g_s = g_d * d1
                    g_c = 2 * g_n * n1
                    Pd, Td = P.astype(np.float64), cur_tgt.astype(np.float64)
                    As, Ac = avg_pool3(g_s), avg_pool3(g_c)
                    gP += avg_pool3(g_a) + 2 * Pd * As + Td * Ac
                    if want_image_grads:
                        # avg_pool3 is its own adjoint; g_my mirrors g_a
                        g_my = g_n * (2 * a * n2 - 2 * a * n1) + g_d * (2 * my * d2 - 2 * my * d1)
                        gT += avg_pool3(g_my) + 2 * Td * As + Pd * Ac
            if want_grads:
                # sampler -> grid -> q -> cam/proj  (A.6)
                gyf = gP.reshape(B, 3, hw_n)
                t64 = {k: (v.astype(np.float64) if v.dtype.kind == 'f' else v) for k, v in t.items()}
                g_xn, g_yn = spatial_transformer_sampler_grad(t64, gyf, h, w)
                g_xn = g_xn * np.where(gr['inx'], 1.0, 2.0)
                g_yn = g_yn * np.where(gr['iny'], 1.0, 2.0)
                q = gr['q'].astype(np.float64)
                z = gr['z'].astype(np.float64)
                hw_, hh_ = float(gr['hw']), float(gr['hh'])
                with np.errstate(divide='ignore', invalid='ignore'):
                    g_q0 = g_xn / (z * hw_)
                    g_q1 = g_yn / (z * hh_)
                    g_q2 = -(g_xn * q[:, 0] / hw_ + g_yn * q[:, 1] / hh_) / (z * z)
                g_q = np.stack([g_q0, g_q1, g_q2], axis=1)
                g_q = np.where(t['any_valid'][:, None], g_q, 0.0)
                P64 = proj.astype(np.float64)
                g_cam = np.einsum('nkp,nkj->njp', g_q, P64[:, :3, :3])
                g_depth += np.sum(g_cam * ray.astype(np.float64), axis=1)
                cam4 = np.concatenate([cam.astype(np.float64), np.ones((B, 1, hw_n))], axis=1)
                dP_all[i][ns] = np.einsum('nkp,njp->nkj', g_q, cam4)
                if want_image_grads:
                    gS[:, i] = sampler_image_adjoint(t, gyf, h, w).reshape(B, 3, h, w)
        if want_image_grads:
            gtgt += resize_images_adjoint(gT, (H, W), dt)
            gsrc += resize_images_adjoint(gS.reshape(B, 3 * S, h, w), (H, W), dt).reshape(src.shape)
        if want_debug:
            debug['P'].append(np.stack(dbgP, 1))
            debug['u0'].append(np.stack(dbgu, 1))
            debug['v0'].append(np.stack(dbgv, 1))
            debug['inb'].append(np.stack(dbgi, 1))
        if want_grads:
            d64 = disp_flat.astype(np.float64)
            gdisp[ns] += (-g_depth / (d64 * d64)).reshape(D.shape)

    total = (1 - ssim_rate) * pixel_loss + ssim_rate * ssim_loss + smooth_loss + exp_loss
    losses = dict(total_loss=total, pixel_loss=pixel_loss, smooth_loss=smooth_loss,
                  exp_loss=exp_loss, ssim_loss=ssim_loss)
    grads = None
    if want_grads:
        gpose = np.zeros((B, S, 6), dt)
        dT_all = np.zeros((B, S, 3, 4), np.float64)
        K_scales = [intrinsics[:, ns] for ns in range(ns_total)]
        for i in range(S):
            gpose[:, i], dT_all[:, i] = _pose_backward(poses[:, i], K_scales, dP_all[i])
        grads = dict(gdisp=[g.astype(dt) for g in gdisp], gpose=gpose,
                     glogits=[g.astype(dt) for g in glogits] if glogits is not None else None,
                     dT=dT_all)
        if want_image_grads:
            grads.update(gtgt=gtgt, gsrc=gsrc)
        if want_intrinsics_grad:
            dP = np.stack([np.stack(dP_all[i], 1) for i in range(S)], 1)
            grads.update(dP=dP, gintrinsics=intrinsics_grad(intrinsics, poses, dP))
    return losses, grads, debug


LOSS_KEYS = ('total_loss', 'pixel_loss', 'smooth_loss', 'exp_loss', 'ssim_loss')


# --------------------------------------------------------------------------------------------------
# The seam either side of the loss (SURVEY section 8(f) rank 1): the last op of each producer
# --------------------------------------------------------------------------------------------------
DISP_SCALING = 10      # models/disp_net.py:7
MIN_DISP = 0.01        # models/disp_net.py:8


def disp_activation(x):
    """disp = DISP_SCALING * F.sigmoid(x) + MIN_DISP (models/disp_net.py:104,110,116,122) and d disp / d x.

    Chainer's sigmoid is tanh(x * 0.5) * 0.5 + 0.5 (functions/activation/sigmoid.py, forward_cpu) with
    backward gy * y * (1 - y); the scaling and the offset are separate elementwise ops, each rounded."""
    t = x.dtype.type
    y = np.tanh(x * t(0.5)) * t(0.5) + t(0.5)
    return t(DISP_SCALING) * y + t(MIN_DISP), t(DISP_SCALING) * y * (t(1) - y)


def pose_from_raw(x, n_sources):
    """PoseNet.pred_pose's tail (models/pose_net.py:52-53): 0.01 * F.mean(poseout, (2, 3)) split into
    n_sources 6-DoF vectors.  x (B, 6*S, h', w') -> (B, S, 6).  numpy reduces the contiguous (h', w') block of
    a channel with its pairwise fp32 sum."""
    t = x.dtype.type
    B = x.shape[0]
    m = np.ascontiguousarray(x).reshape(B, 6 * n_sources, -1).mean(axis=2, dtype=x.dtype)
    return (t(0.01) * m).reshape(B, n_sources, 6)


def sfm_loss_raw(tgt, src, intrinsics, disps_in, poses_in, logits, cfg, raw_disp_scales=0, raw_pose=False, **kw):
    """sfm_loss with the seam included: scales in the bit mask `raw_disp_scales` take the pre-activation
    `dispout` map, `raw_pose` takes the `poseout` map (B, 6*S, h', w').  Gradients are returned w.r.t. what was
    passed in (chain rule through disp_activation / pose_from_raw).  The opt-in gradients of sfm_loss pass through
    as they are: gintrinsics is built from the reduced pose vectors."""
    S = src.shape[1]
    disps, dacts = [], []
    for s, d in enumerate(disps_in):
        if (raw_disp_scales >> s) & 1:
            dd, da = disp_activation(d)
            disps.append(dd)
            dacts.append(da)
        else:
            disps.append(d)
            dacts.append(None)
    poses = pose_from_raw(poses_in, S) if raw_pose else poses_in
    losses, grads, debug = sfm_loss(tgt, src, intrinsics, disps, poses, logits, cfg, **kw)
    if grads is not None:
        grads = dict(grads)
        grads['gdisp'] = [g if da is None else (g.astype(np.float64) * da).astype(g.dtype)
                          for g, da in zip(grads['gdisp'], dacts)]
        if raw_pose:
            n = int(np.prod(poses_in.shape[2:]))
            gp = grads['gpose'].astype(np.float64).reshape(poses_in.shape[0], 6 * S, *([1] * (poses_in.ndim - 2)))
            grads['gpose'] = np.broadcast_to(gp * (0.01 / n), poses_in.shape).astype(poses_in.dtype)
    return losses, grads, dict(debug, disps=disps, poses=poses)


def losses_vec(losses):
    return np.array([losses[k] for k in LOSS_KEYS], np.float64)


# --------------------------------------------------------------------------------------------------
# The data layer in front of the loss (SURVEY section 8(f) rank 3)
# --------------------------------------------------------------------------------------------------
def load_as_float_norm(frame_hwc_u8):
    """datasets/kitti/kitti_raw_dataset.py:12-14: imread(path).astype(float32).transpose(2, 0, 1) / (255. * 0.5) - 1."""
    img = frame_hwc_u8.astype(np.float32).transpose(2, 0, 1)
    return img / (255. * 0.5) - 1


def data_augmentation(imgs, intrinsics, aug):
    """datasets/kitti/kitti_raw_transformed.py:23-74 with the random draws supplied (`aug`: out_h, out_w, off_y,
    off_x, flip, x_scaling, y_scaling as float64).  imgs (1+S, 3, H, W) float32, intrinsics (3,3) float32."""
    _, _, H, W = imgs.shape
    xs, ys = np.float64(aug['x_scaling']), np.float64(aug['y_scaling'])
    imgs = resize_images(imgs, (aug['out_h'], aug['out_w']))                                   # :38
    fx, fy = intrinsics[0, 0] * xs, intrinsics[1, 1] * ys                                      # :39-42 (float32 * float64)
    cx, cy = intrinsics[0, 2] * xs, intrinsics[1, 2] * ys
    K = np.array([[fx, 0., cx], [0., fy, cy], [0., 0., 1.]], dtype='f')                        # make_intrinsics_matrix :16-20
    oy, ox = aug['off_y'], aug['off_x']
    imgs = imgs[:, :, oy:oy + H, ox:ox + W]                                                    # :51
    K = np.array([[K[0, 0], 0., K[0, 2] - ox], [0., K[1, 1], K[1, 2] - oy], [0., 0., 1.]], dtype='f')   # :52-56
    if aug['flip']:                                                                            # :63-65
        imgs = imgs[:, :, :, ::-1]
        K[0, 2] = W - K[0, 2]
    return np.ascontiguousarray(imgs), K


def get_multi_scale_intrinsics(K, n_scales):
    """datasets/kitti/kitti_raw_transformed.py:76-93."""
    out = np.zeros((n_scales, 3, 3), np.float32)
    for s in range(n_scales):
        out[s] = np.array([[K[0, 0] / (2 ** s), 0., K[0, 2] / (2 ** s)], [0., K[1, 1] / (2 ** s), K[1, 2] / (2 ** s)],
                           [0., 0., 1.]], dtype='f')
    return out


def ingest_u8(frames, K, aug=None, n_scales=4):
    """frames (B, 1+S, H, W, 3) uint8, K (B,3,3), aug: list of B dicts or None
    -> tgt (B,3,H,W), src (B,S,3,H,W), intrinsics (B,n_scales,3,3), as the dataset + transform hand them to the model."""
    B, n, H, W, _ = frames.shape
    tgt = np.zeros((B, 3, H, W), np.float32)
    src = np.zeros((B, n - 1, 3, H, W), np.float32)
    Ks = np.zeros((B, n_scales, 3, 3), np.float32)
    for b in range(B):
        imgs = np.stack([load_as_float_norm(frames[b, j]) for j in range(n)])
        Kb = K[b].astype(np.float32)
        if aug is not None:
            imgs, Kb = data_augmentation(imgs, Kb, aug[b])
        tgt[b], src[b] = imgs[0], imgs[1:]
        Ks[b] = get_multi_scale_intrinsics(Kb, n_scales)
    return tgt, src, Ks


# --------------------------------------------------------------------------------------------------
# Inference-side depth evaluation (SURVEY section 8(f) rank 4)
# --------------------------------------------------------------------------------------------------
def compute_depth_errors(gt, pred):
    """kitti_eval/depth_util.py:6-22."""
    thresh = np.maximum((gt / pred), (pred / gt))
    a1 = (thresh < 1.25).mean()
    a2 = (thresh < 1.25 ** 2).mean()
    a3 = (thresh < 1.25 ** 3).mean()
    rmse = np.sqrt(((gt - pred) ** 2).mean())
    rmse_log = np.sqrt(((np.log(gt) - np.log(pred)) ** 2).mean())
    abs_rel = np.mean(np.abs(gt - pred) / gt)
    sq_rel = np.mean(((gt - pred) ** 2) / gt)
    return np.array([abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3], dtype='f')


def evaluate_depth_batch(pred_depth, gt_depth, mask, min_depth, max_depth):
    """One iteration of evaluate_depth's loop, evaluate.py:94-103: resize the prediction (B,1,h,w) to the ground
    truth's size, clip, mask, scale by the ratio of medians, compute the seven errors.  -> (errors (7,), scale)."""
    pred = resize_images(pred_depth, gt_depth.shape[1:])
    pred = np.clip(pred, pred.dtype.type(min_depth), pred.dtype.type(max_depth))[:, 0]
    m = mask.astype(bool)
    pred, gt = pred[m], gt_depth[m]
    scale = np.median(gt) / np.median(pred)
    pred = pred * scale
    return compute_depth_errors(gt, pred), scale
