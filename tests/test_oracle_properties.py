"""Property tests of the oracle (SURVEY section 4, T4) with hypothesis: randomised small shapes, poses and flag sets.
They pin the semantics the multi-GPU decomposition and the kernels' task decomposition rely on."""
import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.distributed import shard_range
from sfm_learner_chainer_b200.synthetic import make_snippets

FLAGS = [dict(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.0), dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15),
         dict(smooth_reg=0.1, exp_reg=0.2, ssim_rate=0.0), dict(smooth_reg=0.2, exp_reg=0.0, ssim_rate=0.0, edge_aware_smooth=True)]
shape = st.tuples(st.integers(2, 4), st.integers(1, 3), st.sampled_from([32, 36, 40]), st.sampled_from([32, 44, 56]))


def _loss(d, cfg, **kw):
    return O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], d['logits'], cfg, **kw)


@settings(max_examples=8, deadline=None)
@given(shape, st.integers(0, 3), st.integers(0, 10 ** 6), st.integers(2, 3))
def test_shard_sums_equal_the_full_batch(sh, fi, seed, world):
    B, S, H, W = sh
    d = make_snippets(B, S, H, W, seed=seed % 1000, harsh=bool(seed & 1))
    Lf, Gf, _ = _loss(d, O.LossConfig(**FLAGS[fi]))
    acc = np.zeros(5)
    for r in range(min(world, B)):
        lo, hi = shard_range(B, r, min(world, B))
        sl = slice(lo, hi)
        part = dict(tgt=d['tgt'][sl], src=d['src'][sl], intrinsics=d['intrinsics'][sl], disps=[x[sl] for x in d['disps']],
                    poses=d['poses'][sl], logits=[x[sl] for x in d['logits']])
        L, G, _ = _loss(part, O.LossConfig(B_global=B, **FLAGS[fi]))
        acc += O.losses_vec(L)
        np.testing.assert_allclose(G['gpose'], Gf['gpose'][sl], rtol=1e-5, atol=1e-9)
        for s in range(4):
            np.testing.assert_allclose(G['gdisp'][s], Gf['gdisp'][s][sl], rtol=1e-5, atol=1e-12)
    np.testing.assert_allclose(acc, O.losses_vec(Lf), rtol=2e-6, atol=1e-12)


@settings(max_examples=6, deadline=None)
@given(shape, st.integers(0, 3), st.integers(0, 10 ** 6))
def test_batch_permutation_equivariance(sh, fi, seed):
    B, S, H, W = sh
    d = make_snippets(B, S, H, W, seed=seed % 1000)
    perm = np.random.RandomState(seed % 997).permutation(B)
    L0, G0, _ = _loss(d, O.LossConfig(**FLAGS[fi]))
    dp = dict(tgt=d['tgt'][perm], src=d['src'][perm], intrinsics=d['intrinsics'][perm], disps=[x[perm] for x in d['disps']],
              poses=d['poses'][perm], logits=[x[perm] for x in d['logits']])
    L1, G1, _ = _loss(dp, O.LossConfig(**FLAGS[fi]))
    np.testing.assert_allclose(O.losses_vec(L1), O.losses_vec(L0), rtol=2e-6, atol=1e-12)
    np.testing.assert_allclose(G1['gpose'], G0['gpose'][perm], rtol=1e-6, atol=1e-10)
    np.testing.assert_array_equal(G1['gdisp'][0], G0['gdisp'][0][perm])


@settings(max_examples=6, deadline=None)
@given(st.sampled_from([32, 40]), st.sampled_from([32, 48]), st.integers(0, 10 ** 6))
def test_out_of_view_poses_give_zero_photometric_terms(H, W, seed):
    """A translation that throws every projection out of the image: warped image 0, mask everywhere, pixel / ssim
    losses 0 and no gradient through the warp (base_model.py:96-100 with the x2 rule of transform.py:128-131)."""
    d = make_snippets(2, 2, H, W, seed=seed % 1000)
    d['poses'][...] = 0
    d['poses'][:, :, 3] = 1e3
    L, G, _ = _loss(d, O.LossConfig(smooth_reg=0.0, exp_reg=0.0, ssim_rate=0.15))
    assert L['pixel_loss'] == 0 and L['ssim_loss'] == 0 and L['total_loss'] == 0
    assert np.all(G['gpose'] == 0) and all(np.all(g == 0) for g in G['gdisp'])


def test_opt_in_gradient_argument_errors():
    d = make_snippets(2, 2, 32, 32, seed=5)
    for kw in (dict(want_image_grads=True), dict(want_intrinsics_grad=True)):
        with pytest.raises(ValueError):
            _loss(d, O.LossConfig(**FLAGS[1]), want_grads=False, **kw)
    with pytest.raises(ValueError):
        _loss(d, O.LossConfig(**FLAGS[3]), want_image_grads=True)
    _, G, _ = _loss(d, O.LossConfig(**FLAGS[3]), want_intrinsics_grad=True)
    assert G['gintrinsics'].shape == (2, 4, 3, 3) and 'gtgt' not in G
