"""-m gpu: the SSIM march runs each stage only on the row steps whose result is used (four head steps without the later
stages, a loop that stops at the segment's last halo row).  Forced task heights put every head / tail shape through it
against the numpy oracle: (hseg + 4) mod 3 of 0, 1 and 2, segments of one to three rows, a segment that covers a whole
scale, one and two warps per task, forward records in registers and in shared memory, raw-disparity input, forward only
and the debug outputs."""
import numpy as np
import pytest

from oracle import sfm_oracle as O
from sfm_learner_chainer_b200.synthetic import make_snippets, make_raw_seam
from tests.gpu_util import to_dev, dev_inputs, host, oracle_tables, assert_grad_close

pytestmark = pytest.mark.gpu

FLAGS = dict(smooth_reg=0.1, exp_reg=0.0, ssim_rate=0.15)
# 72 rows: scale heights 72 / 36 / 18 / 9.  hseg 8: segments of 8 rows (mod 0) and the last ones of 4 / 2 / 1 rows;
# hseg 9 (mod 1): whole segments only, scale 3 in one; hseg 10 (mod 2): last segments of 2 / 6 / 8 rows, scale 3 (9
# rows) in one; hseg 64: scales 1-3 in one segment each, scale 0 = 64 + 8.
HSEGS = [8, 9, 10, 64]
_CACHE = {}


def _op(**kw):
    from sfm_learner_chainer_b200 import ViewSynthesisLoss
    return ViewSynthesisLoss(FLAGS['smooth_reg'], FLAGS['exp_reg'], FLAGS['ssim_rate'], **kw)


def _data():
    if 'd' not in _CACHE:
        d = make_snippets(2, 2, 72, 136, seed=301, harsh=True)
        L, G, _ = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], None, O.LossConfig(**FLAGS))
        _CACHE['d'] = (d, L, G)
    return _CACHE['d']


def _force(monkeypatch, hseg, nw=None, srec=None):
    monkeypatch.setenv('SFM_HSEG', str(hseg))
    for k, v in (('SFM_SSIM_NW', nw), ('SFM_SSIM_SREC', srec)):
        monkeypatch.setenv(k, v) if v is not None else monkeypatch.delenv(k, raising=False)


def _check(losses, grads, L, G, ns=4):
    np.testing.assert_allclose(host(losses), O.losses_vec(L), rtol=1e-5, atol=1e-9)
    assert_grad_close(host(grads['gposes']), G['gpose'], what='gpose')
    for s in range(ns):
        assert_grad_close(host(grads['gdisps'][s]), G['gdisp'][s], what='gdisp[%d]' % s)


@pytest.mark.parametrize('hseg', HSEGS)
@pytest.mark.parametrize('nw,srec', [('1', '1'), ('1', '0'), ('2', '1'), ('2', '0')])
def test_forced_task_heights_match_oracle(hseg, nw, srec, monkeypatch):
    d, L, G = _data()
    g = dev_inputs(d)
    _force(monkeypatch, hseg, nw, srec)
    losses, grads = _op().forward_backward(g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], None)
    _check(losses, grads, L, G)
    # forward only: the instance without the gradient stages
    l2 = _op().forward(g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], None)
    np.testing.assert_allclose(host(l2), O.losses_vec(L), rtol=1e-5, atol=1e-9)


@pytest.mark.parametrize('hseg', HSEGS)
def test_forced_task_heights_raw_disparity(hseg, monkeypatch):
    d, _, _ = _data()
    raw_disps, _ = make_raw_seam(d, (1, 4), seed=302)
    L, G, _ = O.sfm_loss_raw(d['tgt'], d['src'], d['intrinsics'], raw_disps, d['poses'], None, O.LossConfig(**FLAGS),
                             raw_disp_scales=0xF)
    _force(monkeypatch, hseg)
    op = _op(raw_disp_scales=0xF)
    losses, grads = op.forward_backward(to_dev(d['tgt']), to_dev(d['src']), to_dev(d['intrinsics']),
                                        [to_dev(x) for x in raw_disps], to_dev(d['poses']), None)
    _check(losses, grads, L, G)


@pytest.mark.parametrize('hseg', HSEGS)
def test_forced_task_heights_debug_bit_exact(hseg, monkeypatch):
    d, _, _ = _data()
    proj, kinv = oracle_tables(O, d)
    L, _, dbg = O.sfm_loss(d['tgt'], d['src'], d['intrinsics'], d['disps'], d['poses'], None, O.LossConfig(**FLAGS),
                           want_grads=False, want_debug=True,
                           proj_override=np.concatenate([proj, np.zeros_like(proj[..., :1, :])], -2), kinv_override=kinv)
    g = dev_inputs(d)
    _force(monkeypatch, hseg)
    losses, gd = _op().forward(g['tgt'], g['src'], g['intrinsics'], g['disps'], g['poses'], None,
                               proj=to_dev(proj), kinv=to_dev(kinv), debug=True)
    for s in range(4):
        np.testing.assert_array_equal(host(gd['u0'][s]), dbg['u0'][s], err_msg='u0 scale %d' % s)
        np.testing.assert_array_equal(host(gd['v0'][s]), dbg['v0'][s], err_msg='v0 scale %d' % s)
        np.testing.assert_array_equal(host(gd['inb'][s]).astype(bool), dbg['inb'][s], err_msg='inb scale %d' % s)
        np.testing.assert_array_equal(host(gd['P'][s]), dbg['P'][s], err_msg='warped image scale %d' % s)
    np.testing.assert_allclose(host(losses), O.losses_vec(L), rtol=1e-5, atol=1e-9)
