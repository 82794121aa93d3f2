"""bench.py contract checks that need no GPU: the reference arm's JSON line (numpy oracle on the host cores) and the
loud failure of the B200 arm when there is no CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, OMP_NUM_THREADS='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '1', '--steps', '2',
                          '--warmup', '1', '--config', 'cfg1'], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                         env=env, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['unit'] == 'Mpix/s' and line['higher_is_better'] is True
    assert line['metric'].startswith('fwd+bwd warp+photometric loss Mpix/s')
    assert line['value'] > 0 and line['cpu_baseline']['value'] == line['value'] and line['cpu_baseline']['kind'] == 'port'
    assert line['cpu_baseline']['cores'] >= 1 and 'sample' in line['cpu_baseline']
    assert line['e2e'] == dict(value=line['value'], unit='Mpix/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert line['gpu_launches'] == 0 and line['config']['workload'].startswith('cfg1')
    sys.path.insert(0, ROOT)
    import bench
    assert line['config'] == bench.config_dict('cfg1', 1)          # the same `config` object as the B200 arm prints


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '2'],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, timeout=120, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ''


def test_b200_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip('a CUDA device is present')
    env = {k: v for k, v in os.environ.items() if k not in ('WORLD_SIZE', 'RANK', 'LOCAL_RANK')}
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '3'], stdout=subprocess.PIPE, env=env,
                         stderr=subprocess.PIPE, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0
    assert 'no CUDA device' in (out.stderr + out.stdout) and 'no CPU fallback' in (out.stderr + out.stdout)


def test_byte_models_match_survey_section_8d():
    sys.path.insert(0, ROOT)
    import bench
    pix = 4 * bench.pyramid_pixels(128, 416)
    assert pix == 282880
    assert abs(bench.bytes_strict(4, 2, 128, 416, False) / pix - 35.1) < 0.05            # A-strict, S=2, no exp
    assert abs(bench.bytes_strict(32, 4, 128, 416, True) / (8 * pix) - 85.2) < 0.05       # A-strict, S=4, exp
    assert bench.bytes_fused_kernel(4, 2, 128, 416, False) == 44 * pix                    # kernel model 44 B/pix
    assert bench.bytes_fused_kernel(32, 4, 128, 416, True) == 100 * 8 * pix               # 100 B/pix


def test_b200_arm_rejects_a_gpu_count_that_is_not_the_world_size():
    env = {k: v for k, v in os.environ.items() if k not in ('WORLD_SIZE', 'RANK', 'LOCAL_RANK')}
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '2', '--steps', '3'], stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode != 0 and 'torch.distributed.run' in (out.stderr + out.stdout)


def test_timed_steps_are_exactly_K_with_grouped_graphs():
    """bench.replay_timed_steps: K steps from graphs of G consecutive steps when K is a multiple of G and nothing
    runs between the steps; one graph per step otherwise.  Either way every buffer set is visited in rotation."""
    sys.path.insert(0, ROOT)
    import bench

    class Graph(object):
        def __init__(self, log, sets):
            self.log, self.sets = log, sets

        def replay(self):
            self.log.extend(self.sets)

    class Runner(object):
        def __init__(self, nsets, G):
            self.log, self.nsets, self.group = [], nsets, G
            self.group_graphs = [Graph(self.log, list(range(k, k + G))) for k in range(0, nsets, G)] if G > 1 else None

        def step(self, k):
            self.log.append(k % self.nsets)

    r = Runner(28, 4)
    assert bench.replay_timed_steps(r, 20, 3, None, False) == 4
    assert len(r.log) == 20 and r.log == [(4 + k) % 28 for k in range(20)]      # starts at the first group boundary after the warm-up
    assert r.last % 28 == r.log[-1]                                             # --dump-outputs reads the last step's buffer set
    r = Runner(28, 4)
    assert bench.replay_timed_steps(r, 2000, 50, None, False) == 4
    assert len(r.log) == 2000 and set(r.log) == set(range(28))
    assert all(b == (a + 1) % 28 for a, b in zip(r.log, r.log[1:]))              # consecutive steps never share a buffer set
    assert r.last % 28 == r.log[-1]
    for args in ((21, 3, None, False), (20, 3, None, True), (20, 3, lambda k: None, False)):
        r = Runner(28, 4)
        assert bench.replay_timed_steps(r, *args) == 1
        assert r.log == [(3 + k) % 28 for k in range(args[0])]
    r = Runner(3, 1)
    assert bench.replay_timed_steps(r, 20, 3, None, False) == 1 and len(r.log) == 20


def test_dump_outputs_keeps_small_arrays_whole_and_samples_within_the_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 64 * 1024)
    rs = np.random.RandomState(0)
    arrays = dict(losses=rs.standard_normal(5).astype(np.float32), gposes=rs.standard_normal((4, 2, 6)).astype(np.float32),
                  gdisp0=rs.standard_normal((4, 1, 64, 208)).astype(np.float32),
                  gdisp1=rs.standard_normal((4, 1, 32, 104)).astype(np.float32))
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == ['gdisp0.npy', 'gdisp1.npy', 'gposes.npy', 'losses.npy']
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 64 * 1024
    for f in files:
        a, b = np.load(tmp_path / 'a' / f), np.load(tmp_path / 'b' / f)
        assert a.dtype == np.float32
        np.testing.assert_array_equal(a, b)                                      # the same sample every time
    for name in ('losses', 'gposes'):
        np.testing.assert_array_equal(np.load(tmp_path / 'a' / (name + '.npy')), arrays[name])
    big = np.load(tmp_path / 'a' / 'gdisp0.npy')
    assert big.ndim == 1 and 0 < big.size < arrays['gdisp0'].size
    assert np.isin(big, arrays['gdisp0']).all()


def test_bench_rejects_a_step_count_below_one_and_dumps_of_the_reference_arm():
    for extra in (['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'x']):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, stdout=subprocess.PIPE,
                             stderr=subprocess.PIPE, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and out.stdout == '', out.stderr[-2000:]
