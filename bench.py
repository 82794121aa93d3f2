#!/usr/bin/env python
"""bench.py -- fwd+bwd warp+photometric loss throughput of the view-synthesis loss path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config cfg2] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one pass of the hot path (pyramid / tables / smoothness prologue + fused loss forward+backward + epilogue,
single sweep) over one batch of synthetic KITTI-shaped snippets.  Default workload = BASELINE.json configs[1]
(sfm_learner_v1_ssim.yml loss path: SSIM + L1 + smoothness, B=4, S=2, 128x416, 4 scales) per GPU; under N GPUs the
batch is sharded by snippet (weak scaling for `value`: 4 snippets per rank, B_global = 4N) and the path's one
collective -- the 5-float loss-partial all-reduce, sfm_allreduce_partials of the C ABI -- runs EVERY step inside the
timed CUDA-event interval (captured in the step's CUDA graph).

Prints ONE JSON line (rank 0).  Keys beyond the driver's contract:
  roofline        dominant kernel (fused loss): SURVEY 8(d) A-strict bytes / its own duration (CUDA events recorded by
                  the library around that launch) vs the measured HBM copy peak; the pyramid-as-input byte model and
                  the ncu DRAM traffic of the same kernel ride along as extra keys
  roofline_step   whole step vs A-strict
  cpu_baseline    the numpy oracle (port of the reference's numpy/Chainer CPU path) on this box's cores
  e2e             same metric through the C-ABI host-buffer entry point (H2D + kernels + D2H every step)
  other_configs   device-timed numbers for the remaining single-GPU BASELINE shapes (cfg1, cfg4, cfg5)
  strong_scaling  (N > 1) the split the north star names: cfg4 with a GLOBAL batch of 32 (32/N snippets per GPU) and, at
                  N = 8, cfg5 with a global batch of 64, each without a collective, with the per-step loss all-reduce,
                  and with a 159.5 MB stand-in CNN-gradient all-reduce running next to it
"""
import argparse
import ctypes as C
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

from sfm_learner_chainer_b200.synthetic import make_snippets, CONFIGS

METRIC = 'fwd+bwd warp+photometric loss Mpix/s at 128x416'
UNIT = 'Mpix/s'
FALLBACK_HBM_GBS = 6650.0


def pyramid_pixels(H, W, n_scales=4):
    return sum((H >> s) * (W >> s) for s in range(n_scales))


def bytes_strict(B, S, H, W, exp):
    """SURVEY 8(d) A-strict: full-res images once + disp r/w + logits r/w + poses + K."""
    pix = pyramid_pixels(H, W)
    return 4 * (B * (1 + S) * 3 * H * W + 2 * B * pix + (2 * B * S * pix if exp else 0)) + 48 * B * S + 144 * B


def bytes_fused_kernel(B, S, H, W, exp):
    """SURVEY 8(d) secondary model (pyramid as the kernel's input): 4*B*sum_hw*(3 + 3S + 2 + exp*2S)."""
    return 4 * B * pyramid_pixels(H, W) * (3 + 3 * S + 2 + (2 * S if exp else 0))


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return FALLBACK_HBM_GBS, 'fallback (B200_PROFILING.md 6.65 TB/s)'


# ---------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the numpy oracle on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_oracle_run(cfg_name, n_iters, threads):
    """Times fwd+bwd of the numpy restatement of the reference path, sharded by snippet over a thread
    pool (numpy releases the GIL in its array loops).  Returns seconds per step (all B snippets)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import sfm_oracle as O                                  # the timed CPU baseline
    c = dict(CONFIGS[cfg_name])
    B, S, H, W = c.pop('B'), c.pop('S'), c.pop('H'), c.pop('W')
    d = make_snippets(B, S, H, W, seed=0)
    cfg = O.LossConfig(B_global=B, **c)

    def one(b):
        sl = slice(b, b + 1)
        return O.sfm_loss(d['tgt'][sl], d['src'][sl], d['intrinsics'][sl], [x[sl] for x in d['disps']],
                          d['poses'][sl], [x[sl] for x in d['logits']], cfg)[0]

    # every (step, snippet) pair is an independent unit of host work: all of them go through one thread pool so
    # that the arm uses every host core it can even when B is smaller than the core count
    threads = max(1, min(threads, B * max(1, n_iters)))
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(one, range(min(B, threads))))                        # warm-up (page-in, caches)
        t0 = time.perf_counter()
        list(ex.map(one, [b for _ in range(n_iters) for b in range(B)]))
        sec = (time.perf_counter() - t0) / n_iters
    return float(sec), threads, (B, S, H, W)


def config_dict(cfg_name, world):
    """The `config` object of the JSON line -- identical in the B200 arm and the reference arm (same workload)."""
    c = CONFIGS[cfg_name]
    pix = c['B'] * pyramid_pixels(c['H'], c['W'])
    return dict(workload='%s: %s' % (cfg_name, describe(cfg_name)), per_gpu_batch=c['B'], global_batch=c['B'] * world,
                sources=c['S'], H=c['H'], W=c['W'], n_scales=4,
                units='target-pyramid pixels = B * sum_s h_s*w_s (%d per step per GPU)' % pix,
                l2_policy='inputs and outputs rotated over ceil(2 x L2 / A-strict) + 1 buffer sets (more than twice the L2 '
                          'capacity in total), so consecutive steps never find their inputs in L2',
                snippets='4 distinct seeded snippets, tiled to the batch size (separate buffers per tile)')


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    ncpu = os.cpu_count() or 1
    c = CONFIGS[args.config]
    sec, threads, (B, S, H, W) = cpu_oracle_run(args.config, max(1, args.steps), ncpu)
    pix = B * pyramid_pixels(H, W)
    val = pix / sec / 1e6
    sample = '%d full %s steps (B=%d, S=%d, %dx%d, 4 scales), (step, snippet) units over a pool of %d threads' % (
        max(1, args.steps), args.config, B, S, H, W, threads)
    line = dict(impl='reference', metric=METRIC, value=val, unit=UNIT, n_gpus=args.gpus, steps=max(1, args.steps),
                warmup=args.warmup, ms_per_step=sec * 1e3, higher_is_better=True, scaling='weak', vs_baseline=None,
                dtype='f32', data='synthetic',
                config=config_dict(args.config, max(1, int(os.environ.get('WORLD_SIZE', args.gpus)))),
                note='numpy restatement (oracle/) of the reference numpy/Chainer CPU path on the host cores; '
                     'chainer==4.0.0b1 is not installable in this image.  Rank 0 alone runs it (one batch of the per-GPU size)',
                cpu_baseline=dict(value=val, unit=UNIT, cores=threads, kind='port', sample=sample),
                e2e=dict(value=val, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))


def describe(name):
    c = CONFIGS[name]
    return 'B=%d S=%d %dx%d 4 scales, smooth_reg=%g exp_reg=%g ssim_rate=%g' % (
        c['B'], c['S'], c['H'], c['W'], c['smooth_reg'], c['exp_reg'], c['ssim_rate'])


# ---------------------------------------------------------------------------------------------
# clocks (pynvml sampler thread)
# ---------------------------------------------------------------------------------------------
class ClockSampler(object):
    REASONS = {0x1: 'gpu_idle', 0x2: 'applications_clocks_setting', 0x4: 'sw_power_cap', 0x8: 'hw_slowdown',
               0x10: 'sync_boost', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown', 0x100: 'display_clock_setting'}

    def __init__(self, index):
        self.samples = []
        self.ok = False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:                                          # noqa: BLE001
            self.err = repr(e)
            self.max_mhz = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _sample(self):
        nv = self.nv
        return (time.perf_counter(), nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self._sample())
            except Exception:                                           # noqa: BLE001
                pass
            time.sleep(0.01)

    def start(self):
        if self.ok:
            self.t.start()

    def stop(self):
        self._stop.set()
        if self.ok:
            self.t.join()

    def summary(self, t0, t1):
        if not self.ok:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvml unavailable: %s' % getattr(self, 'err', '')])
        inside = [s for s in self.samples if t0 <= s[0] <= t1] or [s for s in self.samples if s[0] >= t0][:1] \
            or self.samples[-1:]
        mhz = float(np.median([s[1] for s in inside])) if inside else None
        mask = 0
        for s in inside:
            mask |= s[2]
        reasons = [n for b, n in self.REASONS.items() if mask & b and n != 'gpu_idle']
        return dict(sm_mhz=mhz, sm_max_mhz=float(self.max_mhz), reasons=reasons, samples=len(inside))


# ---------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------
STEPS_PER_GRAPH = 4


def capture_step_graphs(torch, side, nsets, launch, error_mode='global', allow_groups=True):
    """-> (one graph per buffer set, G, graphs of G consecutive steps each or None).  A trainer captures the loss path
    inside its own step graph, between the CNN forward and backward: there the path's three kernels follow their
    neighbours at kernel-to-kernel latency.  Replaying ONE step per graph adds a graph-to-graph launch boundary
    (~4.5 us on B200) to every step that the path does not have in place; graphs of G = STEPS_PER_GRAPH consecutive
    steps (distinct buffer sets, nothing shared between the steps) pay it once per G steps.  Both figures are
    reported (`timing.one_step_per_graph`)."""
    singles = []
    for k in range(nsets):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side, capture_error_mode=error_mode):
            launch(k, torch.cuda.current_stream())
        singles.append(g)
    G = next((c for c in (STEPS_PER_GRAPH, 2) if nsets % c == 0), 1) if allow_groups else 1
    if os.environ.get('SFM_BENCH_STEPS_PER_GRAPH'):
        G = int(os.environ['SFM_BENCH_STEPS_PER_GRAPH'])
        G = G if (G >= 1 and nsets % G == 0) else 1
    groups = None
    if G > 1:
        groups = []
        for k0 in range(0, nsets, G):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=side, capture_error_mode=error_mode):
                for k in range(k0, k0 + G):
                    launch(k, torch.cuda.current_stream())
            groups.append(g)
    torch.cuda.synchronize()
    return singles, G, groups


def replay_timed_steps(runner, steps, first, per_step, one_step_per_graph):
    """The K timed steps: graphs of G consecutive steps when K is a multiple of G (and nothing runs between the steps),
    else one graph (or one direct call) per step.  Returns the steps per graph used."""
    G = runner.group if runner.group_graphs else 1
    if G > 1 and not one_step_per_graph and per_step is None and steps % G == 0:
        g0 = (first + G - 1) // G
        for j in range(steps // G):
            runner.group_graphs[(g0 + j) % len(runner.group_graphs)].replay()
        runner.last = G * g0 + steps - 1                     # the groups start at the first group boundary >= first
        return G
    for k in range(steps):
        runner.step(first + k)
        if per_step:
            per_step(first + k)
    return 1


class Workload(object):
    """Pre-packed C-ABI calls over `nsets` rotating buffer sets (inputs AND outputs), so that with a
    working set below the 126 MB L2 consecutive steps still touch HBM."""

    def __init__(self, cfg_name, device, B_global=None, min_rotation_bytes=None, B_local=None, seed=0):
        import torch
        from sfm_learner_chainer_b200 import lib as L
        self.torch, self.L = torch, L
        self.lib = L.load()
        c = dict(CONFIGS[cfg_name])
        B, S, H, W = c.pop('B'), c.pop('S'), c.pop('H'), c.pop('W')
        if B_local:
            B = B_local
        self.B, self.S, self.H, self.W, self.flags = B, S, H, W, c
        self.exp = c['exp_reg'] != 0
        self.A_strict = bytes_strict(B, S, H, W, self.exp)
        self.A_kernel = bytes_fused_kernel(B, S, H, W, self.exp)
        self.pix = B * pyramid_pixels(H, W)
        l2 = torch.cuda.get_device_properties(device).L2_cache_size
        rot = min_rotation_bytes if min_rotation_bytes is not None else 2 * l2
        self.nsets = max(2, int(math.ceil(rot / float(self.A_strict))) + 1)
        self.l2_bytes = l2
        nb = min(B, 4)
        base = make_snippets(nb, S, H, W, seed=seed)
        rep = lambda a: np.ascontiguousarray(np.concatenate([a] * (B // nb) + [a[:B % nb]], 0)) if B != nb else a
        self.host = dict(tgt=rep(base['tgt']), src=rep(base['src']), intrinsics=rep(base['intrinsics']),
                         disps=[rep(x) for x in base['disps']], poses=rep(base['poses']),
                         logits=[rep(x) for x in base['logits']])
        self.desc = L.SfmDesc(B, S, H, W, 4, int(B_global or 0), c['smooth_reg'], c['exp_reg'], c['ssim_rate'], 0)
        nws = self.lib.sfm_workspace_bytes(C.byref(self.desc))
        dev = lambda a: torch.from_numpy(a).to(device)
        self.sets = []
        # the loss partials of all buffer sets live in one tensor (row k = set k) so that the multi-GPU run can
        # all-reduce the partials of `nsets` consecutive steps with one NCCL call
        self.all_losses = torch.zeros(self.nsets, 8, device=device)
        for k in range(self.nsets):
            t = dict(tgt=dev(self.host['tgt']), src=dev(self.host['src']), K=dev(self.host['intrinsics']),
                     disps=[dev(x) for x in self.host['disps']], poses=dev(self.host['poses']),
                     logits=[dev(x) for x in self.host['logits']] if self.exp else None,
                     gdisps=[torch.empty_like(dev(x)) for x in self.host['disps']],
                     gposes=torch.empty((B, S, 6), device=device),
                     glogits=[torch.empty((B, S, H >> s, W >> s), device=device) for s in range(4)] if self.exp else None,
                     losses=self.all_losses[k],
                     ws=torch.empty(nws + 256, dtype=torch.uint8, device=device))
            inp, g = L.SfmInputs(), L.SfmGrads()
            inp.tgt, inp.src, inp.intrinsics, inp.poses = (t['tgt'].data_ptr(), t['src'].data_ptr(), t['K'].data_ptr(),
                                                           t['poses'].data_ptr())
            g.gposes = t['gposes'].data_ptr()
            for s in range(4):
                inp.disps[s] = t['disps'][s].data_ptr()
                g.gdisps[s] = t['gdisps'][s].data_ptr()
                if self.exp:
                    inp.logits[s] = t['logits'][s].data_ptr()
                    g.glogits[s] = t['glogits'][s].data_ptr()
            t['inp'], t['g'] = inp, g
            t['wsp'] = C.c_void_p((t['ws'].data_ptr() + 255) // 256 * 256)
            self.sets.append(t)
        self.graphs, self.group, self.group_graphs = None, 1, None

    def launch(self, k, stream, peer=None):
        t = self.sets[k % self.nsets]
        if peer is not None:      # the epilogue kernel completes the five losses across the ranks over NVLink peer memory
            rc = self.lib.sfm_loss_forward_backward_peer(C.byref(self.desc), C.byref(t['inp']), C.c_void_p(t['losses'].data_ptr()),
                                                         C.byref(t['g']), t['wsp'], peer.handle, C.c_void_p(stream))
        else:
            rc = self.lib.sfm_loss_forward_backward(C.byref(self.desc), C.byref(t['inp']), C.c_void_p(t['losses'].data_ptr()),
                                                    C.byref(t['g']), t['wsp'], C.c_void_p(stream))
        if rc:
            self.L.check(rc)

    def capture(self):
        """One CUDA graph per buffer set (prologue + fused + epilogue kernel nodes), and graphs of STEPS_PER_GRAPH
        consecutive steps (consecutive buffer sets) for the timed loops: see steps_per_graph()."""
        torch = self.torch
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for k in range(self.nsets):
                self.launch(k, side.cuda_stream)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        self.graphs, self.group, self.group_graphs = capture_step_graphs(
            torch, side, self.nsets, lambda k, st: self.launch(k, st.cuda_stream))

    def step(self, k):
        if self.graphs is not None:
            self.graphs[k % self.nsets].replay()
        else:
            self.launch(k, self.torch.cuda.current_stream().cuda_stream)

    def outputs(self, k):
        """What a caller of step k receives, copied to the host: the five losses and every gradient."""
        t = self.sets[k % self.nsets]
        out = dict(losses=t['losses'][:5], gposes=t['gposes'])
        for s in range(4):
            out['gdisp%d' % s] = t['gdisps'][s]
            if self.exp:
                out['glogits%d' % s] = t['glogits'][s]
        return {name: v.cpu().numpy() for name, v in out.items()}

    def time_steps(self, steps, warmup, per_step=None, one_step_per_graph=False):
        torch = self.torch
        for k in range(warmup):
            self.step(k)
            if per_step:
                per_step(k)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        replay_timed_steps(self, steps, warmup, per_step, one_step_per_graph)
        e1.record()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        return e0.elapsed_time(e1) / steps, t0, t1

    def time_fused_kernel(self, n=200):
        """Average device duration of the fused loss kernel alone (events recorded by the library right
        around its launch, on the launching stream)."""
        torch = self.torch
        st = torch.cuda.current_stream()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
        for k in range(5):
            self.launch(k, st.cuda_stream)
        torch.cuda.synchronize()
        # torch creates its cudaEvent_t lazily on first record(); record once so the handles exist
        for a, b in evs:
            a.record(); b.record()
        torch.cuda.synchronize()
        for k, (a, b) in enumerate(evs):
            self.lib.sfm_set_kernel_events(C.c_void_p(a.cuda_event), C.c_void_p(b.cuda_event))
            self.launch(k, st.cuda_stream)
        self.lib.sfm_set_kernel_events(None, None)
        torch.cuda.synchronize()
        ts = sorted(a.elapsed_time(b) for a, b in evs)
        return float(np.mean(ts)), float(ts[len(ts) // 2])


def run_e2e(cfg_name, device, n_ctx=3, u8=False, min_steps=200, min_seconds=0.5, repeats=3):
    """Same metric through the host-buffer C-ABI entry point: pinned host inputs -> H2D -> prologue + fused fwd+bwd ->
    D2H of the five losses and every gradient, EVERY step.  `n_ctx` host contexts are used alternately
    (sfm_loss_step_host_submit / _wait), the way a data loader keeps the next step's copies in flight while the
    current one computes; n_ctx=1 is the fully synchronous call.  u8: the step is fed by decoded uint8 frames
    (sfm_loss_step_host_u8_submit; the reference's real data layer, datasets/kitti/kitti_raw_dataset.py:12-14).
    Each repeat runs at least `min_steps` steps and `min_seconds` of wall time whatever --steps says; the MEDIAN of
    `repeats` repeats is returned.  -> dict(value Mpix/s, h2d, d2h, steps, h2d_gbs, repeats=[...])."""
    import torch
    from sfm_learner_chainer_b200 import lib as L
    lib = L.load()
    c = dict(CONFIGS[cfg_name])
    B, S, H, W = c.pop('B'), c.pop('S'), c.pop('H'), c.pop('W')
    exp = c['exp_reg'] != 0
    d = make_snippets(min(B, 4), S, H, W, seed=1)
    if B > 4:
        rep = lambda a: np.ascontiguousarray(np.concatenate([a] * (B // 4) + [a[:B % 4]], 0))
        d = dict(tgt=rep(d['tgt']), src=rep(d['src']), intrinsics=rep(d['intrinsics']), disps=[rep(x) for x in d['disps']],
                 poses=rep(d['poses']), logits=[rep(x) for x in d['logits']])
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()

    def pin_group(arrs):
        """The arrays of one kind (four scales) as views of ONE pinned buffer, scale s+1 right behind scale s: the
        library then moves them in a single copy (every copy has a fixed cost of several microseconds)."""
        buf = torch.empty(sum(a.size for a in arrs), dtype=torch.float32).pin_memory()
        out, off = [], 0
        for a in arrs:
            v = buf[off:off + a.size].view(*a.shape)
            v.copy_(torch.from_numpy(np.ascontiguousarray(a)))
            out.append(v)
            off += a.size
        return out
    hin = dict(tgt=pin(d['tgt']), src=pin(d['src']), K=pin(d['intrinsics']), poses=pin(d['poses']),
               disps=pin_group(d['disps']), logits=pin_group(d['logits']))
    desc = L.SfmDesc(B, S, H, W, 4, 0, c['smooth_reg'], c['exp_reg'], c['ssim_rate'], 0)
    inp = L.SfmInputs()
    inp.tgt, inp.src, inp.intrinsics, inp.poses = hin['tgt'].data_ptr(), hin['src'].data_ptr(), hin['K'].data_ptr(), hin['poses'].data_ptr()
    h2d = hin['tgt'].numel() * 4 + hin['src'].numel() * 4 + hin['K'].numel() * 4 + hin['poses'].numel() * 4
    d2h = 5 * 4 + hin['poses'].numel() * 4
    for s in range(4):
        inp.disps[s] = hin['disps'][s].data_ptr()
        h2d += hin['disps'][s].numel() * 4
        d2h += hin['disps'][s].numel() * 4
        if exp:
            inp.logits[s] = hin['logits'][s].data_ptr()
            h2d += hin['logits'][s].numel() * 4
            d2h += hin['logits'][s].numel() * 4
    if u8:
        # data-layer entry: decoded uint8 frames + augmentation draws instead of float images (sfm_ingest_u8 on the device)
        from sfm_learner_chainer_b200.functions import draw_augmentation
        rs = np.random.RandomState(2)
        imgs = np.concatenate([d['tgt'][:, None], d['src']], 1)
        frames = pin(np.clip(np.round((imgs.transpose(0, 1, 3, 4, 2) + 1) * 127.5), 0, 255).astype(np.uint8))
        K0 = pin(d['intrinsics'][:, 0].copy())
        aug = (L.SfmAugment * B)()
        for b in range(B):
            a = draw_augmentation(H, W, rs)
            aug[b] = L.SfmAugment(a['out_h'], a['out_w'], a['off_y'], a['off_x'], 1 if a['flip'] else 0, 0, a['x_scaling'], a['y_scaling'])
        h2d += frames.numel() + K0.numel() * 4 + C.sizeof(aug) - (hin['tgt'].numel() + hin['src'].numel() + hin['K'].numel()) * 4
    ctxs, outs, grads = [], [], []
    try:
        for k in range(n_ctx):
            ctx = C.c_void_p()
            L.check(lib.sfm_host_ctx_create(C.byref(desc), C.byref(ctx)))
            ctxs.append(ctx)
            ho = dict(gdisps=pin_group([np.zeros_like(x) for x in d['disps']]), glogits=pin_group([np.zeros_like(x) for x in d['logits']]),
                      gposes=pin(np.empty_like(d['poses'])), losses=pin(np.zeros(8, np.float32)))
            g = L.SfmGrads()
            g.gposes = ho['gposes'].data_ptr()
            for s in range(4):
                g.gdisps[s] = ho['gdisps'][s].data_ptr()
                if exp:
                    g.glogits[s] = ho['glogits'][s].data_ptr()
            outs.append(ho)
            grads.append(g)

        def run(n):
            for k in range(n):
                j = k % n_ctx
                if k >= n_ctx:
                    L.check(lib.sfm_loss_step_host_wait(ctxs[j]))      # the step submitted n_ctx steps ago: its results are on the host
                if u8:
                    L.check(lib.sfm_loss_step_host_u8_submit(ctxs[j], C.c_void_p(frames.data_ptr()), C.c_void_p(K0.data_ptr()), aug,
                                                             C.byref(inp), C.c_void_p(outs[j]['losses'].data_ptr()), C.byref(grads[j])))
                else:
                    L.check(lib.sfm_loss_step_host_submit(ctxs[j], C.byref(inp), C.c_void_p(outs[j]['losses'].data_ptr()), C.byref(grads[j])))
            for j in range(n_ctx):
                L.check(lib.sfm_loss_step_host_wait(ctxs[j]))
        run(3 * n_ctx)
        torch.cuda.synchronize()
        # size a repeat: at least min_steps steps and min_seconds of wall time
        t0 = time.perf_counter()
        run(20)
        per = (time.perf_counter() - t0) / 20
        steps = int(max(min_steps, math.ceil(min_seconds / max(per, 1e-7))))
        secs = []
        for _ in range(repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            run(steps)
            secs.append((time.perf_counter() - t0) / steps)
        loss = float(outs[(steps - 1) % n_ctx]['losses'][0])
    finally:
        for ctx in ctxs:
            lib.sfm_host_ctx_destroy(ctx)
    pix = B * pyramid_pixels(H, W)
    med = float(np.median(secs))
    return dict(value=pix / med / 1e6, h2d=h2d, d2h=d2h, steps=steps, h2d_gbs=h2d / med / 1e9, loss=loss,
                repeats=[pix / t / 1e6 for t in secs])


KERNEL_SOURCES = ('common.cuh', 'kernels.h', 'fused_loss.cu', 'ssim_march.cuh', 'prep.cu', 'smooth.cu', 'smooth_task.cuh')


def csrc_sha():
    """Short hash of the KERNEL sources (not the host-side api.cu / comm.cu): profiles/ncu_latest.json records the one it
    was captured with, so a stale capture is not quoted as the traffic of the kernels that run now."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, 'sfm_learner_chainer_b200', 'csrc')
    for f in KERNEL_SOURCES:
        h.update(open(os.path.join(d, f), 'rb').read())
    return h.hexdigest()[:16]


def fused_kernel_name(c):
    return 'sfm_ssim_march_kernel' if (c['ssim_rate'] and not c['exp_reg']) else 'sfm_l1_march_kernel'


def ncu_traffic(cfg_name):
    """dram__bytes_read.sum + dram__bytes_write.sum of the fused kernel from the committed ncu --set full capture
    of THIS source state (tools/ncu_to_json.py), else (None, why)."""
    try:
        prof = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_latest.json')))
    except Exception as e:                                            # noqa: BLE001
        return None, None, 'profiles/ncu_latest.json unreadable: %r' % (e,)
    ent = prof.get(cfg_name)
    if not ent:
        return None, None, 'no capture of %s in profiles/ncu_latest.json' % cfg_name
    if prof.get('csrc_sha') != csrc_sha():
        return None, ent, 'stale: captured with kernel sources %s, running %s' % (prof.get('csrc_sha'), csrc_sha())
    if fused_kernel_name(CONFIGS[cfg_name]) not in ent.get('kernel', ''):
        return None, ent, 'capture is of %s, not of %s' % (ent.get('kernel'), fused_kernel_name(CONFIGS[cfg_name]))
    return ent.get('dram_bytes'), ent, 'ncu --set full capture of this source state (profiles/ncu_latest.json)'


class StepRunner(object):
    """A Workload replayed as CUDA graphs, optionally with the path's collective (sfm_allreduce_partials) captured
    with every step:
      mode 'inline'   the all-reduce of step k's partials follows step k's epilogue on the same stream (the next step
                      starts after it: its latency is exposed every step);
      mode 'overlap'  the graph of step k forks a branch that all-reduces the partials of step k-1 (another buffer set)
                      while step k's kernels run, and joins it at the end -- the way a trainer consumes the reduced
                      losses one iteration late; `finish()` reduces the last step's partials, so every step's partials
                      are reduced inside the timed interval;
      mode 'peer'     no collective call at all: `comm` is a PeerLossSum and the step's own epilogue kernel sums the
                      partials over NVLink peer memory (sfm_loss_forward_backward_peer)."""

    def __init__(self, wl, comm=None, mode='inline'):
        self.wl, self.comm = wl, comm
        self.mode = mode if comm is not None else None
        self.graphs, self.group, self.group_graphs = None, 1, None
        self.last = None
        self.timed_steps_per_graph = 1
        if self.mode == 'overlap':
            torch = wl.torch
            self.side2 = torch.cuda.Stream()

    def _allreduce(self, k, stream):
        wl = self.wl
        t = wl.sets[k % wl.nsets]
        wl.L.check(wl.lib.sfm_allreduce_partials(self.comm._comm, C.c_void_p(t['losses'].data_ptr()), 5, C.c_void_p(stream)))

    def _launch(self, k, stream_obj):
        torch = self.wl.torch
        stream = stream_obj.cuda_stream
        if self.mode == 'overlap':
            fork, join = torch.cuda.Event(), torch.cuda.Event()
            fork.record(stream_obj)
            self.side2.wait_event(fork)
            self._allreduce(k - 1, self.side2.cuda_stream)          # previous step's partials (another buffer set)
            join.record(self.side2)
            self.wl.launch(k, stream)
            stream_obj.wait_event(join)
        elif self.mode == 'peer':
            self.wl.launch(k, stream, self.comm)
        else:
            self.wl.launch(k, stream)
            if self.mode == 'inline':
                self._allreduce(k, stream)

    def capture(self):
        torch = self.wl.torch
        wl = self.wl
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for k in range(wl.nsets):
                self._launch(k, side)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        # thread-local capture mode: torch's NCCL watchdog thread may query events while this thread captures.  Steps that
        # fork an NCCL branch keep one step per graph
        self.graphs, self.group, self.group_graphs = capture_step_graphs(
            torch, side, wl.nsets, lambda k, st: self._launch(k, st), 'thread_local', allow_groups=self.mode in (None, 'peer'))

    def step(self, k):
        if self.graphs is not None:
            self.graphs[k % self.wl.nsets].replay()
        else:
            self._launch(k, self.wl.torch.cuda.current_stream())
        self.last = k

    def finish(self):
        """overlap mode: the partials of the last step are still unreduced."""
        if self.mode == 'overlap' and self.last is not None:
            self._allreduce(self.last, self.wl.torch.cuda.current_stream().cuda_stream)

    def time(self, steps, warmup, per_step=None, before_stop=None, one_step_per_graph=False):
        """ms per step between two CUDA events on the launching stream (all of a step's kernels, and the captured
        all-reduce, are on it or joined into it); `before_stop` runs right before the stop event (e.g. waits for
        side-stream work)."""
        torch = self.wl.torch
        for k in range(warmup):
            self.step(k)
            if per_step:
                per_step(k)
        self.finish()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        self.timed_steps_per_graph = replay_timed_steps(self, steps, warmup, per_step, one_step_per_graph)
        self.finish()
        if before_stop:
            before_stop()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps, t0, time.perf_counter()

    def reduced_rows_ok(self, world):
        """Every rank holds the same synthetic snippets, so a reduced row of partials must be world x the local row.
        Runs one rotation of the buffer sets (+1 step in overlap mode) and compares against plain local steps."""
        torch = self.wl.torch
        wl = self.wl
        n = wl.nsets
        for k in range(n + (1 if self.mode == 'overlap' else 0)):
            self.step(k)
        torch.cuda.synchronize()
        red = wl.all_losses[:, :5].clone()
        plain = StepRunner(wl)
        for k in range(n):
            plain.step(k)
        torch.cuda.synchronize()
        rows = slice(1, n) if self.mode == 'overlap' else slice(0, n)      # overlap: row 0 was rewritten by the extra step
        return bool(torch.allclose(red[rows], wl.all_losses[rows, :5] * world, rtol=1e-5, atol=1e-8))


def trace(msg):
    if os.environ.get('SFM_BENCH_TRACE'):
        sys.stderr.write('[bench rank %s %.1f] %s\n' % (os.environ.get('RANK', '0'), time.perf_counter() % 1000, msg))
        sys.stderr.flush()


def max_over_ranks(ms, device, world):
    if world == 1:
        return ms
    import torch
    import torch.distributed as dist
    t = torch.tensor([ms], device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def strong_scaling_block(args, device, world, rank, comm, peer, peak):
    """The split the north star names (SURVEY 8(e)): a FIXED global batch sharded by snippet.  Per workload: the
    single-GPU time of the whole batch (measured on every rank, the slowest is reported), then the shard of 1/N of
    it per GPU (i) with no collective, (ii) with the five loss partials summed across the ranks inside every step's
    epilogue kernel over NVLink peer memory (the product path: no collective call), (iii) with an NCCL all-reduce of
    every step captured behind the step (its latency exposed), (iv) with that all-reduce captured as a parallel
    branch of the NEXT step's graph, (v) as (ii) with a 159.5 MB fp32 all-reduce -- the size of the DispNet + PoseNet
    gradient (39.9 M parameters, SURVEY 7.6) -- issued every step on NCCL's own stream next to it, the way the
    trainer's gradient exchange would run; every interval ends when all of its collectives have finished."""
    import torch
    import torch.distributed as dist
    out = {}
    names = ['cfg4'] + (['cfg5'] if world >= 8 else [])
    steps = max(20, min(args.steps, 200))
    for name in names:
        c = CONFIGS[name]
        Bg = c['B']
        if Bg % world:
            out[name] = dict(skipped='global batch %d is not divisible by %d ranks' % (Bg, world))
            continue
        ent = dict(workload=describe(name), global_batch=Bg, per_gpu_batch=Bg // world, steps=steps)
        # ---- one GPU, whole batch
        w1 = Workload(name, device)
        r1 = StepRunner(w1)
        r1.capture()
        ms1, _, _ = r1.time(steps, 5)
        ms1 = max_over_ranks(ms1, device, world)
        ent['single_gpu_us_per_step'] = ms1 * 1e3
        del r1, w1
        torch.cuda.empty_cache()
        # ---- the shard
        wl = Workload(name, device, B_global=Bg, B_local=Bg // world)
        dist.barrier()
        res = {}
        for mode in ('no_collective', 'loss_sum_in_epilogue_kernel_over_peer_memory', 'nccl_allreduce_inline', 'nccl_allreduce_overlapped',
                     'loss_sum_in_epilogue_kernel_plus_159MB_gradient_allreduce'):
            rmode = 'peer' if mode.startswith('loss_sum_in_epilogue') else ('inline' if mode == 'nccl_allreduce_inline' else 'overlap')
            if rmode == 'peer' and peer is None:
                res[mode] = dict(skipped='no peer access between the GPUs (CUDA IPC)')
                continue
            cm = None if mode == 'no_collective' else (peer if rmode == 'peer' else comm)
            runner = StepRunner(wl, cm, rmode)
            how = {'inline': 'NCCL all-reduce of step k captured behind step k\'s epilogue (exposed)',
                   'overlap': 'NCCL all-reduce of step k-1 captured as a parallel branch of step k\'s graph',
                   'peer': 'no collective call: the epilogue kernel of every step exchanges the partials over NVLink peer memory'}[rmode]
            try:
                runner.capture()
            except Exception as exc:                                   # noqa: BLE001 -- NCCL refused the capture: call it per step
                runner = StepRunner(wl, cm, 'inline')
                how = 'direct call per step (graph capture failed: %s)' % str(exc)[:80]
            per_step, before_stop = None, None
            if mode.endswith('gradient_allreduce'):
                grad = torch.zeros(39_880_000, device=device)           # 159.5 MB fp32 (SURVEY 7.6)
                works = []

                def per_step(k, grad=grad, works=works):
                    if len(works) >= 2:
                        works.pop(0).wait()
                    works.append(dist.all_reduce(grad, async_op=True))

                def before_stop(works=works):
                    while works:
                        works.pop(0).wait()                             # the compute stream waits for NCCL's stream
            dist.barrier()
            torch.cuda.synchronize()
            trace('%s %s: timing' % (name, mode))
            ms, _, _ = runner.time(steps, 5, per_step, before_stop)
            ms = max_over_ranks(ms, device, world)
            res[mode] = dict(us_per_step=ms * 1e3, global_mpix_s=Bg * pyramid_pixels(c['H'], c['W']) / (ms * 1e-3) / 1e6,
                             efficiency_vs_single_gpu=ms1 / (world * ms), collective=how if cm is not None else None)
            if not mode.endswith('gradient_allreduce') and cm is not None:
                res[mode]['reduced_equals_world_x_local'] = runner.reduced_rows_ok(world)
            del runner
            if mode.endswith('gradient_allreduce'):
                del grad
        ent.update(res)
        ent['roofline_per_gpu_us'] = bytes_strict(Bg // world, c['S'], c['H'], c['W'], c['exp_reg'] != 0) / peak / 1e3
        out[name] = ent
        del wl
        torch.cuda.empty_cache()
    return out


DUMP_LIMIT_BYTES = 64 * 1000 * 1000
NPY_HEADER_BYTES = 128


def dump_outputs(out_dir, arrays):
    """Writes {name: array} as out_dir/<name>.npy in float32, at most DUMP_LIMIT_BYTES in all.  Smaller arrays are kept
    whole; an array larger than its share of the remaining budget is cut to that many elements, taken at positions drawn
    with a seed derived from its name and kept in flat order, so the same configuration always yields the same sample."""
    import zlib
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_LIMIT_BYTES - NPY_HEADER_BYTES * len(arrays)
    items = sorted(arrays.items(), key=lambda kv: (kv[1].size, kv[0]))
    for i, (name, a) in enumerate(items):
        a = np.asarray(a, np.float32)
        share = budget // (len(items) - i) // a.itemsize                  # elements
        if a.size > share:
            idx = np.random.RandomState(zlib.crc32(name.encode())).choice(a.size, share, replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        budget -= a.nbytes
        np.save(os.path.join(out_dir, name + '.npy'), a)


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.gpus != world:
        raise SystemExit('bench.py: --gpus %d but WORLD_SIZE=%d: launch N > 1 as `python -m torch.distributed.run --nnodes=1 '
                         '--nproc-per-node N --master-addr 127.0.0.1 bench.py --gpus N ...` (one process per GPU)' % (args.gpus, world))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the view-synthesis loss path has no CPU fallback)')
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    comm = peer = None
    if world > 1:
        dist.init_process_group('nccl', device_id=device)
        from sfm_learner_chainer_b200.distributed import LossPartialsComm
        comm = LossPartialsComm(rank, world)                 # the C ABI's NCCL communicator (sfm_comm_create): the library-call baseline
        from sfm_learner_chainer_b200.distributed import PeerLossSum
        # slot arrays for the in-kernel sum over NVLink peer memory (CUDA IPC).  Every rank must agree on whether it
        # worked: without peer access between the GPUs the bench falls back to the NCCL all-reduce on all ranks.
        peer_err = ''
        try:
            peer = PeerLossSum(rank, world, barrier=lambda: None)
        except Exception as exc:                              # noqa: BLE001
            peer, peer_err = None, str(exc)[:200]
        flag = torch.tensor([1 if peer is not None else 0], device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0 and peer is not None:
            peer._lib.sfm_peer_destroy(peer._peer)
            peer._peer = None
            peer = None
        if peer is not None:
            peer._barrier = lambda: dist.barrier()
        dist.barrier()
    n_gpus = world
    peak, peak_src = measured_peak()

    c = CONFIGS[args.config]
    wl = Workload(args.config, device, B_global=c['B'] * world)
    use_comm = (peer if peer is not None else comm) if (world > 1 and not args.no_allreduce) else None
    if world > 1:
        dist.barrier()                                        # the ranks enter their first (peer-synchronised) steps together
    if use_comm is not None and use_comm is peer:
        runner = StepRunner(wl, use_comm, 'peer')
        collective_how = ('summed across the ranks inside every step\'s epilogue kernel over NVLink peer memory '
                          '(sfm_loss_forward_backward_peer; no collective call, no extra launch)')
    else:
        runner = StepRunner(wl, use_comm, 'overlap')
        collective_how = ('all-reduced by sfm_allreduce_partials (NCCL), the call of step k-1 captured as a parallel branch of step '
                          'k\'s graph (the in-kernel peer-memory sum is unavailable here: %s)' % peer_err) if use_comm else None
    if not args.no_graph:
        runner.capture()
    elif use_comm is not None and use_comm is not peer:
        runner = StepRunner(wl, use_comm, 'inline')
    trace('captured: %s' % collective_how)
    sampler = ClockSampler(local)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms, t0, t1 = runner.time(args.steps, args.warmup)
    torch.cuda.synchronize()
    trace('timed %.4f ms' % ms)
    # the steps below reuse the buffer sets: take the last timed step's results now, write them at the end
    dumped = wl.outputs(runner.last) if args.dump_outputs and rank == 0 else None
    steps_per_graph = runner.timed_steps_per_graph
    ms_single = ms
    if steps_per_graph > 1:                                   # the same K steps replayed one step per graph, for comparison
        if world > 1:
            dist.barrier()
        ms_single, _, _ = runner.time(args.steps, args.warmup, one_step_per_graph=True)
        torch.cuda.synchronize()
        ms_single = max_over_ranks(ms_single, device, world)
    allreduce_ok = runner.reduced_rows_ok(world) if use_comm is not None else None
    trace('check %s' % allreduce_ok)
    if world > 1:
        dist.barrier()
    ms = max_over_ranks(ms, device, world)
    # The timed region is short (K steps of ~40 us under the driver's flags); the identical steps keep running for
    # ~0.25 s right after it so that the 10 ms clock sampler sees the GPU under this load.
    t_region = t1 - t0
    n_fill = int(min(20000, max(1, 0.25 / (ms * 1e-3))))    # the same count on every rank (ms is the max over ranks): the steps carry a collective
    for k in range(n_fill):
        runner.step(k)
        if k % 64 == 63:
            torch.cuda.synchronize()
    runner.finish()
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    sampler.stop()
    clocks = sampler.summary(t0, t1)
    clocks['window'] = ('the timed region (%.1f ms) plus %.0f ms of the identical steps run right after it: the sampler polls '
                        'every 10 ms' % (t_region * 1e3, (t1 - t0 - t_region) * 1e3))

    total_pix = wl.pix * world
    value = total_pix / (ms * 1e-3) / 1e6
    n_launch = 3                                             # prologue (pyramid + tables + smoothness tasks), fused loss, epilogue
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=n_gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=ms, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic',
                config=config_dict(args.config, world),
                timing=dict(buffer_sets=wl.nsets, rotation_mb=wl.nsets * wl.A_strict / 1e6, l2_mb=wl.l2_bytes / 1e6,
                            launch=('CUDA graph replay, %d consecutive step(s) per graph (each step = %d kernel nodes: prologue = pyramid + '
                                    'tables + smoothness tasks; fused loss; epilogue; programmatic dependent launches between them; '
                                    'consecutive steps use distinct buffer sets and share nothing)' % (steps_per_graph, n_launch))
                            if not args.no_graph else 'direct C-ABI calls',
                            steps_per_graph=steps_per_graph,
                            one_step_per_graph=dict(ms_per_step=ms_single, value=wl.pix * world / (ms_single * 1e-3) / 1e6,
                                                    note='the same K steps with a graph-to-graph launch boundary behind every step '
                                                         '(the figure of the earlier rounds); inside a trainer\'s own step graph the '
                                                         'path has kernel-to-kernel boundaries only'),
                            parallelism=('snippet-sharded x%d (weak scaling: %d snippets per GPU, B_global = %d), no data-path '
                                         'collective call; the five loss partials of EVERY step are %s' % (
                                             world, wl.B, wl.B * world, collective_how)) if world > 1 else 'single GPU',
                            timer='CUDA events on the launching stream around the K steps, barrier + synchronize on both sides, max over ranks'),
                clocks=clocks, gpu_launches=n_launch * args.steps)
    if allreduce_ok is not None:
        line['loss_allreduce_check'] = allreduce_ok

    if rank == 0:
        # ---- roofline of the dominant kernel (fused loss), events around the kernel itself
        k_mean, k_med = wl.time_fused_kernel(200)
        ach = wl.A_strict / (k_mean * 1e-3) / 1e9
        traffic, ncu_ent, traffic_note = ncu_traffic(args.config)
        line['roofline'] = dict(bound='hbm', achieved=ach, peak=peak, unit='GB/s', frac=ach / peak, traffic=traffic,
                                kernel=fused_kernel_name(c), kernel_us=k_mean * 1e3, kernel_us_median=k_med * 1e3,
                                algorithmic_bytes=wl.A_strict, peak_source=peak_src,
                                byte_model='SURVEY 8(d) A-strict (the whole step\'s compulsory bytes: full-res images once + disp r/w + '
                                           'logits r/w + poses + K) over the fused kernel\'s own duration',
                                kernel_model=dict(algorithmic_bytes=wl.A_kernel, frac=wl.A_kernel / (k_mean * 1e-3) / 1e9 / peak,
                                                  byte_model='secondary model of SURVEY 8(d): 4*B*sum_hw*(3 + 3S + 2 + exp*2S), '
                                                             'the images of every scale as the kernel\'s input'),
                                traffic_source=traffic_note, ncu=ncu_ent,
                                note='at B=4 the roofline time is ~1.5 us (below one launch): latency-bound by construction; '
                                     'other_configs holds the bandwidth-relevant shapes.  The fused kernels are issue-bound '
                                     '(SSIM) / issue- and L1-wavefront-bound (L1), not HBM-bound (DESIGN.md section 5)')
        ach_s = wl.A_strict / (ms * 1e-3) / 1e9
        line['roofline_step'] = dict(bound='hbm', achieved=ach_s, peak=peak, unit='GB/s', frac=ach_s / peak,
                                     algorithmic_bytes=wl.A_strict,
                                     byte_model='A-strict: full-res images once + disp r/w + logits r/w + poses + K')
        line['step_share_of_fused_kernel'] = k_mean / ms if world == 1 else None
    del runner
    if world == 1:
        # ---- e2e through the host-buffer C-ABI entry point (primary: the uint8-frame data layer the reference really has)
        e8 = run_e2e(args.config, device, n_ctx=8, u8=True)
        ef = run_e2e(args.config, device, n_ctx=8)
        es = run_e2e(args.config, device, n_ctx=1, repeats=1)
        line['e2e'] = dict(value=e8['value'], unit=UNIT, h2d_bytes_per_step=e8['h2d'], d2h_bytes_per_step=e8['d2h'],
                           steps_per_repeat=e8['steps'], repeats=e8['repeats'], h2d_gbs=e8['h2d_gbs'],
                           api='sfm_loss_step_host_u8_submit/_wait, eight host contexts in rotation (pinned host buffers, the four scales of a kind '
                               'back to back so that they travel as one copy; every step: '
                               'H2D of the decoded uint8 frames, K, augmentation draws, disparities, poses; ingest + prologue + fused '
                               'fwd+bwd + epilogue; D2H of the five losses and every gradient).  Median of three repeats of '
                               '>= 200 steps and >= 0.5 s each',
                           float_images=dict(value=ef['value'], h2d_bytes_per_step=ef['h2d'], d2h_bytes_per_step=ef['d2h'],
                                             repeats=ef['repeats'], h2d_gbs=ef['h2d_gbs'],
                                             api='sfm_loss_step_host_submit/_wait: float32 images in (4 bytes per sample), eight contexts'),
                           synchronous=dict(value=es['value'], api='sfm_loss_step_host, one step at a time, float32 images'))
        # ---- other single-GPU BASELINE shapes, device timed
        if not args.no_other:
            others = {}
            del wl
            torch.cuda.empty_cache()
            for name in ('cfg1', 'cfg4', 'cfg5'):
                if name == args.config:
                    continue
                w2 = Workload(name, device)
                w2.capture()
                oms, _, _ = w2.time_steps(48, 5)
                oms1, _, _ = w2.time_steps(48, 5, one_step_per_graph=True)
                km, _ = w2.time_fused_kernel(50)
                others[name] = dict(workload=describe(name), ms_per_step=oms, value=w2.pix / (oms * 1e-3) / 1e6, unit=UNIT,
                                    steps_per_graph=w2.group if 48 % w2.group == 0 else 1, ms_per_step_one_step_per_graph=oms1,
                                    step_frac_of_hbm_peak=w2.A_strict / (oms * 1e-3) / 1e9 / peak,
                                    fused_kernel_us=km * 1e3,
                                    fused_kernel_frac_of_hbm_peak=w2.A_strict / (km * 1e-3) / 1e9 / peak,
                                    fused_kernel_frac_kernel_model=w2.A_kernel / (km * 1e-3) / 1e9 / peak)
                del w2
                torch.cuda.empty_cache()
            line['other_configs'] = others
        # ---- CPU baseline: bounded sample of the same workload on the host cores
        if not args.no_cpu:
            n_iters = 12 if args.config in ('cfg1', 'cfg2') else 1
            sec, threads, (B, S, H, W) = cpu_oracle_run(args.config, n_iters, 1)
            line['cpu_baseline'] = dict(value=B * pyramid_pixels(H, W) / sec / 1e6, unit=UNIT, cores=threads, kind='port',
                                        sample='%d full %s steps of the numpy oracle (scalar port, 1 thread), mean' % (n_iters, args.config),
                                        ms_per_step=sec * 1e3)
    else:
        # e2e at N GPUs: every rank runs the host-buffer path on its shard; aggregate = total pixels / slowest rank
        trace('e2e')
        dist.barrier()
        e8 = run_e2e(args.config, device, n_ctx=8, u8=True, repeats=3)
        t = torch.tensor([wl.pix / e8['value']], device=device)      # us per step on this rank (pix / Mpix/s)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        line['e2e'] = dict(value=total_pix / float(t.item()), unit=UNIT, h2d_bytes_per_step=e8['h2d'] * world,
                           d2h_bytes_per_step=e8['d2h'] * world, steps_per_repeat=e8['steps'],
                           api='sfm_loss_step_host_u8_submit/_wait on every rank (its snippet shard, eight host contexts); '
                               'median of three repeats of >= 200 steps and >= 0.5 s; total pixels / slowest rank')
        del wl
        torch.cuda.empty_cache()
        if not args.no_other:
            ss = strong_scaling_block(args, device, world, rank, comm, peer, peak)
            if rank == 0:
                line['strong_scaling'] = ss
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        if comm is not None:
            import gc
            gc.collect()                                       # graphs that captured the all-reduce go first
            comm.close()
        if peer is not None:
            peer.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=2000)
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', default='cfg2', choices=sorted(CONFIGS))
    ap.add_argument('--no-graph', action='store_true', help='direct C-ABI calls instead of CUDA graph replay')
    ap.add_argument('--no-other', action='store_true', help='skip the other_configs sweep (N = 1) / the strong_scaling block (N > 1)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-allreduce', action='store_true', help='(diagnostic) skip the loss-partial allreduce at N > 1')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed (rank 0: losses.npy, gposes.npy, gdisp<s>.npy, glogits<s>.npy '
                         'with explainability) as float32 .npy files into DIR, at most 64 MB in all; the inputs are seeded, so '
                         'runs with the same arguments compare output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs is for the b200 arm')
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == 'reference':
        if args.steps > 20:
            args.steps = 20            # bounded sample: each step is ~0.2-0.8 s of host work
        if args.steps < 8:
            args.steps = 8             # enough (step, snippet) units to occupy the host cores
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
