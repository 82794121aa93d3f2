"""Step time of the fused loss with and without one opt-in option: image_grads (ViewSynthesisLoss(image_grads=True)),
intrinsics_grad (ViewSynthesisLoss(intrinsics_grad=True)), snippet_terms (ViewSynthesisLoss(snippet_terms=True) with
per-snippet weights, returning the per-snippet losses), pixel_terms (ViewSynthesisLoss(pixel_terms=True) with random
per-pixel weights in [0, 1] at every scale, returning the per-pixel loss maps) or min_reprojection
(ViewSynthesisLoss(min_reprojection=True), auto-masking on, returning the selection maps; not with the explainability
branch, so its default configs are cfg1, cfg2 and cfg5), full_res_multiscale (ViewSynthesisLoss(full_res_multiscale=True),
Monodepth2's full-resolution photometric terms at every scale; default configs cfg1, cfg2 and cfg5) or
full_res_min_reprojection (min_reprojection with and without full_res_multiscale; default configs cfg2 and cfg5),
mean_norm_smooth (ViewSynthesisLoss(mean_norm_smooth=True), Monodepth2's mean-normalised second-order smoothness),
mean_norm_smooth_edge (the same with edge-aware smoothness on both sides), edge_mean_abs (edge-aware smoothness with and
without Monodepth2's edge weight) or monodepth2 (full_res_multiscale + min_reprojection + edge-aware smoothness with and
without mean_norm_smooth + edge_mean_abs: Monodepth2's whole loss against the same step with the reference's smoothness);
the last four have default configs cfg2 and cfg5.  border_padding (ViewSynthesisLoss(border_padding=True), Monodepth2's
image borders) and monodepth2_border (Monodepth2's whole loss, as the second variant of monodepth2, with and without
border_padding) have default configs cfg2 and cfg5 too.

For each config the step (forward_backward on device tensors) is captured four times into one CUDA graph and the graph
is replayed; the two variants alternate, and the median over the repeats is reported per step.  Prints one JSON line
per config and writes them all, with the card name and its power limit, to the file given as the first argument.
The last column is the relative overhead for image_grads and the added microseconds for intrinsics_grad (the cost of
one extra dependent launch, sfm_intrinsics_grad_kernel) and for snippet_terms, the relative overhead for pixel_terms and
min_reprojection, full_res_multiscale and full_res_min_reprojection, the added microseconds for the next four and the
relative overhead for border_padding and monodepth2_border.
usage: python tools/time_opt_in_grads.py OUT.json {image_grads,intrinsics_grad,snippet_terms,pixel_terms,min_reprojection,
       full_res_multiscale,full_res_min_reprojection,mean_norm_smooth,mean_norm_smooth_edge,edge_mean_abs,monodepth2,
       border_padding,monodepth2_border}
       [cfg ...]"""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from sfm_learner_chainer_b200 import ViewSynthesisLoss
from sfm_learner_chainer_b200.synthetic import CONFIGS, make_snippets

STEPS_PER_GRAPH = 4
# option -> the column that compares the two step times (plain, with)
LAST_COLUMN = {
    'image_grads': ('overhead', lambda p, q: round(q / p - 1.0, 4)),
    'intrinsics_grad': ('extra_us', lambda p, q: round(q - p, 2)),
    'snippet_terms': ('extra_us', lambda p, q: round(q - p, 2)),
    'pixel_terms': ('overhead', lambda p, q: round(q / p - 1.0, 4)),
    'min_reprojection': ('overhead', lambda p, q: round(q / p - 1.0, 4)),
    'full_res_multiscale': ('overhead', lambda p, q: round(q / p - 1.0, 4)),
    'full_res_min_reprojection': ('overhead', lambda p, q: round(q / p - 1.0, 4)),
    'mean_norm_smooth': ('extra_us', lambda p, q: round(q - p, 2)),
    'mean_norm_smooth_edge': ('extra_us', lambda p, q: round(q - p, 2)),
    'edge_mean_abs': ('extra_us', lambda p, q: round(q - p, 2)),
    'monodepth2': ('extra_us', lambda p, q: round(q - p, 2)),
    'border_padding': ('overhead', lambda p, q: round(q / p - 1.0, 4)),
    'monodepth2_border': ('overhead', lambda p, q: round(q / p - 1.0, 4)),
}
EDGE = dict(edge_aware_smooth=True)
MONODEPTH2 = dict(full_res_multiscale=True, min_reprojection=True, edge_aware_smooth=True)
MONODEPTH2_SMOOTH = dict(MONODEPTH2, mean_norm_smooth=True, edge_mean_abs=True)
# operator options of the two variants where they are not (nothing, {option: True})
VARIANTS = {'full_res_min_reprojection': (dict(min_reprojection=True), dict(min_reprojection=True, full_res_multiscale=True)),
            'mean_norm_smooth_edge': (EDGE, dict(EDGE, mean_norm_smooth=True)),
            'edge_mean_abs': (EDGE, dict(EDGE, edge_mean_abs=True)),
            'monodepth2': (MONODEPTH2, MONODEPTH2_SMOOTH),
            'monodepth2_border': (MONODEPTH2_SMOOTH, dict(MONODEPTH2_SMOOTH, border_padding=True))}
DEFAULT_CONFIGS = {'min_reprojection': ['cfg1', 'cfg2', 'cfg5'], 'full_res_multiscale': ['cfg1', 'cfg2', 'cfg5'],
                   'full_res_min_reprojection': ['cfg2', 'cfg5'], 'mean_norm_smooth': ['cfg2', 'cfg5'],
                   'mean_norm_smooth_edge': ['cfg2', 'cfg5'], 'edge_mean_abs': ['cfg2', 'cfg5'], 'monodepth2': ['cfg2', 'cfg5'],
                   'border_padding': ['cfg2', 'cfg5'], 'monodepth2_border': ['cfg2', 'cfg5']}


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    return q


def make_graph(op, args, **kw):
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        for _ in range(3):
            losses, _ = op.forward_backward(*args, **kw)
        side.synchronize()
        assert torch.isfinite(losses).all()
        with torch.cuda.graph(graph, stream=side):
            for _ in range(STEPS_PER_GRAPH):
                op.forward_backward(*args, **kw)
    torch.cuda.synchronize()
    return graph


def time_graph(graph, replays):
    graph.replay()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(replays):
        graph.replay()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / (replays * STEPS_PER_GRAPH)


def main():
    if len(sys.argv) < 3 or sys.argv[2] not in LAST_COLUMN:
        sys.exit(__doc__)
    out, option = sys.argv[1:3]
    names = sys.argv[3:] or DEFAULT_CONFIGS.get(option, ['cfg1', 'cfg2', 'cfg4', 'cfg5'])
    torch.cuda.set_device(0)
    rows = []
    for name in names:
        c = CONFIGS[name]
        d = make_snippets(c['B'], c['S'], c['H'], c['W'], seed=0)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        flags = dict(smooth_reg=c['smooth_reg'], exp_reg=c['exp_reg'], ssim_rate=c['ssim_rate'])
        args = (dev(d['tgt']), dev(d['src']), dev(d['intrinsics']), [dev(x) for x in d['disps']], dev(d['poses']),
                [dev(x) for x in d['logits']] if c['exp_reg'] else None)
        # the operators own the workspaces the graphs write: they live as long as the graphs
        base_kw, option_kw = VARIANTS.get(option, ({}, {option: True}))
        ops = {'plain': ViewSynthesisLoss(**base_kw, **flags), option: ViewSynthesisLoss(**option_kw, **flags)}
        # snippet_terms: weights of a padded batch (the last snippet weighs 0)
        w = torch.full((c['B'],), 1.0, device='cuda')
        w[-1] = 0.0
        kw = {option: dict(snippet_weights=w)} if option == 'snippet_terms' else {}
        if option == 'pixel_terms':
            # pixel_terms: a weight in [0, 1] for every (pixel, source) of every scale; the maps are always returned
            gen = torch.Generator(device='cuda').manual_seed(0)
            pw = [torch.rand((c['B'], c['S'], c['H'] >> s, c['W'] >> s), device='cuda', generator=gen) for s in range(4)]
            kw = {option: dict(pixel_weights=pw)}
        graphs = {k: make_graph(op, args, **kw.get(k, {})) for k, op in ops.items()}
        replays = 10 if name == 'cfg5' else 200
        t = {k: [] for k in graphs}
        for _ in range(7):
            for k, g in graphs.items():
                t[k].append(time_graph(g, replays))
        row = dict(cfg=name, B=c['B'], S=c['S'], H=c['H'], W=c['W'],
                   **{k + '_us': round(float(np.median(v)), 2) for k, v in t.items()},
                   **{k + '_spread_us': round(float(np.max(v) - np.min(v)), 2) for k, v in t.items()})
        key, compare = LAST_COLUMN[option]
        row[key] = compare(row['plain_us'], row[option + '_us'])
        print(json.dumps(row), flush=True)
        rows.append(row)
        del graphs, ops, g
        torch.cuda.empty_cache()
    with open(out, 'w') as f:
        json.dump(dict(card=card(), steps_per_graph=STEPS_PER_GRAPH, rows=rows), f, indent=1)


if __name__ == '__main__':
    main()
