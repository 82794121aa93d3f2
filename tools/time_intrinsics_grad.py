"""Step time of the fused loss with and without the intrinsics gradient (ViewSynthesisLoss(intrinsics_grad=True)).

For each config the step (forward_backward on device tensors) is captured four times into one CUDA graph and the graph
is replayed; the two variants alternate, and the median over the repeats is reported per step.  Prints one JSON line
per config and writes them all, with the card name and its power limit, to the file given as the first argument.
The difference is the cost of the extra dependent launch (sfm_intrinsics_grad_kernel) inside a graph.
usage: python tools/time_intrinsics_grad.py OUT.json [cfg ...]"""
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


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                       stdout=subprocess.PIPE, text=True).stdout.strip()
    return q


def make_graph(op, args):
    side = torch.cuda.Stream()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        for _ in range(3):
            losses, _ = op.forward_backward(*args)
        side.synchronize()
        assert torch.isfinite(losses).all()
        with torch.cuda.graph(graph, stream=side):
            for _ in range(STEPS_PER_GRAPH):
                op.forward_backward(*args)
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
    out = sys.argv[1]
    names = sys.argv[2:] or ['cfg1', 'cfg2', 'cfg4', 'cfg5']
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
        ops = {'plain': ViewSynthesisLoss(**flags), 'intrinsics_grad': ViewSynthesisLoss(intrinsics_grad=True, **flags)}
        graphs = {k: make_graph(op, args) for k, op in ops.items()}
        replays = 10 if name == 'cfg5' else 200
        t = {k: [] for k in graphs}
        for _ in range(7):
            for k, g in graphs.items():
                t[k].append(time_graph(g, replays))
        row = dict(cfg=name, B=c['B'], S=c['S'], H=c['H'], W=c['W'],
                   **{k + '_us': round(float(np.median(v)), 2) for k, v in t.items()},
                   **{k + '_spread_us': round(float(np.max(v) - np.min(v)), 2) for k, v in t.items()})
        row['extra_us'] = round(row['intrinsics_grad_us'] - row['plain_us'], 2)
        print(json.dumps(row), flush=True)
        rows.append(row)
        del graphs, ops, g
        torch.cuda.empty_cache()
    with open(out, 'w') as f:
        json.dump(dict(card=card(), steps_per_graph=STEPS_PER_GRAPH, rows=rows), f, indent=1)


if __name__ == '__main__':
    main()
