"""A/B timing of the SSIM march's stage schedule: this tree against a base revision, on one GPU, in one process tree.

    python tools/ab_ssim_rows.py build [--base REV]        # needs git + nvcc, no GPU: exports REV (default HEAD~1) to
                                                           # build/ab/base and builds libsfmloss.so there and here
    python tools/ab_ssim_rows.py run [--reps 3] [--tag r3a] [--out profiles]
    python tools/ab_ssim_rows.py sweep [--tag r3a] [--out profiles]

`run` alternates `bench.py --no-cpu` (cfg2, 2000 steps, other_configs cfg1 / cfg4 / cfg5 included) between the base tree
and this one, then `bench.py --config cfg5 --no-other --no-cpu --steps 200`, `--reps` times each, and writes every bench
line plus a summary (median and spread of ms_per_step and roofline.kernel_us per build) to <out>/<tag>_ab.json.
`sweep` times the SSIM kernel of this tree at cfg2 and cfg5 for the launch policy's pick and for forced SFM_HSEG x
SFM_SSIM_NW combinations (<out>/<tag>_sweep.json).  Both record the card's name and power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = os.path.join(ROOT, 'build', 'ab', 'base')


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else 'unknown'


def build(args):
    os.makedirs(BASE, exist_ok=True)
    arch = subprocess.run(['git', '-C', ROOT, 'archive', args.base], stdout=subprocess.PIPE, check=True).stdout
    subprocess.run(['tar', '-x', '-C', BASE], input=arch, check=True)
    for tree in (BASE, ROOT):
        subprocess.run([sys.executable, '-c', 'from sfm_learner_chainer_b200 import build as B; print(B.build(force=True))'],
                       cwd=tree, check=True)


def bench(tree, extra):
    out = subprocess.run([sys.executable, os.path.join(tree, 'bench.py'), '--no-cpu'] + extra, cwd=tree,
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    if out.returncode != 0:
        raise RuntimeError('bench.py failed in %s:\n%s' % (tree, out.stderr[-3000:]))
    return json.loads(out.stdout.strip().splitlines()[-1])


def spread(xs):
    return dict(median=statistics.median(xs), min=min(xs), max=max(xs), spread=max(xs) - min(xs), runs=xs)


def run(args):
    if not os.path.exists(os.path.join(BASE, 'sfm_learner_chainer_b200', 'libsfmloss.so')):
        sys.exit('no base build: run `%s build` first' % sys.argv[0])
    trees = dict(base=BASE, new=ROOT)
    legs = dict(cfg2=[], cfg5=['--config', 'cfg5', '--no-other', '--steps', '200'])
    lines = []
    for leg, extra in legs.items():
        for k in range(args.reps):
            for label, tree in trees.items():
                line = bench(tree, extra)
                lines.append(dict(leg=leg, build=label, rep=k, line=line))
                print(leg, label, k, 'ms_per_step %.5f kernel_us %.2f' % (line['ms_per_step'], line['roofline']['kernel_us']),
                      flush=True)
    summary = {}
    for leg in legs:
        for label in trees:
            got = [r['line'] for r in lines if r['leg'] == leg and r['build'] == label]
            s = dict(ms_per_step=spread([g['ms_per_step'] for g in got]),
                     kernel_us=spread([g['roofline']['kernel_us'] for g in got]))
            for name in ('cfg1', 'cfg4', 'cfg5'):
                o = [g['other_configs'][name] for g in got if name in g.get('other_configs', {})]
                if o:
                    s['other_' + name] = dict(ms_per_step=spread([x['ms_per_step'] for x in o]),
                                              fused_kernel_us=spread([x['fused_kernel_us'] for x in o]))
            summary['%s_%s' % (leg, label)] = s
    res = dict(card=card(), base=os.path.relpath(BASE, ROOT), reps=args.reps, summary=summary, lines=lines)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, args.tag + '_ab.json'), 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(card=res['card'], summary={k: {q: (v['median'], v['spread']) for q, v in s.items() if 'median' in v}
                                                     for k, s in summary.items()})))


def sweep(args):
    sys.path.insert(0, ROOT)
    import torch
    import bench
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(0)
    cases = dict(cfg2=[None] + [(h, nw) for nw in (1, 2) for h in (8, 10, 13, 16, 19, 20, 22, 26, 32)],
                 cfg5=[None] + [(h, 1) for h in (32, 64, 96, 128, 192)])
    out = []
    for cfg, hs in cases.items():
        for forced in hs:
            for k in ('SFM_HSEG', 'SFM_SSIM_NW'):
                os.environ.pop(k, None)
            if forced:
                os.environ['SFM_HSEG'], os.environ['SFM_SSIM_NW'] = str(forced[0]), str(forced[1])
            wl = bench.Workload(cfg, dev)
            wl.capture()
            n = 400 if cfg == 'cfg2' else 40
            ms, _, _ = wl.time_steps(n, 10)
            km, kmed = wl.time_fused_kernel(n)
            r = dict(cfg=cfg, forced=forced, step_us=ms * 1e3, fused_us=km * 1e3, fused_us_median=kmed * 1e3)
            print(json.dumps(r), flush=True)
            out.append(r)
            del wl
            torch.cuda.empty_cache()
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, args.tag + '_sweep.json'), 'w') as f:
        json.dump(dict(card=card(), results=out), f, indent=1)


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    sub = ap.add_subparsers(dest='cmd', required=True)
    b = sub.add_parser('build')
    b.add_argument('--base', default='HEAD~1')
    for name in ('run', 'sweep'):
        p = sub.add_parser(name)
        p.add_argument('--tag', default='r3a')
        p.add_argument('--out', default=os.path.join(ROOT, 'profiles'))
        if name == 'run':
            p.add_argument('--reps', type=int, default=3)
    a = ap.parse_args()
    dict(build=build, run=run, sweep=sweep)[a.cmd](a)
