"""Ensemble throughput: B replicas of a small grid stepped together (config['replicas'] = B) against the same B
runs one after another.

    python scripts/replicas_throughput.py [--rounds 3] [--window 0.3] [--bench-parent DIR] [--out result.json]

Per case, a batched model of B replicas and one unbatched model of the same grid are built, warmed up, and then
timed in alternating windows on the same card: CUDA events around `fib_step(ctx, ODE, n)` (no host work inside the
window), n chosen so that a window lasts about --window seconds.  B runs one after another take B times as long as
one run, so their rate is the unbatched model's.  Rates are Gcell-steps/s: replicas * height * width * time steps /
device time; medians of --rounds windows.  Every replica gets its own hole, diff and S1 column, as an ensemble
would; the batched model never runs the persistent kernel, the unbatched 512^2 4v / BR models do (one CTA per SM,
DESIGN section 3.4).  With --bench-parent DIR (a built checkout of the parent commit): `bench.py --gpus 1` on the
parent and on this tree, alternating, two runs each.  Needs a CUDA device; no fall-back."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BASE = {'dt': 0.1, 'dt_per_plot': 10, 'duration': 1, 'timeline': False, 'timeline_name': 'x', 'save_graph': False,
        'skip': False, 'cheby': False, 'ultra_slow': False}
# name, model, height, width, config extras, diff of replica 0, hole (x, y, r) or None, replica counts
CASES = [
    ('4v 512^2 + hole', 'fenton4v', 512, 512, {}, 1.5, (256, 256, 30), [8, 36, 64]),
    ('BR cheby 512^2', 'br', 512, 512, {'cheby': True}, 0.809, None, [16, 64]),
    ('Courtemanche ultra 512^2', 'court_ultra', 512, 512, {}, 1.5, None, [16]),
    ('4v 128^2', 'fenton4v', 128, 128, {}, 1.5, None, [1024]),
    ('4v CV strip 5 x 700', 'fenton4v', 5, 700, {}, 1.5, None, [10]),
]


def make(kind, H, W, extra, diff, hole, B):
    from fib_tf_b200.br import BeelerReuter
    from fib_tf_b200.court_ultra import Courtemanche
    from fib_tf_b200.fenton import Fenton4v
    cls = {'fenton4v': Fenton4v, 'br': BeelerReuter, 'court_ultra': Courtemanche}[kind]
    cfg = dict(BASE, width=W, height=H, diff=diff, **extra)
    if B > 1:
        # an ensemble: diff from 1.0 down to 0.6 times replica 0's (larger values leave the explicit scheme's
        # stability range for 4v at dt = 0.1), holes moving along the diagonal
        cfg.update(replicas=B, diff=[diff * (1.0 - 0.4 * b / (B - 1)) for b in range(B)])
    m = cls(cfg)
    if kind == 'court_ultra':
        m.chronic = True
    if hole is not None:
        x, y, r = hole
        for b in range(B):
            shift = (b * 7) % max(min(H, W) // 4, 1)
            m.add_hole_to_phase_field(x + shift, y + shift, r, replica=b if B > 1 else None)
    m.define()
    return m


def timed(m, n):
    from fib_tf_b200 import _capi
    c = m._ctx
    c.sync()
    c.timer_start()
    c.step(_capi.OP_ODE, n)
    c.timer_stop()
    return c.timer_ms() / 1000.0


def iters_for(m, window):
    t = timed(m, 20) / 20
    return max(20, int(window / max(t, 1e-7)))


def rate(m, n, t, B):
    return B * m.height * m.width * m.dt_per_step * n / t / 1e9


def bench_value(tree, args):
    cmd = [sys.executable, os.path.join(tree, 'bench.py'), '--gpus', '1', '--steps', str(args.bench_steps),
           '--warmup', '3', '--no-cpu', '--no-suite']
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=tree, timeout=1800)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith('{')]
    if r.returncode or not lines:
        raise RuntimeError('bench.py failed in %s: %s' % (tree, r.stderr[-2000:]))
    return json.loads(lines[-1])['value']


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--window', type=float, default=0.3, help='seconds per timed window')
    ap.add_argument('--bench-parent', default=None)
    ap.add_argument('--bench-steps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('replicas_throughput.py needs a CUDA device')
    from fib_tf_b200 import _capi
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    out = {'gpu': gpu, 'metric': 'Gcell-steps/s (device time, CUDA events)', 'rounds': args.rounds, 'cases': []}
    for name, kind, H, W, extra, diff, hole, counts in CASES:
        one = make(kind, H, W, extra, diff, hole, 1)
        timed(one, 20)                                                     # warm-up: module loads, graphs
        n1 = iters_for(one, args.window)
        k1 = _capi.last_kernel()
        for B in counts:
            bat = make(kind, H, W, extra, diff, hole, B)
            timed(bat, 20)
            nb = iters_for(bat, args.window)
            kb = _capi.last_kernel()
            r1, rb = [], []
            for _ in range(args.rounds):
                rb.append(rate(bat, nb, timed(bat, nb), B))
                r1.append(rate(one, n1, timed(one, n1), 1))
            bad = bat.nonfinite_cells()
            row = {'case': name, 'replicas': B, 'cells': B * H * W,
                   'batched': {'gcell_steps_s': rb, 'median': float(np.median(rb)), 'iters_per_window': nb,
                               'kernel': kb},
                   'one_after_another': {'gcell_steps_s': r1, 'median': float(np.median(r1)), 'iters_per_window': n1,
                                         'kernel': k1},
                   'speedup': float(np.median(rb) / np.median(r1)), 'nonfinite_cells': bad}
            out['cases'].append(row)
            print('%-26s B=%5d  batched %8.2f  one after another %8.2f Gcell-steps/s  x%.2f  [%s | %s]'
                  % (name, B, row['batched']['median'], row['one_after_another']['median'], row['speedup'], kb, k1),
                  flush=True)
            bat.close()
        one.close()
    if args.bench_parent:
        vals = {'parent': [], 'this': []}
        for _ in range(2):
            vals['parent'].append(bench_value(os.path.abspath(args.bench_parent), args))
            vals['this'].append(bench_value(ROOT, args))
            print('bench.py value: parent %s  this %s' % (vals['parent'], vals['this']), flush=True)
        out['bench'] = {'metric': 'Gcell-steps/s', 'steps': args.bench_steps, 'alternating': vals}
    else:
        out['bench'] = 'not measured'
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)
    print(json.dumps({'gpu': gpu}))


if __name__ == '__main__':
    main()
