"""Device time of an ODE iteration with the activation maps armed and unarmed (fib_activation_watch), per
kernel family at 4096^2 and for BASELINE configs 1 and 2 (512^2, the persistent kernel).

    python scripts/activation_overhead.py [--iters 40] [--rounds 5] [--out result.json]

Armed and unarmed windows alternate on the same context (`--rounds` of each); every switch is followed by
one untimed iteration (the iteration graph is rebuilt).  A window is CUDA-event timed (fib_timer_*) over
`--iters` iterations; the result is the median per iteration.  Needs a CUDA device; no fall-back."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

BASE = {'dt': 0.1, 'dt_per_plot': 10, 'duration': 1, 'timeline': False, 'timeline_name': 'x', 'save_graph': False,
        'skip': False, 'cheby': False, 'ultra_slow': False}
N = 4096
CASES = [
    # name, model class, config, hole
    ('4v, one step per launch', 'fenton', dict(width=N, height=N, diff=1.5, steps_per_launch=1), False),
    ('4v, two steps per launch', 'fenton', dict(width=N, height=N, diff=1.5, steps_per_launch=2), False),
    ('BR cheby', 'br', dict(width=N, height=N, diff=0.809, cheby=True), False),
    ('BR exact', 'br', dict(width=N, height=N, diff=0.809), False),
    ('Courtemanche all-state (court_ultra)', 'court_ultra', dict(width=N, height=N, diff=1.5), False),
    ('Courtemanche all-state LUT (court_ultra)', 'court_ultra', dict(width=N, height=N, diff=1.5, lut=True), False),
    ('Courtemanche multi-rate fast op (court)', 'court', dict(width=N, height=N, diff=1.5), False),
    ('BASELINE config 1: 4v 512^2 (persistent)', 'fenton', dict(width=512, height=512, diff=1.5), True),
    ('BASELINE config 2: BR 512^2 cheby (persistent)', 'br', dict(width=512, height=512, diff=0.809, cheby=True), True),
]


def model_of(kind, cfg, hole):
    from fib_tf_b200.br import BeelerReuter
    from fib_tf_b200.court import Courtemanche
    from fib_tf_b200.court_ultra import Courtemanche as CourtemancheUltra
    from fib_tf_b200.fenton import Fenton4v
    cls = {'fenton': Fenton4v, 'br': BeelerReuter, 'court': Courtemanche, 'court_ultra': CourtemancheUltra}[kind]
    m = cls(dict(BASE, **cfg))
    if hole:
        m.add_hole_to_phase_field(256, 256, 30)
    m.define()
    return m


def window(ctx, iters):
    ctx.timer_start()
    ctx.step(0, iters)
    ctx.timer_stop()
    return ctx.timer_ms() / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('activation_overhead.py needs a CUDA device')
    from fib_tf_b200 import _capi
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv'], capture_output=True,
                         text=True).stdout.strip()
    rows = []
    for name, kind, cfg, hole in CASES:
        m = model_of(kind, cfg, hole)
        ctx = m._ctx
        ctx.step(0, 3)                                            # warm-up: graphs, lazy module loads
        off, on, kernels = [], [], set()
        for _ in range(args.rounds):
            m.watch_activation()
            ctx.step(0, 1)
            on.append(window(ctx, args.iters))
            kernels.add(_capi.last_kernel())
            m.stop_activation()
            ctx.step(0, 1)
            off.append(window(ctx, args.iters))
            kernels.add(_capi.last_kernel())
        t_off, t_on = float(np.median(off)), float(np.median(on))
        rows.append({'case': name, 'cells': m.height * m.width, 'dt_per_step': m.dt_per_step,
                     'unarmed_ms_per_iter': t_off, 'armed_ms_per_iter': t_on,
                     'overhead_pct': 100.0 * (t_on - t_off) / t_off,
                     'unarmed_spread_pct': 100.0 * (max(off) - min(off)) / t_off,
                     'armed_spread_pct': 100.0 * (max(on) - min(on)) / t_on, 'kernels': sorted(kernels)})
        print('%-48s unarmed %.4f ms  armed %.4f ms per iteration  %+.2f %%  (spread %.2f / %.2f %%)'
              % (name, t_off, t_on, rows[-1]['overhead_pct'], rows[-1]['unarmed_spread_pct'],
                 rows[-1]['armed_spread_pct']), flush=True)
        m.close()
    out = {'gpu': gpu, 'iters_per_window': args.iters, 'rounds': args.rounds, 'results': rows}
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)
    print(json.dumps({'gpu': gpu}))


if __name__ == '__main__':
    main()
