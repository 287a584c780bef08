"""Cost of the per-replica observers (include/fib_b200.h, fib_replica_probe_watch, fib_replica_sums).

    python scripts/replica_observers_overhead.py [--rounds 5] [--window 0.3] [--bench-parent DIR] [--out result.json]

Per ensemble, two batched models of the same config are built: one with the replica probe armed at (20, W//2), as
run() arms it for a replica_cl_observer, and one without.  They are warmed up and timed in alternating windows on the
same card: CUDA events around `fib_step(ctx, ODE, n)`, n chosen so that a window lasts about --window seconds; the
armed model's ring is drained between its windows, outside the timing.  Reported: medians of --rounds windows in
Gcell-steps/s and the cost per iteration of the armed probe.  Then, at B = 1024, one masked_image_means() call
against np.mean(image() * mask) per replica (host wall clock, each call ends in a device synchronise; medians of
--calls calls).  With --bench-parent DIR (a built checkout of the parent commit): `bench.py --gpus 1` on the parent and
on this tree, alternating, two runs each.  Needs a CUDA device; no fall-back."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

from replicas_throughput import bench_value, iters_for, make, rate, timed  # noqa: E402

# name, model, height, width, config extras, diff of replica 0, hole (x, y, r) or None, replicas
CASES = [
    ('4v 128^2', 'fenton4v', 128, 128, {}, 1.5, None, 1024),
    ('4v 512^2 + hole', 'fenton4v', 512, 512, {}, 1.5, (256, 256, 30), 64),
    ('Courtemanche ultra 512^2', 'court_ultra', 512, 512, {}, 1.5, None, 16),
]


def median_call(fn, calls):
    ts = []
    for _ in range(calls):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--window', type=float, default=0.3, help='seconds per timed window')
    ap.add_argument('--calls', type=int, default=10)
    ap.add_argument('--bench-parent', default=None)
    ap.add_argument('--bench-steps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('replica_observers_overhead.py needs a CUDA device')
    from fib_tf_b200 import _capi
    from fib_tf_b200.egm import create_mask
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    out = {'gpu': gpu, 'metric': 'Gcell-steps/s (device time, CUDA events)', 'rounds': args.rounds, 'cases': []}
    for name, kind, H, W, extra, diff, hole, B in CASES:
        armed, bare = make(kind, H, W, extra, diff, hole, B), make(kind, H, W, extra, diff, hole, B)
        cap = armed._ctx.replica_probe_watch(armed._pot_name, 20, W // 2)
        timed(armed, 20)
        timed(bare, 20)
        n = iters_for(bare, args.window)
        ra, rb = [], []
        for _ in range(args.rounds):
            ra.append(rate(armed, n, timed(armed, n), B))
            armed._ctx.replica_probe_fetch(cap)                              # drain, outside the window
            rb.append(rate(bare, n, timed(bare, n), B))
        ma, mb = float(np.median(ra)), float(np.median(rb))
        cells = B * H * W * armed.dt_per_step
        cost_us = (cells / ma - cells / mb) / 1e3                           # per iteration, from the medians
        row = {'case': name, 'replicas': B, 'capacity': cap, 'iters_per_window': n, 'kernel': _capi.last_kernel(),
               'armed': {'gcell_steps_s': ra, 'median': ma}, 'unarmed': {'gcell_steps_s': rb, 'median': mb},
               'armed_over_unarmed': ma / mb, 'cost_us_per_iteration': cost_us}
        out['cases'].append(row)
        print('%-26s B=%5d  armed %8.2f  unarmed %8.2f Gcell-steps/s  ratio %.4f  %+.2f us/iteration'
              % (name, B, ma, mb, ma / mb, cost_us), flush=True)
        armed.close()
        bare.close()
    # one masked_image_means() against the image()-based per-replica means, 4v 128^2 x 1024
    m = make('fenton4v', 128, 128, {}, 1.5, None, 1024)
    m._ctx.step(_capi.OP_ODE, 50)
    mask = create_mask(m, 64, 64, 10)
    slot = m.add_probe_mask(mask)
    dev = m.masked_image_means(slot)
    host = np.mean(m.image().astype(np.float64) * mask, axis=(1, 2))
    t_dev, ts_dev = median_call(lambda: m.masked_image_means(slot), args.calls)
    t_host, ts_host = median_call(lambda: np.mean(m.image() * mask, axis=(1, 2)), args.calls)
    out['masked_means_1024'] = {'device_s': t_dev, 'image_based_s': t_host, 'speedup': t_host / t_dev,
                                'device_calls_s': ts_dev, 'image_calls_s': ts_host,
                                'max_rel_diff': float(np.max(np.abs(dev - host) / np.maximum(np.abs(host), 1e-30)))}
    print('masked_image_means B=1024: %.3f ms, image()-based %.3f ms (x%.1f)' % (t_dev * 1e3, t_host * 1e3,
                                                                                  t_host / t_dev), flush=True)
    m.close()
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
