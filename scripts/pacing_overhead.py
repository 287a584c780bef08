"""What pacing on the device (fib_pace_add, IonicModel.pace) costs and saves against firing from the host.

    python scripts/pacing_overhead.py [--rounds 3] [--bench-parent DIR] [--out result.json]

1. BASELINE configs 1 and 2 (512^2 with a hole, 1000 ms) with a burst train from the left edge: a beat every
   20 ms from 50 ms on, 40 beats.  Run A is the driver loop `for i in run(): if i in beats: fire_op('s1')`, run B
   the same loop with one pace('s1', ...) before it.  Per run: fib_launch_count, device time (CUDA events around
   the loop) and host time; A and B alternate `--rounds` times, medians reported; the final planes of A and B are
   compared bit for bit.
2. With --bench-parent DIR (a built checkout of the parent commit): `bench.py --gpus 1` with nothing armed, the
   parent and this tree alternating, two runs each.
Needs a CUDA device; no fall-back."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def config(kind):
    from fib_tf_b200.br import BeelerReuter
    from fib_tf_b200.fenton import Fenton4v
    if kind == 'fenton':
        cfg = {'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 1000,
               'timeline': False, 'timeline_name': 'x', 'save_graph': False}
        return Fenton4v, cfg, (256, 256, 30), 1.0
    cfg = {'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809, 'duration': 1000,
           'skip': False, 'cheby': True, 'timeline': False, 'timeline_name': 'x', 'save_graph': False}
    return BeelerReuter, cfg, (150, 200, 40), 10.0


def driver_loop(kind, paced, start_ms=50, cl_ms=20, beats=40):
    cls, cfg, hole, v = config(kind)
    model = cls(cfg)
    model.add_hole_to_phase_field(*hole)
    model.define()
    model.add_pace_op('s1', 'left', v)
    model._ctx.sync()
    at, every = model.millisecond_to_step(start_ms), model.millisecond_to_step(cl_ms)
    fire = {at + j * every for j in range(beats)}
    n0 = model._ctx.launch_count()
    t0 = time.perf_counter()
    model._ctx.timer_start()
    if paced:
        model.pace('s1', at, every, beats)
    for i in model.run(None):
        if not paced and i in fire:
            model.fire_op('s1')
    model._ctx.timer_stop()
    device_s = model._ctx.timer_ms() / 1000.0
    host_s = time.perf_counter() - t0
    launches = model._ctx.launch_count() - n0
    state = {name: model._ctx.get_state(name) for name in model._ctx.var_names}
    model.close()
    return device_s, host_s, launches, state


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
    ap.add_argument('--bench-parent', default=None)
    ap.add_argument('--bench-steps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('pacing_overhead.py needs a CUDA device')
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    out = {'gpu': gpu}

    rows = []
    for kind, name in (('fenton', 'BASELINE config 1: 4v 512^2 + hole, 1000 ms, 40 beats every 20 ms from 50 ms'),
                       ('br', 'BASELINE config 2: BR cheby 512^2 + hole, 1000 ms, 40 beats every 20 ms from 50 ms')):
        driver_loop(kind, True)                                              # warm-up: module loads
        res = {'A_fire_op': {'device_s': [], 'host_s': []}, 'B_pace': {'device_s': [], 'host_s': []}}
        for _ in range(args.rounds):
            for key, paced in (('A_fire_op', False), ('B_pace', True)):
                dev, host, launches, state = driver_loop(kind, paced)
                res[key]['device_s'].append(dev)
                res[key]['host_s'].append(host)
                res[key]['launches'] = launches
                res[key]['state'] = state
        same = all(np.array_equal(res['A_fire_op']['state'][v].view(np.uint32), res['B_pace']['state'][v].view(np.uint32))
                   for v in res['A_fire_op']['state'])
        row = {'case': name, 'bit_identical': same}
        for key in ('A_fire_op', 'B_pace'):
            del res[key]['state']
            res[key]['device_s_median'] = float(np.median(res[key]['device_s']))
            res[key]['host_s_median'] = float(np.median(res[key]['host_s']))
            row[key] = res[key]
        rows.append(row)
        print('%-80s A fire_op: %d launches, device %.4f s, host %.4f s | B pace: %d launches, device %.4f s, '
              'host %.4f s | identical %s' % (name, row['A_fire_op']['launches'], row['A_fire_op']['device_s_median'],
                                              row['A_fire_op']['host_s_median'], row['B_pace']['launches'],
                                              row['B_pace']['device_s_median'], row['B_pace']['host_s_median'], same),
              flush=True)
    out['burst_train'] = {'rounds': args.rounds, 'results': rows}

    if args.bench_parent:
        vals = {'parent': [], 'this': []}
        for _ in range(2):
            vals['parent'].append(bench_value(os.path.abspath(args.bench_parent), args))
            vals['this'].append(bench_value(ROOT, args))
            print('bench.py value: parent %s  this %s' % (vals['parent'], vals['this']), flush=True)
        out['bench_nothing_armed'] = {'metric': 'Gcell-steps/s', 'steps': args.bench_steps, 'alternating': vals}
    else:
        out['bench_nothing_armed'] = 'not measured'
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)
    print(json.dumps({'gpu': gpu}))


if __name__ == '__main__':
    main()
