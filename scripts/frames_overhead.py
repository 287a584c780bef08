"""What the frame recorder (fib_frames_watch, IonicModel.record_frames) costs and saves.

    python scripts/frames_overhead.py [--iters 40] [--rounds 5] [--bench-parent DIR] [--out result.json]

1. The reference's driver loop, BASELINE configs 1 and 2 (512^2 with a hole, 1000 ms, a frame every 10 ms), end
   to end on the host clock with a closing sync: run A is the unchanged `cube[i // ds] = model.image() *
   model.phase` loop, run B the same loop with record_frames(10) and one frames() call.  fib_launch_count of each.
2. Large grids (4096^2): device time per ODE iteration armed (every 10, stride 1 and 8) against unarmed, CUDA
   events over `--iters` iterations, windows alternating on one context (`--rounds` of each), median.
3. With --bench-parent DIR (a built checkout of the parent commit): `bench.py --gpus 1` with nothing armed, the
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

BASE = {'dt': 0.1, 'dt_per_plot': 10, 'duration': 1, 'timeline': False, 'timeline_name': 'x', 'save_graph': False,
        'skip': False, 'cheby': False, 'ultra_slow': False}
N = 4096
LARGE = [
    ('4v, one step per launch', 'fenton', dict(width=N, height=N, diff=1.5, steps_per_launch=1)),
    ('4v, two steps per launch', 'fenton', dict(width=N, height=N, diff=1.5, steps_per_launch=2)),
    ('BR cheby', 'br', dict(width=N, height=N, diff=0.809, cheby=True)),
    ('Courtemanche all-state (court_ultra)', 'court_ultra', dict(width=N, height=N, diff=1.5)),
]


def cls_of(kind):
    from fib_tf_b200.br import BeelerReuter
    from fib_tf_b200.court_ultra import Courtemanche as CourtemancheUltra
    from fib_tf_b200.fenton import Fenton4v
    return {'fenton': Fenton4v, 'br': BeelerReuter, 'court_ultra': CourtemancheUltra}[kind]


def driver_loop(kind, recorder):
    """fenton.py / br.py's __main__ loop; with `recorder` the frames come from the device ring instead."""
    if kind == 'fenton':
        cfg = {'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 1000,
               'timeline': False, 'timeline_name': 'x', 'save_graph': False}
        hole, s2_ms, s2_v = (256, 256, 30), 210, 1.0
    else:
        cfg = {'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809, 'duration': 1000,
               'skip': False, 'cheby': True, 'timeline': False, 'timeline_name': 'x', 'save_graph': False}
        hole, s2_ms, s2_v = (150, 200, 40), 300, 10.0
    model = cls_of(kind)(cfg)
    model.add_hole_to_phase_field(*hole)
    model.define()
    model.add_pace_op('s2', 'luq', s2_v)
    model._ctx.sync()
    s2, ds = model.millisecond_to_step(s2_ms), model.millisecond_to_step(10)
    cube = np.zeros([int(model.duration / 10.0), model.height, model.width], dtype=np.float32)
    n0 = model._ctx.launch_count()
    t0 = time.perf_counter()
    if recorder:
        model.record_frames(ds)
    for i in model.run(None):
        if i == s2:
            model.fire_op('s2')
        if not recorder and i % ds == 0:
            cube[i // ds] = model.image() * model.phase
    model._ctx.sync()
    t_loop = time.perf_counter() - t0
    if recorder:
        iters, frames = model.frames()
        cube[(iters - 1) // ds] = frames * model.phase
    sec = time.perf_counter() - t0
    launches = model._ctx.launch_count() - n0
    model.close()
    return sec, t_loop, launches, cube, s2 // ds if s2 % ds == 0 else None


def window(ctx, iters):
    ctx.timer_start()
    ctx.step(0, iters)
    ctx.timer_stop()
    return ctx.timer_ms() / iters


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
    ap.add_argument('--iters', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--bench-parent', default=None)
    ap.add_argument('--bench-steps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('frames_overhead.py needs a CUDA device')
    from fib_tf_b200 import _capi
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    out = {'gpu': gpu}

    rows = []
    for kind, name in (('fenton', 'BASELINE config 1: 4v 512^2 + hole, 1000 ms, frame every 10 ms'),
                       ('br', 'BASELINE config 2: BR cheby 512^2 + hole, 1000 ms, frame every 10 ms')):
        driver_loop(kind, True)                                              # warm-up: module loads
        a_sec, _, a_launches, a_cube, s2f = driver_loop(kind, False)
        b_sec, b_loop, b_launches, b_cube, _ = driver_loop(kind, True)
        # the loop grabs the S2 frame after firing S2; the recorder takes it before the caller acts
        differ = [j for j in range(a_cube.shape[0]) if not np.array_equal(a_cube[j].view(np.uint32),
                                                                          b_cube[j].view(np.uint32))]
        rows.append({'case': name, 'A_image_loop_s': a_sec, 'B_record_frames_s': b_sec,
                     'B_stepping_s': b_loop, 'B_frames_and_cube_s': b_sec - b_loop, 'speedup': a_sec / b_sec,
                     'A_launches': a_launches, 'B_launches': b_launches, 'frames_differing': differ,
                     's2_frame': s2f})
        print('%-66s A %.3f s (%d launches)  B %.3f s = stepping %.3f + frames() and cube %.3f (%d launches)  '
              'differing frames %s (S2 frame %s)' % (name, a_sec, a_launches, b_sec, b_loop, b_sec - b_loop,
                                                     b_launches, differ, s2f), flush=True)
    out['driver_loop'] = rows

    rows = []
    for name, kind, cfg in LARGE:
        m = cls_of(kind)(dict(BASE, **cfg))
        m.define()
        ctx = m._ctx
        ctx.step(0, 3)
        res = {'case': name, 'cells': m.height * m.width}
        times = {'unarmed': [], 'stride1': [], 'stride8': []}
        for _ in range(args.rounds):
            for key in times:
                if key != 'unarmed':
                    ctx.frames_watch(m._pot_name, 1, 10, int(key[6:]), 8)
                ctx.step(0, 1)
                times[key].append(window(ctx, args.iters))
                if key != 'unarmed':
                    ctx.frames_stop()
        t0 = float(np.median(times['unarmed']))
        res['unarmed_ms_per_iter'] = t0
        res['unarmed_spread_pct'] = 100.0 * (max(times['unarmed']) - min(times['unarmed'])) / t0
        for key in ('stride1', 'stride8'):
            t = float(np.median(times[key]))
            res[key + '_ms_per_iter'] = t
            res[key + '_overhead_pct'] = 100.0 * (t - t0) / t0
        res['kernel'] = _capi.last_kernel()
        rows.append(res)
        print('%-40s unarmed %.4f ms  stride 1 %+.2f %%  stride 8 %+.2f %%  (unarmed spread %.2f %%)' % (
            name, t0, res['stride1_overhead_pct'], res['stride8_overhead_pct'], res['unarmed_spread_pct']), flush=True)
        m.close()
    out['large_grids'] = {'iters_per_window': args.iters, 'rounds': args.rounds, 'every': 10, 'results': rows}

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
