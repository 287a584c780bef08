"""What a checkpoint (IonicModel.checkpoint / Checkpoint.wait / restore) costs.

    python scripts/checkpoint_overhead.py [--size 32768] [--iters 40] [--rounds 2] [--baseline-rounds 5]
                                          [--dir DIR] [--bench-parent DIR] [--out result.json]

1. 4v at --size^2 (16 GiB of state at 32768^2), one GPU:
   - how long the host is blocked in checkpoint();
   - device time per ODE iteration (CUDA events over --iters iterations) of windows that start right after
     checkpoint() and so overlap the writer's drain, against windows without a checkpoint, alternating, --rounds
     of each: median and spread;
   - wall time from checkpoint() until wait() returns, and bytes per second to disk;
   - restore() plus 10 iterations (host clock, closing sync), pipelined against FIB_PIPELINE_MIN_CELLS past the
     grid size (upload first, then step).
2. BASELINE config 1 (4v 512^2 with a hole, 1000 iterations): a checkpoint every 100 iterations against none, end
   to end on the host clock, alternating, after one untimed round of each.
3. With --bench-parent DIR (a built checkout of the parent commit): `bench.py --gpus 1` with nothing armed, the
   parent and this tree alternating, two runs each.
Checkpoints go to --dir (default: a temporary directory), which is removed afterwards.  Needs a CUDA device."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BASE = {'dt': 0.1, 'dt_per_plot': 10, 'duration': 1, 'timeline': False, 'timeline_name': 'x', 'save_graph': False}


def stats(v):
    v = np.asarray(v, np.float64)
    return {'median': float(np.median(v)), 'min': float(v.min()), 'max': float(v.max()), 'all': [float(x) for x in v]}


def dir_bytes(path):
    return sum(os.path.getsize(os.path.join(d, f)) for d, _, fs in os.walk(path) for f in fs)


def large(args, root):
    from fib_tf_b200 import _capi
    from fib_tf_b200.fenton import Fenton4v
    N = args.size
    cfg = dict(BASE, width=N, height=N, diff=1.5)
    m = Fenton4v(cfg)
    m.define()
    m.add_pace_op('s2', 'luq', 1.0)
    c = m._ctx
    c.step(_capi.OP_ODE, 5)                         # warm-up: graphs, modules
    c.sync()
    path = os.path.join(root, 'large')
    out = {'size': N, 'state_bytes': 4 * N * N * c.nvars, 'iters_per_window': args.iters}
    blocked, overlap, plain, wall, rate = [], [], [], [], []

    def window():
        c.timer_start()
        c.step(_capi.OP_ODE, args.iters)
        c.timer_stop()
        return c.timer_ms() / args.iters

    for _ in range(args.rounds):
        plain.append(window())
        c.sync()
        t0 = time.perf_counter()
        h = m.checkpoint(path)
        blocked.append((time.perf_counter() - t0) * 1e3)
        overlap.append(window())
        h.wait()
        wall.append(time.perf_counter() - t0)
        rate.append(dir_bytes(path) / wall[-1])
    out.update(host_blocked_in_checkpoint_ms=stats(blocked), ms_per_iteration_overlapping_the_drain=stats(overlap),
               ms_per_iteration_without_checkpoint=stats(plain), checkpoint_to_wait_s=stats(wall),
               bytes_per_s_to_disk=stats(rate), checkpoint_bytes=dir_bytes(path))
    m.close()
    restore = {}
    for label, env in (('pipelined', None), ('upload_then_step', str(N * N + 1))):
        if env is None:
            os.environ.pop('FIB_PIPELINE_MIN_CELLS', None)
        else:
            os.environ['FIB_PIPELINE_MIN_CELLS'] = env
        r = Fenton4v(dict(cfg, duration=10 * 10 * 0.1 * (1 + 1e-9)))
        t0 = time.perf_counter()
        r.restore(path)
        t1 = time.perf_counter()
        opened = r._ctx.upload_state()[0]
        for _ in r.run(None, block=False):
            pass
        t2 = time.perf_counter()
        restore[label] = {'restore_call_s': t1 - t0, 'ten_iterations_s': t2 - t1, 'total_s': t2 - t0,
                          'upload_session_open_at_run': bool(opened)}
        r.close()
    os.environ.pop('FIB_PIPELINE_MIN_CELLS', None)
    out['restore_plus_10_iterations'] = restore
    shutil.rmtree(path, ignore_errors=True)
    return out


def baseline1(args, root):
    from fib_tf_b200.fenton import Fenton4v
    path = os.path.join(root, 'baseline1')
    res = {'none': [], 'every_100': []}
    for r in range(args.baseline_rounds + 1):         # round 0 warms up modules, graphs and the writer: not kept
        for label in ('none', 'every_100'):
            m = Fenton4v(dict(BASE, width=512, height=512, diff=1.5, duration=1000))
            m.add_hole_to_phase_field(256, 256, 30)
            m.define()
            m.add_pace_op('s2', 'luq', 1.0)
            m._ctx.sync()
            s2 = m.millisecond_to_step(210)
            t0 = time.perf_counter()
            for i in m.run(None, block=False):
                if i == s2:
                    m.fire_op('s2')
                if label == 'every_100' and (i + 1) % 100 == 0:
                    m.checkpoint(path)
            m.close()                                     # waits for the last checkpoint
            if r:
                res[label].append(time.perf_counter() - t0)
    shutil.rmtree(path, ignore_errors=True)
    return {k: stats(v) for k, v in res.items()}


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
    ap.add_argument('--size', type=int, default=32768)
    ap.add_argument('--iters', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=2)
    ap.add_argument('--baseline-rounds', type=int, default=5)
    ap.add_argument('--dir', default=None)
    ap.add_argument('--bench-parent', default=None)
    ap.add_argument('--bench-steps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit('checkpoint_overhead.py needs a CUDA device')
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                         capture_output=True, text=True).stdout.strip()
    root = tempfile.mkdtemp(prefix='fib_ck_', dir=args.dir)
    out = {'gpu': gpu, 'checkpoint_dir_free_bytes': shutil.disk_usage(root).free}
    print(json.dumps(out), flush=True)
    try:
        out['baseline_config_1'] = baseline1(args, root)
        print(json.dumps(out['baseline_config_1']), flush=True)
        while args.size > 4096 and shutil.disk_usage(root).free < 2.5 * 16 * args.size ** 2:
            args.size //= 2                            # not enough room for two checkpoints: say so in the result
        out['large'] = large(args, root)
        print(json.dumps(out['large']), flush=True)
        if args.bench_parent:
            vals = {'parent': [], 'this': []}
            for _ in range(2):
                vals['parent'].append(bench_value(os.path.abspath(args.bench_parent), args))
                vals['this'].append(bench_value(ROOT, args))
            out['bench_gcell_steps_per_s'] = vals
            print(json.dumps(vals), flush=True)
    finally:
        shutil.rmtree(root, ignore_errors=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
