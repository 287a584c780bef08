#!/usr/bin/env python
"""
bench.py -- BASELINE.json's headline measurement: Gcell-steps/s (and % of the HBM roofline) of the
Fenton 4v spiral-wave fibrillation run on a 32768x32768 grid, row-sharded over N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--size S] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one run() iteration of the reference driver loop = dt_per_step = 10 explicit time
steps of the whole grid (fenton.py:133-138).  STRONG scaling: the 32768^2 grid is fixed, each rank
owns 32768/N rows.  Rank 0 prints exactly ONE JSON line on stdout.

  value     device-timed (CUDA events on the library's stream, max over ranks), state resident in
            HBM; the state (16 GiB) is >> the 126 MB L2, so no flush is needed between steps.
  e2e       the same K iterations through the public drop-in API (Fenton4v.run() generator) with
            HOST buffers inside the timed region: strip-wise upload of the full initial state
            (16 GiB at 32768^2) from pinned memory (H2D), the headless cycle-length probe every iteration (D2H) and a
            full-frame grab into pinned memory every 10th iteration (the cadence of fenton.py:184).
  roofline  HBM-bound: 32 B per cell-step (4 fp32 planes read + written once) x cells per launch
            / average launch duration, against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline / --impl reference
            the oracle's plain-C + OpenMP port of the same step (oracle/csrc/monodomain_cpu.c) on
            all host cores, on a bounded 2048^2 mirror-tiled sample of the same workload.
            (TensorFlow, the reference's real CPU path, is not installable in this image.)
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TILE = 512
B_ALG = 32.0        # bytes per cell-step: 4 state planes x (read + write) x 4 B  (SURVEY.md 8d)
METRIC = 'Gcell-steps/s'
FALLBACK_HBM = 6650.0


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def fenton_config(size, duration, distributed=False, **kw):
    cfg = {'width': size, 'height': size, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5,
           'duration': duration, 'timeline': False, 'timeline_name': 'unused.json',
           'save_graph': False, 'distributed': distributed}
    cfg.update(kw)
    return cfg


# ---------------------------------------------------------------------------------------------
# synthetic input: a developed 512^2 spiral, mirror-tiled (SURVEY.md 8d item 5)
# ---------------------------------------------------------------------------------------------
def strips_of(tile_plane, width):
    """[512, width] strips for even / odd tile rows: alternate tiles are mirrored so that every
    tile seam is a mirror plane, i.e. a no-flux boundary of the small problem."""
    pair = np.hstack([tile_plane, tile_plane[:, ::-1]])
    reps = -(-width // pair.shape[1])
    even = np.tile(pair, reps)[:, :width]
    return even, even[::-1]


def pinned_strips(tile, width):
    """The synthetic input as it sits in page-locked host memory: per state variable the two
    [512, width] strips (even / odd tile rows) of the mirror-tiled field."""
    from fib_tf_b200 import _capi
    out = {}
    for name, plane in tile.items():
        even, odd = strips_of(plane, width)
        bufs = [_capi.pinned_empty((TILE, width)), _capi.pinned_empty((TILE, width))]
        bufs[0][:] = even
        bufs[1][:] = odd
        out[name] = bufs
    return out


def upload_tiled(ctx, strips, row0, rows, width, descending=False):
    """Strip-wise H2D upload (from pinned memory) of the mirror-tiled state for global rows
    [row0, row0+rows): every 512-row strip of every plane is one ENQUEUE-ONLY fib_set_rect_async, issued
    block by block with all planes of a strip together, so that the library can step behind the copies
    (csrc/fib_capi.cu finish_upload_session).  Top to bottom, or -- odd ranks of a sharded run -- bottom to
    top, so that both shards of a seam begin or end their uploads there (fib_step_behind_upload)."""
    pieces = []
    g = row0
    while g < row0 + rows:
        t, r = divmod(g, TILE)
        n = min(TILE - r, row0 + rows - g)
        pieces.append((g, t, r, n))
        g += n
    nbytes = 0
    for g, t, r, n in (reversed(pieces) if descending else pieces):
        for name, pinned in strips.items():
            ctx.set_rect_async(name, g, 0, pinned[t & 1][r:r + n])
            nbytes += n * width * 4
    return nbytes


def tiled_host(tile, size):
    out = {}
    for name, plane in tile.items():
        even, odd = strips_of(plane, size)
        blocks = [(even if (t & 1) == 0 else odd) for t in range(-(-size // TILE))]
        out[name] = np.ascontiguousarray(np.vstack(blocks)[:size])
    return out


# ---------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, device):
        self.device, self.rows, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '--query-gpu=' + self.Q, '--format=csv,noheader,nounits', '-lms', '100'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(',')]
            if len(f) >= 8 and f[0] == str(self.device):
                self.rows.append(f)

    def stop(self):
        if self.proc:
            # a run shorter than nvidia-smi's start-up (reduced --size) would end without any
            # sample: wait for the first one rather than report nothing
            t0 = time.time()
            while not self.rows and time.time() - t0 < 2.0 and self.proc.poll() is None:
                time.sleep(0.05)
            self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown',
                                'sw_power_cap'), r[4:8]):
                if v.lower() == 'active':
                    reasons.add(name)
        smax = [float(r[2]) for r in self.rows if r[2].replace('.', '').isdigit()]
        pw = [float(r[3]) for r in self.rows if r[3].replace('.', '').isdigit()]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(smax) if smax else None,
                'power_w_max': max(pw) if pw else None, 'samples': len(self.rows),
                'reasons': sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# CPU baseline: the oracle's C/OpenMP port on a bounded sample
# ---------------------------------------------------------------------------------------------
def cpu_sample_run(tile, iterations, budget_s, sample=2048, warmup=1):
    """Times `iterations` run() iterations (10 steps each) of the C port on a sample^2
    mirror-tiled grid after `warmup` untimed ones; stops early when the time budget is spent.
    -> (gcell_steps_per_s, seconds per iteration, iterations timed, info)"""
    from oracle import cpu_port
    L = cpu_port.port()
    st = tiled_host(tile, sample)
    tmp = np.empty_like(st['U'])

    u, t = st['U'], tmp
    per_iter = []
    t_all = time.perf_counter()
    done = 0
    for it in range(iterations + warmup):
        t0 = time.perf_counter()
        for _ in range(10):
            L.fib_cpu_fenton_step(sample, sample, u, t, st['V'], st['W'], st['S'], None, 0.1, 1.5)
            u, t = t, u
        dt = time.perf_counter() - t0
        if it >= warmup:
            per_iter.append(dt)
            done += 1
        if time.perf_counter() - t_all > budget_s and done >= 1:
            break
    sec = float(np.mean(per_iter))
    val = sample * sample * 10 / sec / 1e9
    info = {'value': val, 'unit': METRIC, 'cores': int(L.fib_cpu_threads()), 'kind': 'port',
            'sample': 'oracle C/OpenMP port, Fenton 4v %dx%d mirror-tiled spiral, %d iterations x 10 '
                      'steps after %d warm-up (%.2f s/iteration); reference publishes 0.052 Gcell-steps/s for '
                      'its TF CPU path on a 1.7 GHz quad-core (details.md:264)' % (sample, sample, done, warmup, sec),
            'host_cpus': os.cpu_count()}
    return val, sec, done, info


def numpy_restatement_baseline(iterations=20):
    """BASELINE.md 3.2: the reference's CPU path is TensorFlow executing fenton.py's graph on tf.device
    CPU.  TensorFlow cannot be installed here and /root/reference does not exist on the GPU box, so the
    closest thing that runs is the oracle's NumPy restatement (oracle/monodomain_np.py: bit-identical to
    the unmodified reference executed through the NumPy TF facade, tests/test_oracle_golden.py), one
    core, BASELINE config 1 (4v 512^2 with the hole of fenton.py:169): `iterations` x 10 time steps."""
    from oracle import monodomain_np as onp
    cfg = fenton_config(TILE, 1)
    m = onp.OracleModel('fenton4v', cfg)
    m.add_hole(256, 256, 30)
    m.define()
    m.iterate()                                   # warm-up
    t0 = time.perf_counter()
    for _ in range(iterations):
        m.iterate()
    sec = time.perf_counter() - t0
    out = {'value': TILE * TILE * 10 * iterations / sec / 1e9, 'unit': METRIC, 'cores': 1,
           'kind': 'port (NumPy restatement, bit-identical to the reference under the NumPy TF facade)',
           'sample': 'BASELINE config 1: Fenton 4v 512x512 + hole, %d time steps in %.1f s' % (10 * iterations, sec)}
    rec = os.path.join(ROOT, 'profiles', 'r2_facade_baseline.json')
    if os.path.exists(rec):                       # the reference's own solve() under tfshim, timed in the build container
        out['facade_recorded'] = json.load(open(rec))
    return out


def spiral_tile_cpu():
    """The developed 512^2 spiral WITHOUT a GPU: the S1-S2 protocol of fenton.py:155-185 (no hole) run
    to 400 ms with the oracle's C/OpenMP port, about 3 s on 16 cores.  Both arms start from it: the
    reference arm must not map the product's .so, and our arm's input must not depend on the build
    being measured, so that --dump-outputs of two builds can be compared cell by cell.  Every cell is
    updated independently, so the result does not depend on the number of threads."""
    from oracle import cpu_port
    m = cpu_port.CPortModel('fenton4v', fenton_config(TILE, 400))
    m.define()
    m.add_pace('s2', 'luq', 1.0)
    for i in range(400):
        m.iterate()
        if i == 210:
            m.fire('s2')
    return {n: np.ascontiguousarray(m.state[n]) for n in ('U', 'V', 'W', 'S')}


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the reference arm is the CPU path "with all
    # the host threads it can use", so undo that before libgomp is loaded
    if int(os.environ.get('WORLD_SIZE', 1)) > 1 or 'TORCHELASTIC_RUN_ID' in os.environ:
        os.environ['OMP_NUM_THREADS'] = str(os.cpu_count() or 1)
    tile = spiral_tile_cpu()
    W = max(args.warmup, 3)
    val, sec, done, info = cpu_sample_run(tile, args.steps, budget_s=150.0, warmup=W)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': METRIC, 'n_gpus': args.gpus,
        'steps': done, 'warmup': W, 'ms_per_step': sec * 1e3, 'higher_is_better': True,
        'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.size, args.gpus),
        'cpu_baseline': info,
        'e2e': {'value': val, 'unit': METRIC, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
        'note': 'reference arm = the reference algorithm on host cores (oracle C/OpenMP port; '
                'TensorFlow is not installable offline); each step is one run() iteration of a '
                'bounded 2048^2 sample of the workload; no GPU and no product code is touched',
    }
    emit(line)


def workload_config(size, n):
    # same rule as fib_tf_b200.fenton.Fenton4v._steps_per_launch (kept torch/CUDA-free for the reference arm)
    env = os.environ.get('FIB_STEPS_PER_LAUNCH')
    spl = int(env) if env else (2 if size * size >= 3072 * 3072 else 1)
    spl = 2 if (spl == 2 and size % 4 == 0 and size // n >= 2) else 1
    halo = ('2 rows of U, V, W, S per neighbour per launch (= two time steps) over NCCL send/recv' if spl == 2
            else '1 row of U per neighbour per time step over NCCL send/recv')
    return {'workload': 'Fenton 4v spiral-wave fibrillation %dx%d (BASELINE.json configs[4]), dt=0.1 ms, '
                        'diff=1.5, no phase field, mirror-tiled developed 512^2 spiral' % (size, size),
            'grid': [size, size], 'time_steps_per_step': 10, 'time_steps_per_launch': spl,
            'parallelism': 'row-shard x%d' % n, 'halo': halo if n > 1 else 'none',
            'l2': 'state %.1f GiB >> 126 MB L2: no flush needed' % (size * size * 16 / 2 ** 30),
            'seed': 0}


# ---------------------------------------------------------------------------------------------
# --dump-outputs: what the timed steps computed, for comparing two builds output for output
# ---------------------------------------------------------------------------------------------
DUMP_ROWS = 64      # full rows of every plane: 64 x 32768 x 4 planes x 4 B = 32 MiB at the default size


def dump_rows(size):
    """The fixed, seeded sample of global rows that --dump-outputs writes (every row of a smaller grid)."""
    return np.sort(np.random.default_rng(0).choice(size, min(DUMP_ROWS, size), replace=False))


def read_dump_rows(ctx, size):
    """(global rows, {plane: [len(rows), size] float32}) for the dump rows inside this rank's shard."""
    rows = [int(r) for r in dump_rows(size) if ctx.row0 <= r < ctx.row0 + ctx.rows]
    return rows, {n: np.array([ctx.get_rect(n, r, r + 1, 0, size)[0] for r in rows],
                              np.float32).reshape(len(rows), size) for n in ctx.var_names}


def write_dump(out_dir, parts):
    """parts: read_dump_rows of every rank -> out_dir/<plane>.npy, rows in ascending order, and
    out_dir/rows.npy with their global indices."""
    rows = np.concatenate([np.asarray(r, np.float64) for r, _ in parts])
    order = np.argsort(rows)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'rows.npy'), rows[order])
    for name in parts[0][1]:
        np.save(os.path.join(out_dir, name + '.npy'), np.concatenate([p[name] for _, p in parts])[order])


# ---------------------------------------------------------------------------------------------
# the other kernels / BASELINE configurations, device-timed (N = 1 only): `suite` in the JSON line
# ---------------------------------------------------------------------------------------------
def run_suite(device, peak, budget_s=45.0):
    """Device-timed throughput (CUDA events on the library stream, 3 warm-up iterations) of the 4096^2
    roofline points of every kernel family and of BASELINE configs 1-4 at their own sizes, through the
    drop-in model classes.  frac = B_alg x Gcell-steps/s / measured HBM peak, B_alg = 8 bytes x state
    planes (+4 with a phase field) per cell-step (SURVEY.md 8d)."""
    from fib_tf_b200 import _capi
    from fib_tf_b200.br import BeelerReuter
    from fib_tf_b200.court import Courtemanche
    from fib_tf_b200.court_ultra import Courtemanche as CourtUltra
    from fib_tf_b200.fenton import Fenton4v
    cases = [
        # name, class, N, extra config, hole, B_alg, iterations, slow_every
        ('config1: 4v 512^2 + hole(256,256,30), one fib_step per iteration (driver loop)', Fenton4v, 512, {'diff': 1.5}, (256, 256, 30), 36, 300, 0),
        ('config1: 4v 512^2 + hole(256,256,30), one fib_step for 300 iterations', Fenton4v, 512, {'diff': 1.5}, (256, 256, 30), 36, 300, -1),
        ('config1 without the persistent kernel (one launch per step, CUDA graph)', Fenton4v, 512, {'diff': 1.5, 'persist': False}, (256, 256, 30), 36, 300, 0),
        ('config2: BR 512^2 cheby + hole(150,200,40), one fib_step per iteration (driver loop)', BeelerReuter, 512, {'diff': 0.809, 'cheby': True}, (150, 200, 40), 68, 300, 0),
        ('config2: BR 512^2 cheby + hole(150,200,40), one fib_step for 300 iterations', BeelerReuter, 512, {'diff': 0.809, 'cheby': True}, (150, 200, 40), 68, 300, -1),
        ('config2 without the persistent kernel (one launch per step, CUDA graph)', BeelerReuter, 512, {'diff': 0.809, 'cheby': True, 'persist': False}, (150, 200, 40), 68, 300, 0),
        ('config3: BR 2048^2 cheby+skip', BeelerReuter, 2048, {'diff': 0.809, 'cheby': True, 'skip': True}, None, 64, 30, 0),
        ('config4: Courtemanche 2048^2 multi-rate loop (slow every 10)', Courtemanche, 2048, {'diff': 0.809}, None, 168, 60, 10),
        ('config4: Courtemanche 2048^2 ultra + LUT', CourtUltra, 2048, {'diff': 1.5, 'lut': True}, None, 168, 30, 0),
        ('4096^2: 4v, one step per launch', Fenton4v, 4096, {'diff': 1.5, 'steps_per_launch': 1}, None, 32, 8, 0),
        ('4096^2: 4v, two steps per launch', Fenton4v, 4096, {'diff': 1.5, 'steps_per_launch': 2}, None, 32, 8, 0),
        ('4096^2: BR cheby', BeelerReuter, 4096, {'diff': 0.809, 'cheby': True}, None, 64, 8, 0),
        ('4096^2: BR exact gates', BeelerReuter, 4096, {'diff': 0.809}, None, 64, 8, 0),
        ('4096^2: BR cheby+skip', BeelerReuter, 4096, {'diff': 0.809, 'cheby': True, 'skip': True}, None, 64, 8, 0),
        ('4096^2: Courtemanche ultra', CourtUltra, 4096, {'diff': 1.5}, None, 168, 8, 0),
        ('4096^2: Courtemanche ultra + LUT', CourtUltra, 4096, {'diff': 1.5, 'lut': True}, None, 168, 8, 0),
    ]
    out, t_start = [], time.perf_counter()
    for name, cls, N, extra, hole, balg, iters, slow_every in cases:
        if time.perf_counter() - t_start > budget_s:
            out.append({'case': name, 'skipped': 'suite time budget'})
            continue
        cfg = {'width': N, 'height': N, 'dt': 0.1, 'dt_per_plot': 10, 'duration': 1, 'timeline': False,
               'timeline_name': 'x', 'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False,
               'device': device}
        cfg.update(extra)
        m = cls(cfg)
        if hole:
            m.add_hole_to_phase_field(*hole)
        m.define()
        c = m._ctx

        def go(n):
            if slow_every < 0:                  # one C-ABI call for all iterations
                c.step(0, n)
                return
            for i in range(n):
                c.step(0, 1)
                if slow_every > 0 and i % slow_every == 0:
                    c.step(1, 1)
        go(3)
        c.sync()
        c.timer_start()
        go(iters)
        c.timer_stop()
        ms = c.timer_ms()
        steps = iters * m.dt_per_step
        g = N * N * steps / (ms * 1e-3) / 1e9
        out.append({'case': name, 'grid': [N, N], 'time_steps': steps, 'us_per_time_step': ms * 1e3 / steps,
                    'value': g, 'unit': METRIC, 'bytes_per_cell_step': balg, 'frac': g * balg / peak,
                    'kernel': _capi.last_kernel(), 'l2_resident': N * N * 4 * c.nvars < 100e6})
        m.close()
    return out


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly ONE line, the JSON: everything else any library prints there (NCCL's version
    banner, for one) is sent to stderr by pointing fd 1 at fd 2 for the life of the run."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours')
    ap.add_argument('--size', type=int, default=32768)
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-suite', action='store_true', help='skip the per-kernel suite (N = 1)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the state after the timed steps to DIR/<plane>.npy (a fixed sample of %d '
                         'full rows, float32; their indices in DIR/rows.npy)' % DUMP_ROWS)
    args = ap.parse_args()
    if args.impl == 'reference':
        return run_reference_arm(args)
    if 'TORCHELASTIC_RUN_ID' in os.environ:
        # torchrun exports OMP_NUM_THREADS=1: share the host cores among the ranks of this node for the
        # CPU-built input instead.  Before torch is imported: it loads the libgomp the oracle port uses.
        local_world = int(os.environ.get('LOCAL_WORLD_SIZE', 1))
        os.environ['OMP_NUM_THREADS'] = str(max(1, (os.cpu_count() or 1) // local_world))

    import torch
    import torch.distributed as dist
    from fib_tf_b200 import _capi
    from fib_tf_b200.fenton import Fenton4v

    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: fib_tf_b200 has no CPU fallback')
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # rank 0 prints exactly ONE line on stdout: keep NCCL's version banner off it
        os.environ['NCCL_DEBUG'] = os.environ.get('FIB_NCCL_DEBUG', 'WARN')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    K, Wm, size = args.steps, max(args.warmup, 3), args.size

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device='cuda', dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return float(x)
        t = torch.tensor([float(x)], device='cuda', dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    tile = spiral_tile_cpu()
    model = Fenton4v(fenton_config(size, K * 10 * 0.1, distributed=world > 1, device=local))
    model.define(s1=False)
    ctx = model._ctx
    row0, rows = model._row0, model._rows
    strips = pinned_strips(tile, size)
    upload_tiled(ctx, strips, row0, rows, size)

    sampler = ClockSampler(local)
    sampler.start()
    ctx.step(0, Wm)                                     # warm-up (also instantiates the graph)
    barrier()
    # EXACTLY K steps in the timed region, bracketed by barrier + synchronize
    n0 = ctx.launch_count()
    ctx.timer_start()
    ctx.step(0, K)
    ctx.timer_stop()
    ms_dev = ctx.timer_ms()
    barrier()
    launches_rank = ctx.launch_count() - n0
    ms = max_over_ranks(ms_dev)
    launches = int(sum_over_ranks(launches_rank))
    dump = read_dump_rows(ctx, size) if args.dump_outputs else None
    cells = float(size) * size
    value = cells * K * 10 / (ms * 1e-3) / 1e9

    # ---- e2e through the public API, host buffers inside the timed region ----
    frame = _capi.pinned_empty((rows, size))
    probes = []
    model.cl_observer = lambda i, cl: probes.append((i, cl))
    d2h = 0
    barrier()
    t0 = time.perf_counter()
    h2d = upload_tiled(ctx, strips, row0, rows, size, descending=(world > 1 and rank % 2 == 1))
    with contextlib.redirect_stdout(sys.stderr):
        for i in model.run(None):
            if i % 10 == 9 or i == K - 1:                 # a frame every 10 iterations (fenton.py:184) + the last
                if d2h:
                    model.image_wait()
                model.image_async(frame)                  # pinned target, overlaps the next steps
                d2h += frame.nbytes
        model.image_wait()
    d2h += 4 * K                                          # the per-iteration probe read
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = cells * K * 10 / e2e_s / 1e9
    clocks = sampler.stop()

    peaks_path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))['hbm_gbs']), 'of measured (MEASURED_PEAKS.json hbm_gbs)'
    else:
        peak, peak_src = FALLBACK_HBM, 'of fallback (B200_PROFILING.md)'
    # one time step of this rank's shard = one step kernel (three launches when sharded: the two
    # boundary rows first, then the interior, so that the halo exchange overlaps the interior)
    # With two time steps per launch (csrc/fib_fused.cuh, the default at this size) every plane is
    # read and written once per TWO steps, so the algorithmic 32 B per cell-step (SURVEY.md 8d, which
    # temporal blocking does not change) can exceed the HBM peak: frac > 1 is expected then, and
    # `traffic` (ncu DRAM bytes per time step) is what shows the saving.
    spl = int(getattr(model, 'steps_per_launch_used', 1))
    launch_ms = ms_dev / (K * 10)
    achieved = B_ALG * rows * size / (launch_ms * 1e-3) / 1e9
    # `traffic`: DRAM bytes PER LAUNCH of the dominant kernel = ncu dram__bytes_read.sum + write.sum per
    # cell and time step (profiles/traffic.json, one `ncu --set full` capture of this kernel at 4096^2)
    # x the cells and the time steps one launch of this rank covers.  dram_frac = that traffic / the
    # launch duration measured here / the HBM peak: how busy HBM really is (frac, on the ALGORITHMIC
    # 32 B per cell-step, exceeds 1 with two steps per launch because the planes move once per two steps).
    traffic, dram_frac, traffic_src = None, None, None
    tpath = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tpath):
        tj = json.load(open(tpath)).get('fenton4v_fused2_step' if spl == 2 else 'fenton4v_step')
        if tj:
            traffic = tj['dram_bytes_per_cell'] * rows * size * spl
            dram_frac = traffic / (launch_ms * spl * 1e-3) / 1e9 / peak
            traffic_src = 'profiles/traffic.json: %s B per cell and time step (ncu --set full)' % tj['dram_bytes_per_cell']
    roofline = {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s',
                'frac': achieved / peak, 'traffic': traffic, 'dram_frac': dram_frac,
                'traffic_source': traffic_src, 'peak_source': peak_src,
                'kernel': 'fib::fenton_fused2_kernel (2 time steps per launch)' if spl == 2
                          else 'fib::step_kernel<Fenton4v,...>',
                'bytes_per_cell_step': B_ALG, 'time_steps_per_launch': spl,
                'avg_launch_ms': launch_ms * spl, 'ms_per_time_step': launch_ms,
                'cells_per_launch': rows * size,
                'launches_per_time_step': launches_rank / (K * 10.0)}

    line = {
        'metric': METRIC, 'value': value, 'unit': METRIC, 'n_gpus': world, 'steps': K, 'warmup': Wm,
        'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(size, world),
        'e2e': {'value': e2e_value, 'unit': METRIC, 'h2d_bytes_per_step': sum_over_ranks(h2d) / K,
                'd2h_bytes_per_step': sum_over_ranks(d2h) / K, 'seconds': e2e_s},
        'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline,
    }
    if rank == 0 and world == 1 and not args.no_suite:
        line['suite'] = run_suite(local, peak)
    if rank == 0 and world == 1 and not args.no_cpu:
        _v, _s, _d, info = cpu_sample_run(tile, 8, budget_s=20.0, warmup=3)
        info['numpy_restatement'] = numpy_restatement_baseline()
        line['cpu_baseline'] = info
    if rank == 0:
        emit(line)
    if dump is not None:
        parts = [dump]
        if world > 1:
            parts = [None] * world
            dist.all_gather_object(parts, dump)
        if rank == 0:
            write_dump(args.dump_outputs, parts)
    for p in [b for bufs in strips.values() for b in bufs] + [frame]:
        _capi.pinned_free(p)
    model.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
