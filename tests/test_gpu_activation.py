"""GPU: device-side activation maps (include/fib_b200.h fib_activation_watch, csrc/fib_activation.cuh).

  * bit for bit equal to the NumPy restatement (oracle/activation_np.py) fed with the device's own samples,
    on every kernel family, asserting which instantiation ran;
  * invariant, bit for bit, under every stepping path: graph or direct launches, the persistent kernel,
    two time steps per launch, in-process shard groups, deferred batches cut by a read, an upload that
    would otherwise be pipelined; re-arming resets;
  * the published conduction-velocity table from the LAST map, in the same run as measure_cv;
  * the reference's spiral runs: the maps equal events() on the probe traces, and a run without probe
    reads keeps the persistent kernel's 64-iteration batches;
  * argument and state errors."""
import numpy as np
import pytest

import cv_common as cv
from oracle.activation_np import ActivationMapNP

pytestmark = pytest.mark.gpu

BASE = {'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.0, 'duration': 1, 'timeline': False, 'timeline_name': 'x',
        'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False}
MAPS = ('first', 'last', 'previous', 'repol', 'count')


@pytest.fixture(scope='module')
def capi(cuda_device):
    from fib_tf_b200 import _capi
    return _capi


def _model(kind, H, W, hole=False, **extra):
    from cuda_adapter import CLASSES
    m = CLASSES[kind](dict(BASE, width=W, height=H, **extra))
    if kind in ('court', 'court_ultra'):
        m.chronic = True
    if hole:
        m.add_hole_to_phase_field(W // 2, H // 2, max(min(H, W) // 6, 2))
    m.define()
    return m


def _level(m):
    return float(m.min_v) + 0.5 * (float(m.max_v) - float(m.min_v))


def _perturb(m, seed=7):
    """A band of the potential around the level, so that cells cross it both ways within a few iterations."""
    rng = np.random.default_rng(seed)
    name, lv, span = m._pot_name, _level(m), float(m.max_v) - float(m.min_v)
    x = m._ctx.get_state(name)
    H = x.shape[0]
    band = slice(H // 4, H // 4 + max(H // 3, 1))
    x[band] = (lv + 0.3 * span * rng.uniform(-1.0, 1.0, x[band].shape)).astype(np.float32)
    m._ctx.set_state(name, x)


def _device_maps(ctx, capi):
    return [ctx.activation_get(k) for k in (capi.ACT_FIRST, capi.ACT_LAST, capi.ACT_PREV, capi.ACT_REPOL,
                                              capi.ACT_COUNT)]


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(np.asarray(a, np.float32).view(np.uint32),
                                                 np.asarray(b, np.float32).view(np.uint32))


def _assert_maps_equal(got, want, what=''):
    for name, g, w in zip(MAPS, got, want):
        assert _same_bits(g, w), (what, name, int(np.sum(g.view(np.uint32) != w.view(np.uint32))))


# ---- 1. bit for bit against the restatement, on the device's own samples -------------------------------------
ORACLE_CASES = [
    # kind, H, W, config extras, hole, slow every 10, stimulus, iterations, expected kernel name
    # (4v: a cell first repolarises after ~130 iterations of 1 ms)
    ('fenton4v', 48, 96, {'persist': False}, False, False, False, 250, 'step_kernel<Fenton4v'),
    ('fenton4v', 48, 96, {}, False, False, False, 250, 'persist_kernel<Fenton4v,TH=2,PHASE=0,ACT=1>'),
    ('fenton4v', 48, 96, {'persist': False}, True, False, True, 250, 'step_kernel<Fenton4v'),
    ('br', 40, 72, {'persist': False, 'cheby': True}, False, False, False, 120, 'BeelerReuter<cheby,slow>'),
    ('br', 40, 72, {'persist': False, 'cheby': True, 'skip': True}, False, False, False, 120, 'BeelerReuter<cheby,fast>'),
    ('br', 40, 72, {'persist': False}, False, False, False, 120, 'BeelerReuter<exact,slow>'),
    ('br', 40, 72, {'persist': False, 'skip': True}, False, False, True, 120, 'BeelerReuter<exact,fast>'),
    ('court', 32, 64, {}, False, True, False, 150, 'Courtemanche<fast>'),
    ('court_ultra', 32, 64, {}, False, False, False, 150, 'Courtemanche<all>'),
    ('court_ultra', 32, 64, {'lut': True}, True, False, True, 150, 'Courtemanche<all,lut>'),
]


@pytest.mark.parametrize('kind,H,W,extra,hole,slow,stim,iters,kernel', ORACLE_CASES,
                         ids=['%s-%d-%s%s%s' % (c[0], i, '-'.join('%s=%s' % kv for kv in sorted(c[3].items())),
                                                '-hole' if c[4] else '', '-stim' if c[6] else '')
                              for i, c in enumerate(ORACLE_CASES)])
def test_maps_equal_the_restatement_bit_for_bit(capi, kind, H, W, extra, hole, slow, stim, iters, kernel):
    m = _model(kind, H, W, hole=hole, **extra)
    m.add_pace_op('s2', 'luq', float(m.max_v))
    _perturb(m)
    ctx, name, lv = m._ctx, m._pot_name, _level(m)
    m.watch_activation()
    o = ActivationMapNP(ctx.get_state(name), lv, lv)
    kernels = set()
    for i in range(iters):
        ctx.step(m.ode_op(i), 1)
        kernels.add(capi.last_kernel())
        o.update(ctx.get_state(name))                  # the sample: before anything the driver does
        if slow and i % 10 == 0:
            m.fire_op('slow')
        if stim and i == iters // 3:
            m.fire_op('s2')
    assert any(kernel in k for k in kernels), (kernel, kernels)
    got = _device_maps(ctx, capi)
    _assert_maps_equal(got, o.planes(), kind)
    assert o.count.sum() > 0 and np.isfinite(o.repol).any()       # both kinds of event happened
    m.close()


# ---- 2. path invariance ------------------------------------------------------------------------------------
def _drive(m, iters, cut=None, capi=None):
    """Arm, step with the driver's stimulus schedule, return (maps, state)."""
    m.add_pace_op('s2', 'luq', float(m.max_v))
    _perturb(m)
    m.watch_activation()
    for i in range(iters):
        m._ctx.step(m.ode_op(i), 1)
        if i == iters // 2:
            m.fire_op('s2')
        if cut is not None and i == cut:
            m._ctx.activation_get(capi.ACT_LAST)
    maps = _device_maps(m._ctx, capi)
    state = {v: m._ctx.get_state(v) for v in m._ctx.var_names}
    return maps, state


def _compare(a, b, what):
    _assert_maps_equal(a[0], b[0], what)
    for v in a[1]:
        assert _same_bits(a[1][v], b[1][v]), (what, v)
    assert np.nansum(a[0][4]) > 0, what


@pytest.mark.parametrize('kind,extra', [('fenton4v', {}), ('br', {'cheby': True, 'skip': True})])
def test_graph_and_direct_launches_agree(capi, kind, extra):
    runs = []
    for graph in (True, False):
        m = _model(kind, 40, 600, persist=False, graph=graph, **extra)
        runs.append(_drive(m, 80, capi=capi))
        m.close()
    _compare(runs[0], runs[1], kind)


@pytest.mark.parametrize('kind,H,W,hole,th', [('fenton4v', 512, 512, True, 4), ('br', 512, 512, True, 4),
                                              ('fenton4v', 301, 500, False, 4), ('fenton4v', 1184, 300, True, 8),
                                              ('fenton4v', 64, 97, False, 2), ('br', 7, 5, False, 2)])
def test_persistent_kernel_agrees_with_one_launch_per_step(capi, kind, H, W, hole, th):
    runs = []
    for persist in (True, False):
        m = _model(kind, H, W, hole=hole, persist=persist)
        runs.append(_drive(m, 70, capi=capi))
        if persist:
            m._ctx.step(0, 1)
            m._ctx.flush()
            assert 'persist_kernel' in capi.last_kernel() and ',ACT=1>' in capi.last_kernel(), capi.last_kernel()
            assert 'TH=%d' % th in capi.last_kernel()
        m.close()
    _compare(runs[0], runs[1], (kind, H, W))


def test_two_steps_per_launch_agree_with_one(capi):
    runs = []
    for spl in (1, 2):
        m = _model('fenton4v', 64, 600, hole=True, persist=False, steps_per_launch=spl)
        assert m.steps_per_launch_used == spl
        runs.append(_drive(m, 60, capi=capi))
        m.close()
    _compare(runs[0], runs[1], 'fuse')


@pytest.mark.parametrize('kind,extra,spl', [('fenton4v', {}, 1), ('fenton4v', {}, 2), ('br', {'cheby': True}, 1),
                                            ('court_ultra', {}, 1)])
@pytest.mark.parametrize('nshards', [2, 3])
def test_in_process_shard_group_agrees_with_the_unsharded_run(capi, kind, extra, spl, nshards):
    from fib_tf_b200.sharding import partition_rows
    H, W, iters = 60, 200, 50
    ref = _model(kind, H, W, persist=False, **dict(extra, steps_per_launch=spl) if kind == 'fenton4v' else extra)
    _perturb(ref)
    init = {v: ref._ctx.get_state(v) for v in ref._ctx.var_names}
    ref.watch_activation()
    lv = _level(ref)
    for _ in range(iters):
        ref._ctx.step(capi.OP_ODE, 1)
    want = _device_maps(ref._ctx, capi)
    want_state = ref._ctx.get_state(ref._pot_name)
    flags = (capi.F_CHEBY if extra.get('cheby') else 0) | (ref._flags() if kind == 'court_ultra' else 0)
    ctxs = []
    for row0, rows in partition_rows(H, nshards):
        c = capi.Context(ref.MODEL_ID, H, W, ref.dt, ref.diff, flags=flags, row0=row0, rows=rows,
                         steps_per_launch=spl)
        for v, a in init.items():
            c.set_state(v, a[row0:row0 + rows])
        if extra.get('cheby'):
            c.set_table(capi.TABLE_BR_CHEBY, ref.chebyshev_table())
        c.activation_watch(lv, lv)
        ctxs.append(c)
    for _ in range(iters):
        capi.step_group(ctxs, capi.OP_ODE, 1)
    got = [np.concatenate(p, axis=0) for p in zip(*[_device_maps(c, capi) for c in ctxs])]
    _assert_maps_equal(got, want, (kind, nshards))
    assert _same_bits(np.concatenate([c.get_state(0) for c in ctxs]), want_state)
    assert want[4].sum() > 0
    for c in ctxs:
        c.close()
    ref.close()


def test_a_read_cutting_a_deferred_batch_changes_nothing(capi):
    a = _model('fenton4v', 512, 512)
    cut = _drive(a, 100, cut=37, capi=capi)
    b = _model('fenton4v', 512, 512)
    n0 = b._ctx.launch_count()
    whole = _drive(b, 100, capi=capi)
    assert b._ctx.launch_count() - n0 < 20                   # batched: a few persistent launches, not 100
    _compare(cut, whole, 'cut at 37')
    a.close()
    b.close()


def test_an_armed_map_turns_pipelined_uploads_into_ordered_copies(capi):
    H = W = 2048                                             # at least 2^22 cells: eligible for the pipeline
    runs = []
    for asynchronous in (True, False):
        m = _model('fenton4v', H, W, persist=False)
        _perturb(m)
        state = {v: m._ctx.get_state(v) for v in m._ctx.var_names}
        lv = _level(m)
        m._ctx.activation_watch(lv, lv)
        pinned = {v: capi.pinned_empty((H, W)) for v in state}
        for v in state:
            pinned[v][...] = state[v]
            pinned[v][:, :W // 3] = state[v][:, :W // 3] * np.float32(0.5)    # the upload changes the state
        for r in range(0, H, 512):
            for v in state:
                if asynchronous:
                    m._ctx.set_rect_async(v, r, 0, pinned[v][r:r + 512])
                else:
                    m._ctx.set_rect(v, r, 0, pinned[v][r:r + 512])
        if asynchronous:
            assert m._ctx.upload_state()[0] is False           # nothing to run behind the upload
        m._ctx.step(capi.OP_ODE, 6)
        runs.append((_device_maps(m._ctx, capi), {v: m._ctx.get_state(v) for v in state}))
        for v in state:
            capi.pinned_free(pinned[v])
        m.close()
    _compare(runs[0], runs[1], 'upload')


@pytest.mark.parametrize('persist', [True, False])
def test_rearming_resets_the_maps(capi, persist):
    m = _model('fenton4v', 64, 128, persist=persist)
    _perturb(m)
    ctx, lv = m._ctx, _level(m)
    m.watch_activation()
    ctx.step(capi.OP_ODE, 30)
    assert ctx.activation_get(capi.ACT_COUNT).sum() > 0
    m.watch_activation(up=0.4, down=0.6)
    first, count = ctx.activation_get(capi.ACT_FIRST), ctx.activation_get(capi.ACT_COUNT)
    assert np.isnan(first).all() and (count == 0).all()
    o = ActivationMapNP(ctx.get_state('U'), 0.4, 0.6)
    for _ in range(40):
        ctx.step(capi.OP_ODE, 1)
        o.update(ctx.get_state('U'))
    _assert_maps_equal(_device_maps(ctx, capi), o.planes(), 're-armed')
    m.stop_activation()
    with pytest.raises(capi.FibError):
        ctx.activation_get(capi.ACT_LAST)
    ctx.step(capi.OP_ODE, 3)                                  # stepping after stop: the graphs were rebuilt
    ctx.sync()
    m.close()


# ---- 3. the published CV table from the maps ------------------------------------------------------------
@pytest.mark.parametrize('kind,table', [('fenton4v', cv.CV_TABLE_4V), ('br', cv.CV_TABLE_BR)])
def test_published_cv_table_from_the_last_map(capi, kind, table):
    from cuda_adapter import CudaModel
    width = 700 if kind == 'fenton4v' else 520
    c1, c2 = (300, 600) if kind == 'fenton4v' else (200, 400)
    level = 0.5 if kind == 'fenton4v' else -30.0
    got, from_map = {}, {}
    for diff in sorted(table):
        m = CudaModel(kind, cv.strip_config(diff, width))
        m.define()
        m.m.watch_activation(level, level)
        dt_iter = m.m.dt_per_step * 0.1
        got[diff] = cv.measure_cv(m, level, c1, c2, dt_iter, 6000,
                                  lambda mm: mm.m._ctx.get_rect(mm.m._pot_name, 2, 3, 0, width)[0])
        last = m.m.activation_maps()['last'][2]
        from_map[diff] = (c2 - c1) / (last[c2] - last[c1])
        assert abs(from_map[diff] - got[diff]) <= 1e-5 * got[diff], (diff, from_map[diff], got[diff])
        m.close()
    dx, worst = cv.fit_dx(from_map, table)
    assert 0.0290 < dx < 0.0312, dx


# ---- 4. the reference's spiral runs ---------------------------------------------------------------------
def _spiral(which, read_probes):
    import test_spiral_statistics as ss
    from cuda_adapter import CLASSES
    meta, ref_probes, _ = ss.load(which)
    model = CLASSES['fenton4v' if which == 'fenton' else which](meta['config'])
    model.add_hole_to_phase_field(*meta['hole'])
    if meta.get('extra_hole'):
        model.add_hole_to_phase_field(*meta['extra_hole'])
    model.define()
    model.add_pace_op('s2', 'luq', meta['s2_value'])
    model.watch_activation()
    n0 = model._ctx.launch_count()
    probes = []
    if read_probes:                                     # sample s[0]: the plane the map was armed on
        probes.append([model._ctx.probe(model._pot_name, r, c) for r, c in meta['probes']])
    for i in model.run(None):
        if read_probes:
            probes.append([model._ctx.probe(model._pot_name, r, c) for r, c in meta['probes']])
        if i == meta['s2_iter']:
            model.fire_op('s2')
    launches = model._ctx.launch_count() - n0
    maps = model.activation_maps()
    raw = _device_maps(model._ctx, _capi_mod())
    samples = model.samples
    model.close()
    return meta, ref_probes, np.asarray(probes, np.float32), maps, raw, launches, samples


def _capi_mod():
    from fib_tf_b200 import _capi
    return _capi


@pytest.mark.parametrize('which', ['fenton', 'br'])
def test_spiral_run_maps_match_the_probe_traces(capi, which):
    import test_spiral_statistics as ss
    meta, ref_probes, probes, maps, raw, launches, samples = _spiral(which, True)
    lo, hi = {'fenton': (0.0, 1.0), 'br': (-90.0, 30.0)}[which]
    level = lo + 0.5 * (hi - lo)
    dt_iter = meta['dt_per_step'] * meta['config']['dt']
    s2_ms = meta['s2_iter'] * dt_iter
    assert probes.shape[0] == samples + 1
    compared = 0
    for k, (r, c) in enumerate(meta['probes']):
        # probes[j] is sample j of the map, so events() on it gives the map's times (in float64)
        up_c, dn_c = ss.events(probes[:, k], level, dt_iter)
        assert maps['count'][r, c] == len(up_c), (k, maps['count'][r, c], len(up_c))
        for key, want in (('first', up_c[:1]), ('last', up_c[-1:]), ('previous', up_c[-2:-1]), ('repol', dn_c[-1:])):
            if len(want):
                assert abs(maps[key][r, c] - want[0]) <= 1e-6 * want[0] + 1e-6, (k, key, maps[key][r, c], want[0])
            else:
                assert np.isnan(maps[key][r, c]), (k, key, maps[key][r, c])
        # against the reference's golden trace (its sample j is the map's sample j + 1): the first activation
        # before S2 within test_spiral_statistics.py's bound, the number of activations within one
        up_r, _ = ss.events(ref_probes[:, k], level, dt_iter)
        pre_r = up_r[up_r < s2_ms]
        if len(pre_r):
            assert abs(maps['first'][r, c] - dt_iter - pre_r[0]) <= 0.25 * dt_iter + 2e-3 * pre_r.max(), \
                (k, maps['first'][r, c], pre_r[0])
            compared += 1
        assert abs(maps['count'][r, c] - len(up_r)) <= 1, (k, maps['count'][r, c], len(up_r))
    assert compared >= 3
    if which == 'fenton':
        *_, raw2, launches2, _ = _spiral(which, False)
        _assert_maps_equal(raw2, raw, 'no probes')
        assert launches >= samples                                 # probe reads: one persistent launch per iteration
        assert launches2 <= samples // 64 + 8, launches2           # none: 64-iteration batches


# ---- 5. errors ------------------------------------------------------------------------------------------
def test_activation_errors(capi):
    import ctypes as C
    m = _model('fenton4v', 16, 32)
    ctx = m._ctx
    L = capi.lib()
    buf = np.empty(16 * 32, np.float32)
    p = buf.ctypes.data_as(C.c_void_p)
    assert L.fib_activation_get(ctx._h, capi.ACT_LAST, p, buf.size) == -4          # no watch: FIB_E_STATE
    assert 'armed' in L.fib_last_error().decode()
    assert L.fib_activation_watch(ctx._h, float('nan'), 0.5) == -1
    assert L.fib_activation_watch(ctx._h, 0.5, float('inf')) == -1
    assert 'finite' in L.fib_last_error().decode()
    m.watch_activation()
    assert L.fib_activation_get(ctx._h, capi.ACT_LAST, p, buf.size - 1) == -1        # wrong n
    assert L.fib_activation_get(ctx._h, 5, p, buf.size) == -1                       # unknown map
    assert L.fib_activation_get(ctx._h, -1, p, buf.size) == -1
    assert L.fib_activation_get(ctx._h, capi.ACT_COUNT, p, buf.size) == 0
    assert (buf == 0).all()
    m.stop_activation()
    m.stop_activation()                                                             # idempotent
    m.close()


# ---- 6. NCCL row shards -----------------------------------------------------------------------------------
@pytest.mark.parametrize('ranks', [2, 8])
def test_nccl_sharded_maps_equal_the_unsharded_maps(cuda_device, ranks):
    import os
    import socket
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < ranks:
        pytest.skip('needs >= %d GPUs, found %d' % (ranks, torch.cuda.device_count()))
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(ranks),
           '--master-addr', '127.0.0.1', '--master-port', str(port), os.path.join(root, 'tests', 'dist_activation.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    tail = '\n'.join((r.stdout + r.stderr).splitlines()[-30:])
    assert r.returncode == 0 and 'DIST ACTIVATION OK' in r.stdout, tail
