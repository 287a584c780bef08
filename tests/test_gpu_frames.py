"""GPU: the device-side frame recorder (include/fib_b200.h fib_frames_watch, IonicModel.record_frames / frames).

The reference for every check is a twin context: the same model, stepped through the same iterations, read back
with fib_get_state(var)[::stride, ::stride] at each recorded k.
  * bit for bit on every kernel family (graph and direct launches, two steps per launch, the persistent kernel
    for 4v and BR at TH = 2, 4 and 8 with partial last tiles, Courtemanche multi-rate with 'slow' and ultra with
    the LUT), strides 1, 3 and 8, first 0 and 1, potential and non-potential planes, asserting which
    instantiation ran;
  * the persistent kernel keeps its 64-iteration batches with the recorder armed;
  * recorder, activation map and probe ring together equal each armed alone;
  * in-process shard groups: the concatenated frames equal the unsharded frames;
  * ring overflow, re-arming, stop, errors; the pipelined-upload fall-back;
  * the reference's driver loop (fenton.py) against frames() on BASELINE config 1."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BASE = {'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.0, 'duration': 1, 'timeline': False, 'timeline_name': 'x',
        'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False}


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
    m.add_pace_op('s2', 'luq', float(m.max_v))
    return m


def _same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _recorded(k, first, every):
    return k >= first and (k - first) % every == 0


def _twin_run(make, var, first, every, stride, iters, slow=False, capacity=256):
    """The armed model, its (iters, frames), the twin's frames {k: plane[::s, ::s]} and the names of the
    kernels the armed model launched."""
    from fib_tf_b200 import _capi
    a, b = make(), make()
    a._ctx.frames_watch(var, first, every, stride, capacity)
    want, kernels = {}, set()
    if first == 0:
        want[0] = b._ctx.get_state(var)[::stride, ::stride]
    for i in range(iters):
        for m in (a, b):
            m._ctx.step(m.ode_op(i), 1)
            if m is a:
                kernels.add(_capi.last_kernel())
            elif _recorded(i + 1, first, every):
                want[i + 1] = b._ctx.get_state(var)[::stride, ::stride]
            if slow and i % 10 == 0:                        # what the driver does between iterations
                m.fire_op('slow')
            if i == iters // 2:
                m.fire_op('s2')
            if m is a:
                kernels.add(_capi.last_kernel())
    a._ctx.flush()
    kernels.add(_capi.last_kernel())
    got_k, got = a._ctx.frames_fetch(capacity)
    b.close()
    return a, got_k, got, want, kernels


def _assert_frames(got_k, got, want):
    assert [int(k) for k in got_k] == sorted(want), (list(got_k), sorted(want))
    for k, f in zip(got_k, got):
        assert _same_bits(f, want[int(k)]), (int(k), int(np.sum(f != want[int(k)])))


FAMILIES = [
    # kind, H, W, config extras, hole, var, stride, first, every, slow, kernel substring
    ('fenton4v', 41, 70, {'persist': False}, False, 'U', 3, 1, 10, False, 'step_kernel<Fenton4v'),
    ('fenton4v', 41, 70, {'persist': False, 'graph': False}, True, 'S', 8, 0, 7, False, 'step_kernel<Fenton4v'),
    ('fenton4v', 45, 68, {'persist': False, 'steps_per_launch': 2}, True, 'U', 3, 1, 5, False,
     'fenton_fused2_kernel<PHASE=1>'),
    ('fenton4v', 250, 77, {}, True, 'U', 1, 1, 10, False, 'persist_kernel<Fenton4v,TH=2,PHASE=1,FRAMES=1>'),
    ('fenton4v', 301, 100, {}, False, 'S', 3, 0, 10, False, 'persist_kernel<Fenton4v,TH=4,PHASE=0,FRAMES=1>'),
    ('fenton4v', 1183, 64, {}, True, 'U', 8, 1, 3, False, 'persist_kernel<Fenton4v,TH=8,PHASE=1,FRAMES=1>'),
    ('br', 150, 70, {'cheby': True}, True, 'V', 3, 1, 10, False, 'persist_kernel<BeelerReuter<cheby,slow>,TH=2,PHASE=1,FRAMES=1>'),
    ('br', 299, 50, {}, False, 'C', 8, 0, 4, False, 'persist_kernel<BeelerReuter<exact,slow>,TH=4,PHASE=0,FRAMES=1>'),
    ('br', 101, 90, {'cheby': True, 'skip': True}, True, 'V', 1, 1, 10, False,
     'persist_kernel<BeelerReuter<cheby,slow>,TH=2,PHASE=1,FRAMES=1>'),
    ('court', 33, 50, {}, False, 'V', 3, 1, 10, True, 'Courtemanche<fast>'),
    ('court_ultra', 35, 40, {'lut': True}, True, 'V', 8, 0, 6, False, 'Courtemanche<all,lut>'),
]


@pytest.mark.parametrize('kind,H,W,extra,hole,var,stride,first,every,slow,kernel', FAMILIES,
                         ids=['%s-%dx%d-%s-%s-s%d-f%d' % (c[0], c[1], c[2], '-'.join('%s=%s' % kv for kv in sorted(c[3].items())),
                                                        c[5], c[6], c[7]) for c in FAMILIES])
def test_frames_equal_the_twin_bit_for_bit(capi, kind, H, W, extra, hole, var, stride, first, every, slow, kernel):
    iters = 100                                            # not a multiple of 64: the last batch is partial
    a, got_k, got, want, ran = _twin_run(lambda: _model(kind, H, W, hole=hole, **extra), var, first, every,
                                         stride, iters, slow=slow)
    assert any(kernel in k for k in ran), (kernel, ran)
    assert a._ctx.frames_shape() == (-(-H // stride), -(-W // stride))
    _assert_frames(got_k, got, want)
    assert len(want) >= 10
    a.close()


def test_an_armed_recorder_keeps_the_persistent_batches(capi):
    counts = []
    for armed in (False, True):
        m = _model('fenton4v', 512, 512, hole=True)
        if armed:
            m._ctx.frames_watch('U', 1, 10, 1, 64)
        n0 = m._ctx.launch_count()
        m._ctx.step(capi.OP_ODE, 64)
        for _ in range(64):
            m._ctx.step(capi.OP_ODE, 1)
        counts.append(m._ctx.launch_count() - n0)
        if armed:
            k, f = m._ctx.frames_fetch(64)
            assert list(k) == list(range(1, 129, 10)) and f.shape == (13, 512, 512)
        m.close()
    assert counts == [2, 2], counts


@pytest.mark.parametrize('persist', [True, False])
def test_observers_together_equal_each_alone(capi, persist):
    def run(frames, act, probe):
        m = _model('fenton4v', 200, 120, hole=True, persist=persist)
        if frames:
            m._ctx.frames_watch('U', 1, 3, 3, 64)
        if act:
            m.watch_activation()
        if probe:
            m._ctx.probe_watch('U', 20, 60)
        for i in range(90):
            m._ctx.step(capi.OP_ODE, 1)
            if i == 40:
                m.fire_op('s2')
        out = {}
        if frames:
            out['frames'] = m._ctx.frames_fetch(64)
        if act:
            out['act'] = m._ctx.activation_get(capi.ACT_LAST)
        if probe:
            out['probe'] = m._ctx.probe_fetch(200)
        out['state'] = m._ctx.get_state('U')
        m.close()
        return out
    both = run(True, True, True)
    fr, act, pr = run(True, False, False), run(False, True, False), run(False, False, True)
    assert list(both['frames'][0]) == list(fr['frames'][0]) and len(fr['frames'][0]) == 30
    assert _same_bits(both['frames'][1], fr['frames'][1])
    assert _same_bits(both['act'], act['act'])
    assert _same_bits(both['probe'], pr['probe']) and len(pr['probe']) == 90
    for o in (fr, act, pr):
        assert _same_bits(both['state'], o['state'])


@pytest.mark.parametrize('kind,extra', [('fenton4v', {}), ('fenton4v', {'steps_per_launch': 2}),
                                        ('br', {'cheby': True}), ('court_ultra', {})])
@pytest.mark.parametrize('nshards', [2, 3])
def test_shard_group_frames_concatenate_to_the_unsharded_frames(capi, kind, extra, nshards):
    from fib_tf_b200.sharding import partition_rows
    H, W, iters, stride = 61, 52, 40, 3
    spl = extra.get('steps_per_launch', 1)
    ref = _model(kind, H, W, persist=False, **extra)
    init = {v: ref._ctx.get_state(v) for v in ref._ctx.var_names}
    ref._ctx.frames_watch(0, 0, 4, stride, 32)
    for _ in range(iters):
        ref._ctx.step(capi.OP_ODE, 1)
    want_k, want = ref._ctx.frames_fetch(32)
    flags = (capi.F_CHEBY if extra.get('cheby') else 0) | (ref._flags() if kind == 'court_ultra' else 0)
    ctxs = []
    parts = partition_rows(H, nshards)
    assert any(rows % stride for _, rows in parts)
    for row0, rows in parts:
        c = capi.Context(ref.MODEL_ID, H, W, ref.dt, ref.diff, flags=flags, row0=row0, rows=rows,
                         steps_per_launch=spl)
        for v, a in init.items():
            c.set_state(v, a[row0:row0 + rows])
        if extra.get('cheby'):
            c.set_table(capi.TABLE_BR_CHEBY, ref.chebyshev_table())
        c.frames_watch(0, 0, 4, stride, 32)
        ctxs.append(c)
    for _ in range(iters):
        capi.step_group(ctxs, capi.OP_ODE, 1)
    fetched = [c.frames_fetch(32) for c in ctxs]
    for k, _ in fetched:
        assert list(k) == list(want_k) == list(range(0, iters + 1, 4))
    got = np.concatenate([f for _, f in fetched], axis=1)
    assert _same_bits(got, want)
    for c in ctxs:
        c.close()
    ref.close()


@pytest.mark.parametrize('persist', [True, False])
def test_ring_overflow_rearm_and_stop(capi, persist):
    m = _model('fenton4v', 64, 50, persist=persist)
    ctx = m._ctx
    ctx.frames_watch('U', 1, 2, 1, 4)
    want = {}
    twin = _model('fenton4v', 64, 50, persist=persist)
    for i in range(30):
        ctx.step(capi.OP_ODE, 1)
        twin._ctx.step(capi.OP_ODE, 1)
        want[i + 1] = twin._ctx.get_state('U')
    k, f = ctx.frames_fetch(10)
    assert list(k) == [23, 25, 27, 29]                     # the newest four, with their k
    for kk, ff in zip(k, f):
        assert _same_bits(ff, want[int(kk)])
    assert len(ctx.frames_fetch(10)[0]) == 0
    ctx.step(capi.OP_ODE, 3)
    ctx.frames_watch('U', 0, 1, 2, 8)                      # re-arm: reset, k = 0 re-taken
    assert ctx.frames_shape() == (32, 25)
    k, f = ctx.frames_fetch(10)
    assert list(k) == [0] and _same_bits(f[0], ctx.get_state('U')[::2, ::2])
    ctx.step(capi.OP_ODE, 2)
    assert list(ctx.frames_fetch(10)[0]) == [1, 2]
    ctx.frames_stop()
    L = capi.lib()
    n = C.c_size_t()
    buf = np.empty(64 * 50, np.float32)
    it = np.empty(1, np.uint64)
    assert L.fib_frames_fetch(ctx._h, buf.ctypes.data_as(C.c_void_p), it.ctypes.data_as(C.POINTER(C.c_uint64)),
                              1, C.byref(n)) == -4          # FIB_E_STATE: the ring is gone
    r, c = C.c_int(), C.c_int()
    assert L.fib_frames_shape(ctx._h, C.byref(r), C.byref(c)) == -4
    ctx.step(capi.OP_ODE, 3)                               # stepping after stop records nothing, fails nothing
    ctx.sync()
    ctx.frames_stop()                                      # idempotent
    twin.close()
    m.close()


def test_frames_errors(capi):
    m = _model('fenton4v', 16, 32)
    L = capi.lib()
    h = m._ctx._h
    n = C.c_size_t()
    assert L.fib_frames_fetch(h, None, None, 0, C.byref(n)) == -4                # no watch: FIB_E_STATE
    assert 'armed' in L.fib_last_error().decode()
    for args in ((0, 1, 0, 1, 4), (0, 1, 1, 0, 4), (0, 1, 1, 1, 0), (0, -1, 1, 1, 4), (4, 1, 1, 1, 4), (-1, 1, 1, 1, 4)):
        assert L.fib_frames_watch(h, *args) == -1, args
    assert L.fib_frames_watch(h, 0, 1, 1, 1, 1 << 30) == -2                      # 2^30 frames of 2 KiB: no memory
    m.close()


def test_an_armed_recorder_turns_pipelined_uploads_into_ordered_copies(capi):
    H = W = 2048                                           # at least 2^22 cells: eligible for the pipeline
    runs = []
    for asynchronous in (True, False):
        m = _model('fenton4v', H, W, persist=False)
        state = {v: m._ctx.get_state(v) for v in m._ctx.var_names}
        m._ctx.frames_watch('U', 1, 1, 8, 16)
        pinned = {v: capi.pinned_empty((H, W)) for v in state}
        for v in state:
            pinned[v][...] = state[v]
            pinned[v][:, :W // 3] = state[v][:, :W // 3] * np.float32(0.5)
        for r in range(0, H, 512):
            for v in state:
                if asynchronous:
                    m._ctx.set_rect_async(v, r, 0, pinned[v][r:r + 512])
                else:
                    m._ctx.set_rect(v, r, 0, pinned[v][r:r + 512])
        if asynchronous:
            assert m._ctx.upload_state()[0] is False       # nothing runs behind the upload
        m._ctx.step(capi.OP_ODE, 6)
        runs.append((m._ctx.frames_fetch(16), m._ctx.get_state('U')))
        for v in state:
            capi.pinned_free(pinned[v])
        m.close()
    (ka, fa), ua = runs[0]
    (kb, fb), ub = runs[1]
    assert list(ka) == list(kb) == [1, 2, 3, 4, 5, 6]
    assert _same_bits(fa, fb) and _same_bits(ua, ub) and _same_bits(fa[-1], ua[::8, ::8])


def test_the_reference_driver_loop_equals_frames(capi):
    """fenton.py's loop, cube[i // 10] = model.image() * model.phase, against record_frames(10) / frames()
    on BASELINE config 1 (512^2 with a hole), 300 iterations: bit for bit, the S2 frame up to the stimulus the
    loop fires before grabbing it."""
    from fib_tf_b200.fenton import Fenton4v
    cfg = {'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 300,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False}
    cubes, launches = [], []
    for recorder in (False, True):
        model = Fenton4v(cfg)
        model.add_hole_to_phase_field(256, 256, 30)
        model.define()
        model.add_pace_op('s2', 'luq', 1.0)
        s2, every = model.millisecond_to_step(210), model.millisecond_to_step(10)
        cube = np.zeros([int(model.duration / 10.0), model.height, model.width], dtype=np.float32)
        if recorder:
            model.record_frames(every)
        n0 = model._ctx.launch_count()
        for i in model.run(None):
            if i == s2:
                model.fire_op('s2')
            if not recorder and i % every == 0:
                cube[i // every] = model.image() * model.phase
        launches.append(model._ctx.launch_count() - n0)
        if recorder:
            iters, frames = model.frames()
            assert list(iters) == list(range(1, 300, 10))
            assert 'FRAMES=1' in capi.last_kernel(), capi.last_kernel()
            # The loop grabs frame s2 // every AFTER firing s2 in the same loop body; the recorder takes every
            # frame before the caller acts (k = 211 ends before the stimulus).  That frame is the recorded one
            # with the stimulus applied: U := max(U, 1 inside 'luq', min_v elsewhere).
            assert s2 % every == 0
            stim = np.full((512, 512), np.float32(model.min_v), np.float32)
            stim[1:256, 1:256] = np.float32(1.0)
            stimulated = np.maximum(frames[s2 // every], stim) * model.phase
            cube = frames * model.phase
        cubes.append(cube)
        model.close()
    j = s2 // every
    others = [f for f in range(30) if f != j]
    assert _same_bits(cubes[0][others], cubes[1][others])
    assert not _same_bits(cubes[0][j], cubes[1][j])
    assert _same_bits(cubes[0][j], stimulated)
    assert launches[0] >= 30 and launches[1] <= 8, launches     # the grabs cut the batches; the recorder does not


@pytest.mark.parametrize('ranks', [2])
def test_nccl_sharded_frames_equal_the_unsharded_frames(cuda_device, ranks):
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
           '--master-addr', '127.0.0.1', '--master-port', str(port), os.path.join(root, 'tests', 'dist_frames.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    tail = '\n'.join((r.stdout + r.stderr).splitlines()[-30:])
    assert r.returncode == 0 and 'DIST FRAMES OK' in r.stdout, tail
