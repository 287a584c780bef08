"""GPU: pacing on the device (include/fib_b200.h fib_pace_add / fib_pace_remove, IonicModel.pace / stop_pacing).

The reference for every check is a twin context: the same model, stepped through the same iterations, with
fib_stimulate called after each iteration at which an entry fires.  Every plane must be equal bit for bit.
  * every kernel family: the persistent kernel for 4v and BR (TH = 2 and 4, BR's skip schedule included), graph and
    direct launches, two steps per launch, Courtemanche multi-rate with 'slow' interleaved and ultra with the LUT,
    asserting which instantiation ran; several entries firing at the same k, count = 0 until removal, removal
    mid-run;
  * probe ring, activation maps and frames armed together: the probe after the stimulus, maps and frames before;
  * in-process shard groups with a rectangle across the seams, fired inside one multi-iteration fib_step_group;
  * a burst train on BASELINE config 1 keeps the persistent kernel's batches;
  * checkpoint mid-train and restore continue bit for bit with the uninterrupted run;
  * fenton.py's config 1 loop with pace('s2', s2) equals the loop with fire_op('s2')."""
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
    return m


def _same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _fires(k, first, every, count):
    if k < first:
        return False
    if count == 1:
        return k == first
    return (k - first) % every == 0 and (count == 0 or (k - first) // every < count)


def _schedule(m, H, W):
    """Entries (rect, value, floor, first, every, count): a train until removed, a finite train that shares beats
    with it, and a single beat on the same k as both."""
    hi, lo = float(m.max_v), float(m.min_v)
    return [((1, H // 2, 1, W // 2), hi, lo, 5, 7, 0),
            ((H // 3, 2 * H // 3, 0, 5), hi, lo, 12, 7, 4),
            ((0, H, W - 6, W), 0.8 * hi, lo, 19, 0, 1)]


def _twin_run(make, H, W, iters, remove_at=None, slow=False, observe=None):
    """Steps the paced model `a` and its twin `b` (fib_stimulate at the same iterations) one iteration per fib_step;
    `remove_at`: the first entry is removed after that iteration.  Returns a, b and the kernels `a` launched."""
    from fib_tf_b200 import _capi
    a, b = make(), make()
    sched = _schedule(a, H, W)
    ids = [a._ctx.pace_add(*rect, v, fl, first, every, count) for rect, v, fl, first, every, count in sched]
    live = [True] * len(sched)
    if observe:
        for m in (a, b):
            observe(m)
    kernels = set()
    pot = a._pot_name
    for i in range(iters):
        for m in (a, b):
            m._ctx.step(m.ode_op(i), 1)
            if m is a:
                kernels.add(_capi.last_kernel())
            else:
                for e, (rect, v, fl, first, every, count) in enumerate(sched):
                    if live[e] and _fires(i + 1, first, every, count):
                        b._ctx.stimulate(pot, *rect, v, fl)
            if slow and i % 10 == 0:
                m.fire_op('slow')
        if i == remove_at:
            a._ctx.pace_remove(ids[0])
            live[0] = False
    a._ctx.flush()
    kernels.add(_capi.last_kernel())
    return a, b, kernels


def _assert_twins(a, b):
    for v in a._ctx.var_names:
        assert _same_bits(a._ctx.get_state(v), b._ctx.get_state(v)), v


FAMILIES = [
    # kind, H, W, config extras, hole, slow, kernel substring
    ('fenton4v', 250, 77, {}, True, False, 'persist_kernel<Fenton4v,TH=2,PHASE=1,PACE=1>'),
    ('fenton4v', 301, 100, {}, False, False, 'persist_kernel<Fenton4v,TH=4,PHASE=0,PACE=1>'),
    ('br', 150, 70, {'cheby': True}, True, False, 'persist_kernel<BeelerReuter<cheby,slow>,TH=2,PHASE=1,PACE=1>'),
    ('br', 299, 50, {}, False, False, 'persist_kernel<BeelerReuter<exact,slow>,TH=4,PHASE=0,PACE=1>'),
    ('br', 101, 90, {'cheby': True, 'skip': True}, True, False,
     'persist_kernel<BeelerReuter<cheby,slow>,TH=2,PHASE=1,PACE=1>'),
    ('fenton4v', 41, 70, {'persist': False}, True, False, 'step_kernel<Fenton4v'),
    ('fenton4v', 41, 70, {'persist': False, 'graph': False}, True, False, 'step_kernel<Fenton4v'),
    ('fenton4v', 45, 68, {'persist': False, 'steps_per_launch': 2}, True, False, 'fenton_fused2_kernel<PHASE=1>'),
    ('court', 33, 50, {}, False, True, 'Courtemanche<fast>'),
    ('court_ultra', 35, 40, {'lut': True}, True, False, 'Courtemanche<all,lut>'),
]


@pytest.mark.parametrize('kind,H,W,extra,hole,slow,kernel', FAMILIES,
                         ids=['%s-%dx%d-%s' % (c[0], c[1], c[2], '-'.join('%s=%s' % kv for kv in sorted(c[3].items())))
                              for c in FAMILIES])
def test_pacing_equals_the_twin_bit_for_bit(capi, kind, H, W, extra, hole, slow, kernel):
    iters = 100                                            # not a multiple of 64: the last batch is partial
    a, b, ran = _twin_run(lambda: _model(kind, H, W, hole=hole, **extra), H, W, iters, remove_at=60, slow=slow)
    assert any(kernel in k for k in ran), (kernel, ran)
    _assert_twins(a, b)
    a.close()
    b.close()


@pytest.mark.parametrize('persist', [True, False])
def test_observers_see_the_stimulus_as_after_fib_stimulate(capi, persist):
    """Probe after the stimulus, activation maps and frames before it: all equal to the twin's."""
    def observe(m):
        m._ctx.frames_watch('U', 1, 1, 1, 128)
        m.watch_activation()
        m._ctx.probe_watch('U', 30, 10)
    a, b, ran = _twin_run(lambda: _model('fenton4v', 200, 120, hole=True, persist=persist), 200, 120, 90,
                          remove_at=50, observe=observe)
    if persist:
        assert any('FRAMES=1,PACE=1' in k and 'ACT=1' in k for k in ran), ran
    ka, fa = a._ctx.frames_fetch(128)
    kb, fb = b._ctx.frames_fetch(128)
    assert list(ka) == list(kb) == list(range(1, 91))
    assert _same_bits(fa, fb)
    for which in (capi.ACT_FIRST, capi.ACT_LAST, capi.ACT_PREV, capi.ACT_REPOL, capi.ACT_COUNT, capi.ACT_SAMPLE):
        assert _same_bits(a._ctx.activation_get(which), b._ctx.activation_get(which)), which
    pa, pb = a._ctx.probe_fetch(200), b._ctx.probe_fetch(200)
    assert len(pa) == 90 and _same_bits(pa, pb)
    # the probe cell lies in the first entry's rectangle: after iteration 5 the probe holds the stimulated value,
    # the frame the value before the stimulus
    assert pa[4] == max(fa[4][30, 10], np.float32(a.max_v))
    _assert_twins(a, b)
    a.close()
    b.close()


@pytest.mark.parametrize('kind,extra', [('fenton4v', {}), ('fenton4v', {'steps_per_launch': 2}),
                                        ('br', {'cheby': True})])
@pytest.mark.parametrize('nshards', [2, 3])
def test_shard_group_beats_on_the_seams(capi, kind, extra, nshards):
    """A rectangle across every seam, fired inside fib_step_group(n) calls: equal to the unsharded twin."""
    from fib_tf_b200.sharding import partition_rows
    H, W, iters = 61, 52, 40
    spl = extra.get('steps_per_launch', 1)
    ref = _model(kind, H, W, hole=True, persist=False, **extra)
    init = {v: ref._ctx.get_state(v) for v in ref._ctx.var_names}
    beats = (3, 5, 6, 17, 18)                               # k: consecutive beats too
    rect, v, fl = (2, H - 2, 10, 30), float(ref.max_v), float(ref.min_v)
    for i in range(iters):
        ref._ctx.step(capi.OP_ODE, 1)
        if i + 1 in beats:
            ref._ctx.stimulate(0, *rect, v, fl)
    flags = capi.F_CHEBY if extra.get('cheby') else 0
    ctxs = []
    for row0, rows in partition_rows(H, nshards):
        c = capi.Context(ref.MODEL_ID, H, W, ref.dt, ref.diff, flags=flags, row0=row0, rows=rows,
                         steps_per_launch=spl)
        for name, a in init.items():
            c.set_state(name, a[row0:row0 + rows])
        c.set_phase(ref.phase, 0)
        if extra.get('cheby'):
            c.set_table(capi.TABLE_BR_CHEBY, ref.chebyshev_table())
        c.pace_add(*rect, v, fl, 3, 2, 2)                  # k = 3, 5
        c.pace_add(*rect, v, fl, 6, 11, 0)                 # k = 6, 17, 28, ... until removed
        c.pace_add(*rect, v, fl, 18, 0, 1)                 # k = 18
        ctxs.append(c)
    capi.step_group(ctxs, capi.OP_ODE, 20)                 # every beat but the last inside this call
    for c in ctxs:
        c.pace_remove(1)
    capi.step_group(ctxs, capi.OP_ODE, iters - 20)
    for name in ref._ctx.var_names:
        got = np.concatenate([c.get_state(name) for c in ctxs])
        assert _same_bits(got, ref._ctx.get_state(name)), name
    for c in ctxs:
        c.close()
    ref.close()


def test_a_burst_train_keeps_the_persistent_batches(capi):
    """BASELINE config 1 (512^2 with a hole), 640 iterations one fib_step at a time, a burst every 4 iterations:
    the same launches as with no train."""
    counts, states = [], []
    for train in (False, True):
        m = _model('fenton4v', 512, 512, hole=True, diff=1.5)
        if train:
            m._ctx.pace_add(1, 256, 1, 256, 1.0, float(m.min_v), 3, 4, 150)
        n0 = m._ctx.launch_count()
        for _ in range(640):
            m._ctx.step(capi.OP_ODE, 1)
        counts.append(m._ctx.launch_count() - n0)
        if train:
            assert 'PACE=1' in capi.last_kernel(), capi.last_kernel()
        states.append(m._ctx.get_state('U'))
        m.close()
    assert counts == [10, 10], counts
    assert not _same_bits(states[0], states[1])


def test_errors_and_limits(capi):
    import ctypes as C
    m = _model('fenton4v', 16, 32)
    L, h = capi.lib(), m._ctx._h
    i = C.c_int()
    for first, every, count in ((0, 1, 1), (1, 0, 2), (1, 0, 0), (1, 1, -1)):
        assert L.fib_pace_add(h, 0, 1, 0, 1, 1.0, 0.0, first, every, count, C.byref(i)) == -1, (first, every, count)
    ids = [m._ctx.pace_add(0, 4, 0, 4, 1.0, 0.0, 1, 0, 1) for _ in range(4)]
    assert ids == [0, 1, 2, 3]
    assert L.fib_pace_add(h, 0, 1, 0, 1, 1.0, 0.0, 1, 0, 1, C.byref(i)) == -4      # a fifth: FIB_E_STATE
    m._ctx.step(capi.OP_ODE, 1)                                                    # all four fire and finish
    assert m._ctx.pace_add(0, 4, 0, 4, 1.0, 0.0, 1, 0, 1) == 4
    m._ctx.pace_remove(0)                                                          # finished: a no-op
    assert L.fib_pace_remove(h, 5) == -1                                           # never handed out
    m._ctx.pace_remove(-1)
    m._ctx.step(capi.OP_ODE, 2)
    m.close()


def _config1(duration, persist=True):
    from fib_tf_b200.fenton import Fenton4v
    model = Fenton4v({'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': duration,
                      'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'persist': persist})
    model.add_hole_to_phase_field(256, 256, 30)
    return model


def test_checkpoint_mid_train_restores_bit_for_bit(capi, tmp_path):
    whole = _config1(200)
    whole.define()
    whole.add_pace_op('s1', 'left', 1.0)
    whole.add_pace_op('s2', 'luq', 1.0)
    whole.pace('s1', 10, 30, 6)                            # after 11, 41, ..., 161
    whole.pace('s2', 120, 0, 1)
    for _ in whole.run():
        pass
    want = {v: whole._ctx.get_state(v) for v in whole._ctx.var_names}
    whole.close()

    first = _config1(100)
    first.define()
    first.add_pace_op('s1', 'left', 1.0)
    first.add_pace_op('s2', 'luq', 1.0)
    first.pace('s1', 10, 30, 6)
    first.pace('s2', 120, 0, 1)
    for _ in first.run():
        pass
    first.checkpoint(str(tmp_path / 'ck')).wait()
    first.close()
    from fib_tf_b200 import checkpoint as ck
    man = ck.load_manifest(str(tmp_path / 'ck'))
    assert sorted((p['name'], p['next'], p['count']) for p in man['pacing']) == [('s1', 101, 3), ('s2', 121, 1)]

    second = _config1(100)
    second.restore(str(tmp_path / 'ck'))
    assert second.iterations == 100
    for _ in second.run():
        pass
    for v, a in want.items():
        assert _same_bits(second._ctx.get_state(v), a), v
    second.close()


def test_the_reference_driver_loop_with_pace(capi):
    """fenton.py's config 1 loop, 300 iterations: pace('s2', s2) before the loop equals fire_op('s2') inside it,
    with fewer launches."""
    states, launches = [], []
    for paced in (False, True):
        model = _config1(300)
        model.define()
        model.add_pace_op('s2', 'luq', 1.0)
        s2 = model.millisecond_to_step(210)
        if paced:
            model.pace('s2', s2)
        n0 = model._ctx.launch_count()
        for i in model.run(None):
            if not paced and i == s2:
                model.fire_op('s2')
        launches.append(model._ctx.launch_count() - n0)
        states.append({v: model._ctx.get_state(v) for v in model._ctx.var_names})
        model.close()
    for v in states[0]:
        assert _same_bits(states[0][v], states[1][v]), v
    assert launches[1] < launches[0], launches


@pytest.mark.parametrize('ranks', [2])
def test_nccl_sharded_pacing_equals_the_unsharded_run(cuda_device, ranks):
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
           '--master-addr', '127.0.0.1', '--master-port', str(port), os.path.join(root, 'tests', 'dist_pacing.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    tail = '\n'.join((r.stdout + r.stderr).splitlines()[-30:])
    assert r.returncode == 0 and 'DIST PACING OK' in r.stdout, tail
