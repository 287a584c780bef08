"""GPU: checkpoint and restart (include/fib_b200.h fib_checkpoint_*, fib_tf_b200/checkpoint.py, IonicModel.checkpoint /
restore).  Run A steps 2n iterations uninterrupted; run B steps n, checkpoint(), n more in the same model (the
save overlaps them); run C is a fresh model that restore()s B's checkpoint and steps n.  B's and C's final planes
must equal A's bit for bit:
  * on every kernel family, asserting the instantiation that ran: 4v one and two steps per launch, the persistent
    kernel on BASELINE config 1 (512^2 + hole), BR cheby / exact / skip, Courtemanche multi-rate with 'slow'
    every 10 iterations, ultra with _us_ and with the LUT;
  * the checkpoint holds the state at iteration n although n more iterations were enqueued before its writer
    finished;
  * with an activation map and a frame recorder armed before iteration 0: C's six map planes and frames equal A's;
  * saved from two in-process shard contexts, restored into one unsharded context and into three shards;
  * a 2048^2 4v restore with nothing armed steps behind its own upload;
  * NCCL shards (tests/dist_checkpoint.py) when at least two GPUs are visible."""
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
    return m


def _same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _drive(m, n, slow, s2, kernels, at=None):
    """n iterations through run(), the driver's schedule offset by model.iterations: 'slow' every 10, S2 once.
    at = (iteration, callback): called after that global iteration."""
    from fib_tf_b200 import _capi
    i0 = m.iterations
    m.duration = n * m.dt_per_step * m.dt * (1 + 1e-9)
    for i in m.run(None, block=False):
        g = i0 + i
        kernels.add(_capi.last_kernel())
        if slow and g % 10 == 0:
            m.fire_op('slow')
        if g == s2:
            m.fire_op('s2')
        if at is not None and g == at[0]:
            at[1]()
    kernels.add(_capi.last_kernel())
    assert m.iterations == i0 + n


def _planes(m):
    return {v: m._ctx.get_state(v) for v in m._ctx.var_names}


def _abc(tmp_path, make, n, slow=False, observers=False):
    """(A, B, C, planes of A at iteration n, kernels A ran, path)."""
    from fib_tf_b200 import checkpoint as ck
    path = str(tmp_path / 'ck')
    s2 = n // 2 + 1
    kernels = {'A': set(), 'B': set(), 'C': set()}
    A, B = make(), make()
    for m in (A, B):
        m.define()
        m.add_pace_op('s2', 'luq', float(m.max_v))
        if observers:
            m.watch_activation()
            m.record_frames(every=3, stride=2, first=1, capacity=256)
    at_n = {}
    _drive(A, 2 * n, slow, s2, kernels['A'], at=(n - 1, lambda: at_n.update(_planes(A))))
    _drive(B, n, slow, s2, kernels['B'])
    h = B.checkpoint(path)
    _drive(B, n, slow, s2, kernels['B'])             # enqueued while the writer runs
    h.wait()
    for v, want in at_n.items():
        assert _same_bits(ck.read_rows(path, v, 0, A.height), want), ('checkpoint is not iteration n', v)
    C = make()
    C.restore(path)
    assert C.iterations == n
    C.add_pace_op('s2', 'luq', float(C.max_v))
    _drive(C, n, slow, s2, kernels['C'])
    return A, B, C, kernels, path


FAMILIES = [
    # kind, H, W, config extras, hole, slow, kernel substring
    ('fenton4v', 41, 70, {'persist': False}, False, False, 'step_kernel<Fenton4v'),
    ('fenton4v', 45, 68, {'persist': False, 'steps_per_launch': 2}, True, False, 'fenton_fused2_kernel<PHASE=1>'),
    ('fenton4v', 512, 512, {'diff': 1.5}, True, False, 'persist_kernel<Fenton4v,TH=4,PHASE=1>'),
    ('br', 150, 70, {'cheby': True}, True, False, 'persist_kernel<BeelerReuter<cheby,slow>'),
    ('br', 299, 50, {'persist': False}, False, False, 'BeelerReuter<exact'),
    ('br', 101, 90, {'cheby': True, 'skip': True}, True, False, 'persist_kernel<BeelerReuter<cheby,slow>'),
    ('court', 33, 50, {}, False, True, 'Courtemanche<fast>'),
    ('court_ultra', 35, 40, {'ultra_slow': True}, True, True, 'Courtemanche<all,us>'),
    ('court_ultra', 35, 40, {'lut': True}, True, False, 'Courtemanche<all,lut>'),
]


@pytest.mark.parametrize('kind,H,W,extra,hole,slow,kernel', FAMILIES,
                         ids=['%s-%dx%d-%s' % (c[0], c[1], c[2], '-'.join('%s=%s' % kv for kv in sorted(c[3].items())))
                              for c in FAMILIES])
def test_restored_run_equals_the_uninterrupted_run(capi, tmp_path, kind, H, W, extra, hole, slow, kernel):
    n = 40 if kind.startswith('court') else 70             # 70: not a multiple of the persistent batch
    A, B, C, ran, _ = _abc(tmp_path, lambda: _model(kind, H, W, hole=hole, **extra), n, slow=slow)
    for who in 'ABC':
        assert any(kernel in k for k in ran[who]), (who, kernel, ran[who])
    for v in A._ctx.var_names:
        a = A._ctx.get_state(v)
        assert _same_bits(B._ctx.get_state(v), a), ('B', v)
        assert _same_bits(C._ctx.get_state(v), a), ('C', v)
    for m in (A, B, C):
        m.close()


@pytest.mark.parametrize('kind,extra', [('fenton4v', {}), ('fenton4v', {'persist': False, 'graph': False}),
                                        ('br', {'cheby': True, 'skip': True})])
def test_observers_armed_before_iteration_zero_continue(capi, tmp_path, kind, extra):
    n = 70
    A, B, C, ran, path = _abc(tmp_path, lambda: _model(kind, 200, 120, hole=True, **extra), n, observers=True)
    from fib_tf_b200 import checkpoint as ck
    for which in ck._ACT_MAPS:
        assert _same_bits(C._ctx.activation_get(which), A._ctx.activation_get(which)), which
        assert _same_bits(B._ctx.activation_get(which), A._ctx.activation_get(which)), which
    a_k, a_cube = A.frames()
    c_k, c_cube = C.frames()
    assert list(c_k) == [k for k in a_k if k > n] and len(c_k) >= 20
    assert _same_bits(c_cube, a_cube[len(a_k) - len(c_k):])
    b_k, b_cube = B.frames()
    assert list(b_k) == list(a_k) and _same_bits(b_cube, a_cube)
    for m in (A, B, C):
        m.close()


def _contexts(capi, H, W, n_shards, init):
    out = []
    for row0, rows in __import__('fib_tf_b200.sharding', fromlist=['x']).partition_rows(H, n_shards):
        c = capi.Context(capi.FENTON4V, H, W, 0.1, 1.3, flags=capi.F_NO_PERSIST,
                         row0=row0 if n_shards > 1 else 0, rows=rows if n_shards > 1 else 0)
        if init is not None:
            for v, a in init.items():
                c.set_state(v, a[row0:row0 + rows])
        out.append(c)
    return out


def _step(capi, ctxs, n):
    if len(ctxs) == 1:
        ctxs[0].step(capi.OP_ODE, n)
    else:
        capi.step_group(ctxs, capi.OP_ODE, n)


def test_shard_groups_save_and_restore_on_other_partitions(capi, tmp_path):
    from fib_tf_b200 import checkpoint as ck
    H, W, n = 91, 64, 30
    rng = np.random.default_rng(7)
    init = {'U': rng.uniform(0, 1, (H, W)).astype(np.float32), 'V': np.ones((H, W), np.float32),
            'W': np.ones((H, W), np.float32), 'S': np.zeros((H, W), np.float32)}
    init['U'][:, :8] = 1.0
    (a,) = _contexts(capi, H, W, 1, init)
    _step(capi, [a], 2 * n)
    want = {v: a.get_state(v) for v in a.var_names}
    group = _contexts(capi, H, W, 2, init)
    _step(capi, group, n)
    path = str(tmp_path / 'ck')
    import os
    os.makedirs(path)
    writers = [ck.save_shard(c, path) for c in group]
    _step(capi, group, n)
    assert all(w.join() for w in writers), [w.error for w in writers]
    ck.write_manifest(path, ck.manifest(group[0], writers[0].info, [w.record for w in writers]))
    man = ck.load_manifest(path)
    assert man['iterations'] == n
    for v in a.var_names:
        assert _same_bits(np.concatenate([c.get_state(v) for c in group]), want[v]), ('group', v)
    for n_load in (1, 3):
        ctxs = _contexts(capi, H, W, n_load, None)
        pinned = []
        for rank, c in enumerate(ctxs):
            ck.check_compatible(man, c)
            pinned.append(ck.restore_context(c, path, bottom_up=rank % 2 == 1, man=man))
        _step(capi, ctxs, n)
        for v in a.var_names:
            assert _same_bits(np.concatenate([c.get_state(v) for c in ctxs]), want[v]), (n_load, v)
        for c, p in zip(ctxs, pinned):
            c.sync()
            ck.release(p)
            c.close()
    for c in group + [a]:
        c.close()


def test_a_large_restore_steps_behind_its_upload(capi, tmp_path):
    n = 10
    make = lambda: _model('fenton4v', 2048, 2048, hole=True, diff=1.5)
    path = str(tmp_path / 'ck')
    A, B = make(), make()
    for m in (A, B):
        m.define()
        m.add_pace_op('s2', 'luq', 1.0)
    seen = set()
    _drive(A, 2 * n, False, 3, seen)
    _drive(B, n, False, 3, seen)
    B.checkpoint(path).wait()
    B.close()
    C = make()
    C.restore(path)
    opened = [C._ctx.upload_state()]
    C.duration = n * C.dt_per_step * C.dt * (1 + 1e-9)
    for i in C.run(None, block=False):
        if i == 0:
            opened.append(C._ctx.upload_state())            # the first iteration is still behind the copies
    assert opened[0][0] and opened[0][1] and opened[0][2] == 1 and opened[0][3] >= 1, opened
    assert opened[1][0], opened
    for v in A._ctx.var_names:
        assert _same_bits(C._ctx.get_state(v), A._ctx.get_state(v)), v
    assert not C.__dict__.get('_restore_pinned')          # the host copies were released after run()
    for m in (A, C):
        m.close()


def test_checkpoint_entry_point_errors(capi):
    import ctypes as C
    m = _model('fenton4v', 41, 70, persist=False)
    m.define()
    ctx = m._ctx
    info = capi.CheckpointInfo()
    info.struct_size = 4
    L = capi.lib()
    assert L.fib_checkpoint_begin(ctx._h, C.byref(info)) == -1          # struct_size
    buf = np.zeros((3, 70), np.float32)
    with pytest.raises(capi.FibError, match='no checkpoint'):
        ctx.checkpoint_read(0, 0, buf)
    ctx.checkpoint_end()                                                  # a no-op without one
    got = ctx.checkpoint_begin()
    assert got['nparts'] == 4 and got['iterations'] == 0 and not got['act_armed'] and not got['fr_armed']
    with pytest.raises(capi.FibError, match='already in flight'):
        ctx.checkpoint_begin()
    with pytest.raises(capi.FibError, match='out of range'):
        ctx.checkpoint_read(4, 0, buf)
    with pytest.raises(capi.FibError, match='not inside'):
        ctx.checkpoint_read(0, 40, buf)
    ctx.checkpoint_read(3, 38, buf)
    assert _same_bits(buf, ctx.get_state('S')[38:41])
    ctx.checkpoint_end()
    with pytest.raises(capi.FibError, match='no activation map'):
        ctx.activation_set(capi.ACT_SAMPLE, np.zeros((41, 70), np.float32))
    ctx.activation_resume(0.5, 0.5, 12)
    assert np.isnan(ctx.activation_get(capi.ACT_SAMPLE)).all() and (ctx.activation_get(capi.ACT_COUNT) == 0).all()
    ctx.frames_resume('U', 0, 10, 1, 4, 7)
    assert len(ctx.frames_fetch(4)[0]) == 0                               # nothing is taken at arming
    ctx.step(capi.OP_ODE, 3)
    k, f = ctx.frames_fetch(4)
    assert list(k) == [10] and _same_bits(f[0], ctx.get_state('U'))
    info = ctx.checkpoint_begin()
    assert (info['iterations'], info['act_k'], info['fr_k'], info['nparts']) == (3, 15, 10, 10)
    ctx.checkpoint_end()
    m.close()


@pytest.mark.parametrize('ranks', [2])
def test_nccl_shards_save_and_restore_on_another_rank_count(cuda_device, ranks):
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
           '--master-addr', '127.0.0.1', '--master-port', str(port), os.path.join(root, 'tests', 'dist_checkpoint.py')]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=root)
    tail = '\n'.join((r.stdout + r.stderr).splitlines()[-30:])
    assert r.returncode == 0 and 'DIST CHECKPOINT OK' in r.stdout, tail
