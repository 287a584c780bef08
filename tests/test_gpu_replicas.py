"""GPU: replicas (include/fib_b200.h "Replicas", config['replicas']).

The check throughout: replica b of a batched context is bit-identical to an unbatched context given replica b's
inputs -- its own diff, its own hole (one touching the replica's top border, one its bottom border, so that a
REFLECT or clamp across a seam shows), its own S2 iteration -- on an odd height and on widths that are and are not
a multiple of 4.  Every kernel family, every plane, with fib_last_kernel proving that the batched launch (Z=B) ran.
Then the observers, pacing, checkpoint / restore, fib_set_rect_async, the CV-vs-diff table of test_cv_table.py as
one context of ten replicas, and the refusals."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

BASE = {'dt': 0.1, 'dt_per_plot': 10, 'duration': 1, 'timeline': False, 'timeline_name': 'x', 'save_graph': False,
        'skip': False, 'cheby': False, 'ultra_slow': False}
B = 3
DIFFS = {'fenton4v': [1.5, 0.9, 1.2], 'br': [0.809, 0.5, 1.1], 'court': [1.5, 1.0, 1.25],
         'court_ultra': [1.5, 1.0, 1.25]}


@pytest.fixture(scope='module')
def capi(cuda_device):
    from fib_tf_b200 import _capi
    return _capi


def _holes(H, W):
    """One hole per replica: touching the top border, touching the bottom border, inside."""
    r = max(min(H, W) // 6, 2)
    return [(W // 2, 0, r), (W // 3, H - 1, r), (2 * W // 3, H // 2, r)]


def _make(kind, H, W, extra, replica=None, diffs=None, holes=True):
    """The batched model (replica None) or the unbatched twin of replica `replica`."""
    from cuda_adapter import CLASSES
    diffs = diffs or DIFFS[kind]
    cfg = dict(BASE, width=W, height=H, **extra)
    if replica is None:
        cfg.update(replicas=len(diffs), diff=list(diffs))
    else:
        cfg.update(diff=diffs[replica])
    m = CLASSES[kind](cfg)
    if kind in ('court', 'court_ultra'):
        m.chronic = True
    if holes:
        for b, (x, y, r) in enumerate(_holes(H, W)[:len(diffs)]):
            if replica is None:
                m.add_hole_to_phase_field(x, y, r, replica=b)
            elif replica == b:
                m.add_hole_to_phase_field(x, y, r)
    m.define()
    m.add_pace_op('s2', 'luq', float(m.max_v))
    return m


def _same_bits(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def _s2_at(b):
    return 4 + 3 * b


def _run(m, iters, replica, slow=False):
    """`iters` iterations, S2 of replica b after iteration _s2_at(b) (a batched model: every replica's own)."""
    from fib_tf_b200 import _capi
    kernels = set()
    for i in range(iters):
        m._ctx.step(m.ode_op(i), 1)
        kernels.add(_capi.last_kernel())
        if slow and i % 10 == 0:
            m.fire_op('slow')
        if replica is None:
            for b in range(m.replicas):
                if i == _s2_at(b):
                    m.fire_op('s2', replica=b)
        elif i == _s2_at(replica):
            m.fire_op('s2')
    m._ctx.flush()
    return kernels


def _assert_replicas(bat, singles, H, W):
    for v in bat._ctx.var_names:
        planes = bat._ctx.get_state(v).reshape(len(singles), H, W)
        for b, s in enumerate(singles):
            assert _same_bits(planes[b], s._ctx.get_state(v)), (v, b)


FAMILIES = [
    # kind, H, W, config extras, slow op, kernel substring
    ('fenton4v', 37, 64, {'steps_per_launch': 1}, False, 'step_kernel<Fenton4v'),
    ('fenton4v', 37, 50, {'steps_per_launch': 1}, False, 'step_kernel<Fenton4v'),
    ('fenton4v', 37, 264, {'steps_per_launch': 2}, False, 'fenton_fused2_kernel<PHASE=1>'),
    ('br', 37, 50, {}, False, 'BeelerReuter<exact'),
    ('br', 37, 64, {'cheby': True}, False, 'BeelerReuter<cheby'),
    ('br', 37, 50, {'cheby': True, 'skip': True}, False, 'BeelerReuter<cheby'),
    ('br', 37, 64, {'skip': True}, False, 'BeelerReuter<exact'),
    ('br', 37, 50, {'cheby': True, 'cheby_strict': True}, False, 'BeelerReuter<strict'),
    ('court', 37, 50, {}, True, 'Courtemanche<fast'),
    ('court_ultra', 37, 64, {}, False, 'Courtemanche<all>'),
    ('court_ultra', 37, 50, {'lut': True}, False, 'Courtemanche<all,lut>'),
    ('court_ultra', 37, 64, {'ultra_slow': True}, False, 'Courtemanche<all,us>'),
]


@pytest.mark.parametrize('kind,H,W,extra,slow,kernel', FAMILIES,
                         ids=['%s-%dx%d-%s' % (f[0], f[1], f[2], '-'.join(sorted(f[3])) or 'plain') for f in FAMILIES])
def test_replica_equals_its_unbatched_twin(capi, kind, H, W, extra, slow, kernel):
    iters = 24
    bat = _make(kind, H, W, extra)
    singles = [_make(kind, H, W, extra, replica=b) for b in range(B)]
    kernels = _run(bat, iters, None, slow)
    assert any(kernel in k and k.endswith(',Z=%d' % B) for k in kernels), kernels
    if extra.get('steps_per_launch') == 2:
        assert bat.steps_per_launch_used == 2
    for b, s in enumerate(singles):
        _run(s, iters, b, slow)
    _assert_replicas(bat, singles, H, W)
    # the replicas really differ from each other
    u = bat._ctx.get_state(bat._pot_name).reshape(B, H, W)
    assert not _same_bits(u[0], u[1]) and not _same_bits(u[1], u[2])
    for m in [bat] + singles:
        m.close()


def test_batched_contexts_never_run_the_persistent_kernel(capi):
    bat = _make('fenton4v', 37, 64, {})
    kernels = _run(bat, 3, None)
    assert not any('persist' in k for k in kernels), kernels
    bat.close()


def test_observers_and_pacing(capi):
    """Activation maps and frames bit for bit against the twins; pace(replica=None) and pace(replica=b) against
    unbatched pacing; fib_count_nonfinite over the replicas."""
    from fib_tf_b200 import _capi
    H, W, stride, iters = 36, 64, 3, 40
    kind, extra = 'fenton4v', {'steps_per_launch': 1}
    bat = _make(kind, H, W, extra)
    singles = [_make(kind, H, W, extra, replica=b) for b in range(B)]
    for m in [bat] + singles:
        m.watch_activation()
        m.record_frames(every=4, stride=stride)
    bat.pace('s2', 6, every=9, count=3)
    bat.pace('s2', 11, replica=1)
    for b, s in enumerate(singles):
        s.pace('s2', 6, every=9, count=3)
        if b == 1:
            s.pace('s2', 11)
    for m in [bat] + singles:
        for i in range(iters):
            m._ctx.step(m.ode_op(i), 1)
            m.iterations += 1
        if m is bat:
            assert _capi.last_kernel().endswith(',Z=%d' % B), _capi.last_kernel()
    _assert_replicas(bat, singles, H, W)
    for which in (_capi.ACT_FIRST, _capi.ACT_LAST, _capi.ACT_PREV, _capi.ACT_REPOL, _capi.ACT_COUNT):
        got = bat._ctx.activation_get(which).reshape(B, H, W)
        for b, s in enumerate(singles):
            assert _same_bits(got[b], s._ctx.activation_get(which)), (which, b)
    maps = bat.activation_maps()
    assert maps['last'].shape == (B, H, W)
    it, cube = bat.frames()
    assert cube.shape == (iters // 4, B, H // stride, -(-W // stride))
    for b, s in enumerate(singles):
        it_s, cube_s = s.frames()
        assert np.array_equal(it, it_s) and _same_bits(cube[:, b], cube_s), b
    assert bat.nonfinite_cells() == {}
    u = bat.pot().eval()
    u[1, 5, 7] = np.nan
    bat.pot().assign(u)
    assert bat.nonfinite_cells() == {'U': 1}
    for m in [bat] + singles:
        m.close()


def test_checkpoint_restore_continues_bit_for_bit(capi, tmp_path):
    kind, H, W, extra = 'br', 37, 64, {'cheby': True}
    full = _make(kind, H, W, extra)
    part = _make(kind, H, W, extra)
    _run(full, 30, None)
    _run(part, 15, None)
    part.iterations = 15
    part.checkpoint(str(tmp_path / 'ck')).wait()
    part.close()
    from cuda_adapter import CLASSES
    cfg = dict(BASE, width=W, height=H, replicas=B, diff=DIFFS[kind], **extra)

    def fresh(**over):
        m = CLASSES[kind](dict(cfg, **over))
        for b, (x, y, r) in enumerate(_holes(H, W)):
            m.add_hole_to_phase_field(x, y, r, replica=b)
        return m

    m = fresh()
    m.restore(str(tmp_path / 'ck'))
    m.add_pace_op('s2', 'luq', float(m.max_v))
    for i in range(15, 30):
        m._ctx.step(m.ode_op(i), 1)
        for b in range(B):
            if i == _s2_at(b):
                m.fire_op('s2', replica=b)
    for v in m._ctx.var_names:
        assert _same_bits(m._ctx.get_state(v), full._ctx.get_state(v)), v
    m.close()
    full.close()
    with pytest.raises(ValueError, match='replicas'):
        other = CLASSES[kind](dict(cfg, replicas=B + 1, diff=DIFFS[kind] + [1.0]))
        other.restore(str(tmp_path / 'ck'))
    with pytest.raises(ValueError, match='diff'):
        fresh(diff=[0.809, 0.5, 1.0]).restore(str(tmp_path / 'ck'))


def test_set_rect_async_equals_set_state(capi):
    from fib_tf_b200 import _capi
    H, W = 37, 64
    a = _capi.Context(_capi.FENTON4V, H, W, 0.1, 1.5, replicas=B)
    ref = _capi.Context(_capi.FENTON4V, H, W, 0.1, 1.5, replicas=B)
    rng = np.random.default_rng(3)
    pinned = []
    planes = {v: rng.uniform(0, 1, (B * H, W)).astype(np.float32) for v in a.var_names}
    for s in range(0, B * H, 16):
        for v in a.var_names:
            blk = _capi.pinned_empty((min(16, B * H - s), W))
            blk[...] = planes[v][s:s + 16]
            pinned.append(blk)
            a.set_rect_async(v, s, 0, blk)
    for v in a.var_names:
        ref.set_state(v, planes[v])
    assert a.upload_state()[0] == 0          # never an upload session
    a.step(_capi.OP_ODE, 3)
    ref.step(_capi.OP_ODE, 3)
    for v in a.var_names:
        assert _same_bits(a.get_state(v), ref.get_state(v)), v
    a.close()
    ref.close()
    for blk in pinned:
        _capi.pinned_free(blk)


def test_cv_table_as_one_context_of_ten_replicas(capi):
    """test_cv_table.py's 4v strips, one context per diff there, here one context of ten replicas: each
    replica's LAST activation map equals its own context's bit for bit."""
    import cv_common as cv
    from fib_tf_b200 import _capi
    from cuda_adapter import CLASSES
    diffs = sorted(cv.CV_TABLE_4V)
    width, iters = 700, 300
    bat = CLASSES['fenton4v'](dict(cv.strip_config(diffs[0], width), replicas=len(diffs), diff=diffs))
    bat.define()
    bat.watch_activation()
    bat._ctx.step(_capi.OP_ODE, iters)
    assert _capi.last_kernel().endswith(',Z=%d' % len(diffs)), _capi.last_kernel()
    last = bat._ctx.activation_get(_capi.ACT_LAST).reshape(len(diffs), 5, width)
    assert np.isfinite(last[:, 2, 20]).all()        # the front has passed column 20 of every strip
    for b, d in enumerate(diffs):
        m = CLASSES['fenton4v'](cv.strip_config(d, width))
        m.define()
        m.watch_activation()
        m._ctx.step(_capi.OP_ODE, iters)
        assert _same_bits(last[b], m._ctx.activation_get(_capi.ACT_LAST)), d
        m.close()
    bat.close()


def test_refusals(capi):
    from fib_tf_b200 import _capi
    H, W = 36, 64
    with pytest.raises(_capi.FibError, match='row shard'):
        _capi.Context(_capi.BR, H, W, 0.1, 1.0, row0=0, rows=10, replicas=2)
    with pytest.raises(_capi.FibError, match='replicas'):
        _capi.Context(_capi.BR, H, W, 0.1, 1.0, replicas=70000)
    c = _capi.Context(_capi.BR, H, W, 0.1, 1.0, replicas=B)
    with pytest.raises(_capi.FibError, match='replicas'):
        c.weighted_sum('V')
    c.set_weights(0, np.ones((B * H, W), np.float32))
    with pytest.raises(_capi.FibError, match='replicas'):
        c.masked_sum('V', 0)
    with pytest.raises(_capi.FibError, match='replicas'):
        c.count_below('V', 0.0, 1.0, 0.2, 1e-3)
    with pytest.raises(_capi.FibError, match='stride'):
        c.frames_watch('V', 1, 1, 5, 4)
    c.frames_watch('V', 1, 1, 4, 4)
    with pytest.raises(_capi.FibError, match='batched'):
        c.comm_init(2, 0, bytes(128))
    with pytest.raises(_capi.FibError, match='batched'):
        _capi.step_group([c])
    with pytest.raises(_capi.FibError):
        c.set_replica_diff([1.0, 2.0])
    with pytest.raises(_capi.FibError):
        c.stimulate('V', 0, 1, 0, 1, 1.0, 0.0, replica=B)
    one = _capi.Context(_capi.BR, H, W, 0.1, 1.0)
    with pytest.raises(_capi.FibError):
        one.set_replica_diff([1.0])
    c.close()
    one.close()
