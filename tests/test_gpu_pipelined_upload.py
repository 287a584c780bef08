"""GPU: the pipelined upload (fib_set_rect_async of full-width row blocks, top to bottom, every plane, then
fib_step before anything looks at the state).  The copies run on their own stream and the deferred
iterations run block by block behind them with a skewed row schedule (csrc/fib_capi.cu
finish_upload_session); the state and the probe ring must be those of upload-everything-then-step, bit for
bit, for every kernel family (one step per launch, two steps per launch, multi-rate, in-place planes)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def cuda(cuda_device):
    import cuda_adapter
    return cuda_adapter


def _init(names, H, W, seed):
    rng = np.random.default_rng(seed)
    out = {}
    if '_m_' in names:                       # Courtemanche: the resting state, V and the gates perturbed
        from fib_tf_b200.court import INITIAL_STATE
        rest = dict(INITIAL_STATE)
        for v in names:
            base = np.full((H, W), rest.get(v, 0.0), np.float32)
            if v == 'V':
                base = rng.uniform(-85.0, 10.0, (H, W)).astype(np.float32)
            elif v.startswith('_') and not v.startswith('_Ca') and 0.0 <= rest.get(v, 0.0) <= 1.0:
                base = np.clip(base + rng.uniform(-0.1, 0.1, (H, W)), 1e-4, 0.9999).astype(np.float32)
            out[v] = base
        return out
    for v in names:
        if v == 'V' and 'C' in names:
            out[v] = rng.uniform(-85.0, 20.0, (H, W)).astype(np.float32)
        elif v == 'C':
            out[v] = rng.uniform(5e-5, 5e-3, (H, W)).astype(np.float32)
        else:
            out[v] = rng.uniform(1e-3, 0.998, (H, W)).astype(np.float32)
    return out


CASES = [
    ('4v two steps per launch', 'FENTON4V', 0, {'steps_per_launch': 2}, 6),
    ('4v one step per launch', 'FENTON4V', 0, {'steps_per_launch': 1}, 5),
    ('br cheby+skip', 'BR', 'F_CHEBY|F_SKIP', {}, 5),
    ('br exact', 'BR', 0, {}, 4),
    ('courtemanche multi-rate', 'COURT', 0, {}, 12),
    ('courtemanche all-state', 'COURT_ULTRA', 'F_ULTRA_SLOW', {}, 12),
    ('courtemanche all-state lut', 'COURT_ULTRA', 'F_LUT|F_ULTRA_SLOW', {}, 12),
]


@pytest.mark.parametrize('label,model,flags,kw,iters', CASES, ids=[c[0] for c in CASES])
def test_stepping_behind_the_upload_is_bit_identical(cuda, monkeypatch, label, model, flags, kw, iters):
    from fib_tf_b200 import _capi
    from fib_tf_b200.br import BeelerReuter
    monkeypatch.setenv('FIB_PIPELINE_MIN_CELLS', '0')        # read by fib_create
    monkeypatch.setenv('FIB_PIPELINE_BLOCK_ROWS', '100')
    H, W, block = 610, 192, 150                              # five blocks, the last one short
    fl = 0
    for f in (flags.split('|') if flags else []):
        fl |= getattr(_capi, f)
    mk = lambda extra=0: _capi.Context(getattr(_capi, model), H, W, 0.02 if 'COURT' in model else 0.1, 1.0,
                                       flags=fl | extra, **kw)
    pipe, ref = mk(_capi.F_NO_PERSIST), mk(_capi.F_NO_PERSIST)
    init = _init(ref.var_names, H, W, 5)
    yy, xx = np.mgrid[0:H, 0:W]
    phase = np.maximum(0.5 * (np.tanh(np.hypot(yy - 300.0, xx - 90.0) - 40.0) + 1.0), 1e-5).astype(np.float32)
    if fl & _capi.F_CHEBY:
        cfg = {'width': W, 'height': H, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.0, 'duration': 1, 'cheby': True,
               'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False}
        table = BeelerReuter(cfg).chebyshev_table()
    for c in (pipe, ref):
        c.set_phase(phase, 0)
        if fl & _capi.F_CHEBY:
            c.set_table(_capi.TABLE_BR_CHEBY, table)
        if fl & _capi.F_LUT:
            c.build_lut()
        for v in c.var_names:                                # something else in the buffers first
            c.set_state(v, np.full((H, W), 0.5, np.float32))
        c.step(0, 1)
    pinned = {}
    for v, a in init.items():
        pinned[v] = _capi.pinned_empty((H, W))
        pinned[v][...] = a
    n0 = pipe.launch_count()
    for r0 in range(0, H, block):                            # block-major: every plane of a block, then the next
        for v in pipe.var_names:
            pipe.set_rect_async(v, r0, 0, pinned[v][r0:min(r0 + block, H)])
    for v in ref.var_names:
        ref.set_state(v, init[v])
    watch = ref.var_names[0]
    for c in (pipe, ref):
        c.probe_watch(watch, 149, 77)                        # a row that changes block as the frontier recedes
    for it in range(iters):
        pipe.step(0, 1)
        ref.step(0, 1)
    got, want = pipe.probe_fetch(), ref.probe_fetch()
    assert got.size == iters and np.array_equal(got, want)
    # it really ran behind the copies: five blocks x the iteration's launches each (+ one record per iteration)
    n_pipe = pipe.launch_count() - n0
    steps_per_launch = kw.get('steps_per_launch', 1)
    launches = iters * pipe.dt_per_step // steps_per_launch
    assert n_pipe == 5 * launches + iters, (n_pipe, launches)
    for v in ref.var_names:
        a, b = pipe.get_state(v), ref.get_state(v)
        assert np.array_equal(a, b, equal_nan=True), (label, v, float(np.nanmax(np.abs(a - b))))
    # afterwards the context steps as usual
    pipe.step(0, 2)
    ref.step(0, 2)
    for v in ref.var_names:
        assert np.array_equal(pipe.get_state(v), ref.get_state(v), equal_nan=True), (label, v)
    pipe.close()
    ref.close()


def test_upload_sessions_fall_back_when_they_cannot_be_pipelined(cuda, monkeypatch):
    """Out-of-order blocks, partial widths, a read between upload and step, too many deferred iterations for
    the first block: same results through the ordinary path."""
    from fib_tf_b200 import _capi
    monkeypatch.setenv('FIB_PIPELINE_MIN_CELLS', '0')
    monkeypatch.setenv('FIB_PIPELINE_BLOCK_ROWS', '100')
    H, W = 300, 128
    init = _init(('U', 'V', 'W', 'S'), H, W, 9)
    pinned = {v: _capi.pinned_empty((H, W)) for v in init}
    for v in init:
        pinned[v][...] = init[v]
    ref = _capi.Context(_capi.FENTON4V, H, W, 0.1, 1.5, flags=_capi.F_NO_PERSIST)
    for v in init:
        ref.set_state(v, init[v])
    ref.step(0, 30)
    want = {v: ref.get_state(v) for v in init}
    ref.close()

    def run(upload, iters_first, flags=_capi.F_NO_PERSIST):
        c = _capi.Context(_capi.FENTON4V, H, W, 0.1, 1.5, flags=flags)
        upload(c)
        c.step(0, iters_first)
        c.step(0, 30 - iters_first)
        out = {v: c.get_state(v) for v in init}
        c.close()
        return out

    def bottom_up(c):
        for r0 in (200, 100, 0):
            for v in init:
                c.set_rect_async(v, r0, 0, pinned[v][r0:r0 + 100])

    def with_a_read(c):
        for r0 in (0, 100, 200):
            for v in init:
                c.set_rect_async(v, r0, 0, pinned[v][r0:r0 + 100])
        assert c.probe('U', 250, 3) == init['U'][250, 3]

    def plane_major(c):                                      # still a valid session: blocks complete late
        for v in init:
            for r0 in (0, 100, 200):
                c.set_rect_async(v, r0, 0, pinned[v][r0:r0 + 100])

    # (the last one: small enough for the persistent on-chip kernel, which takes over after the copies)
    for upload, first, flags in ((bottom_up, 3, _capi.F_NO_PERSIST), (with_a_read, 3, _capi.F_NO_PERSIST),
                                 (plane_major, 3, _capi.F_NO_PERSIST), (plane_major, 29, _capi.F_NO_PERSIST),
                                 (plane_major, 3, 0)):
        got = run(upload, first, flags)
        for v in init:
            assert np.array_equal(got[v], want[v]), (upload.__name__, first, flags, v)
