"""CPU: the host side of the frame recorder (include/fib_b200.h fib_frames_watch, IonicModel.record_frames /
frames / stop_frames) against a fake context that keeps the ring the way the library does, and the new entry
points' argument checks without a GPU."""
import ctypes as C

import numpy as np
import pytest

from fib_tf_b200 import _capi
from fib_tf_b200.br import BeelerReuter
from fib_tf_b200.court import Courtemanche
from fib_tf_b200.fenton import Fenton4v

PERSIST_BATCH = 64


class FrameRingContext:
    """Records the calls; keeps a ring of `capacity` frames of the potential as fib_capi.cu does: frame j at
    k = first + j * every in slot j % capacity, the oldest lost on overflow.  It also keeps the persistent path's
    deferred-iteration count, so that a fetch that has to launch deferred iterations (a cut batch) shows up."""
    NAMES = {_capi.FENTON4V: ['U', 'V', 'W', 'S'],
             _capi.BR: ['V', 'C', 'M', 'H', 'J', 'D', 'F', 'XI'],
             _capi.COURT: ['V', '_Na_i_', '_m_', '_h_', '_j_', '_K_i_', '_oa_', '_oi_', '_ua_', '_ui_',
                           '_xr_', '_xs_', '_Ca_i_', '_d_', '_f_', '_f_Ca_', '_Ca_rel_', '_u_', '_v_',
                           '_w_', '_Ca_up_']}
    STEPS = {_capi.FENTON4V: 10, _capi.BR: 5, _capi.COURT: 1}

    def __init__(self, model, height, width, dt, diff, flags=0, device=0, row0=0, rows=0, steps_per_launch=0):
        self.model, self.height, self.width = model, height, width
        self.rows, self.row0 = rows or height, row0
        self.var_names = list(self.NAMES[model])
        self.nvars, self.dt_per_step = len(self.var_names), self.STEPS[model]
        self.state, self.calls = {}, []
        self.k, self.pending, self.launched = 0, 0, 0       # iterations: stepped, deferred, launched
        self.fr = None

    def set_state(self, var, host):
        self.state[var] = np.array(host, dtype=np.float32)

    def get_state(self, var, out=None):
        return self.state[var].copy()

    def set_phase(self, rows, first_row=0):
        pass

    def set_table(self, table, data):
        pass

    def _plane(self, k):
        """A distinct plane per iteration: the potential of iteration k."""
        rng = np.random.default_rng(k)
        base = self.state[self.var_names[0]]
        return (base + rng.uniform(-1, 1, base.shape)).astype(np.float32)

    def _launch(self):
        """The deferred iterations become one launch: their frames enter the ring."""
        fr = self.fr
        for k in range(self.launched + 1, self.launched + self.pending + 1):
            if fr is not None and k >= fr['first'] and (k - fr['first']) % fr['every'] == 0:
                self._record(k)
        self.launched += self.pending
        self.pending = 0
        self.calls.append(('launch', self.launched))

    def _record(self, k):
        fr = self.fr
        j = (k - fr['first']) // fr['every']
        fr['ring'][j % fr['capacity']] = (k, self._plane(k)[::fr['stride'], ::fr['stride']])
        fr['total'] = j + 1

    def step(self, op=0, n_iter=1):
        self.calls.append(('step', op, n_iter))
        if op != _capi.OP_ODE:
            return
        for _ in range(n_iter):
            self.k += 1
            self.pending += 1
            if self.pending == PERSIST_BATCH:
                self._launch()

    def frames_watch(self, var, first, every, stride, capacity):
        self.calls.append(('frames_watch', var, first, every, stride, capacity))
        if self.pending:
            self._launch()
        self.launched = 0
        self.k = 0
        self.fr = {'first': first, 'every': every, 'stride': stride, 'capacity': capacity, 'ring': {},
                   'total': 0, 'fetched': 0}
        if first == 0:
            self._record(0)

    def frames_stop(self):
        self.calls.append(('frames_stop',))
        self.fr = None

    def frames_shape(self):
        s = self.fr['stride']
        return -(-self.rows // s), -(-self.width // s)

    def frames_fetch(self, max_frames):
        fr = self.fr
        if fr['total'] - fr['fetched'] < max_frames and self.pending:
            self._launch()                                     # the library flushes only in this case
        first = max(fr['fetched'], fr['total'] - fr['capacity'])
        take = min(fr['total'] - first, max_frames)
        got = [fr['ring'][j % fr['capacity']] for j in range(first, first + take)]
        fr['fetched'] = first + take
        self.calls.append(('fetch', max_frames, take, self.launched))
        rows, cols = self.frames_shape()
        return (np.array([g[0] for g in got], np.uint64),
                np.array([g[1] for g in got], np.float32).reshape(take, rows, cols))

    def stimulate(self, *a):
        pass

    def probe_watch(self, *a):
        pass

    def sync(self):
        self.calls.append(('sync',))

    def close(self):
        pass


@pytest.fixture
def fake(monkeypatch):
    monkeypatch.setattr(_capi, 'Context', FrameRingContext)
    return FrameRingContext


CFG = {'width': 40, 'height': 30, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'timeline': False,
       'timeline_name': 'unused.json', 'save_graph': False, 'skip': False, 'cheby': False}


def _fenton(iters):
    m = Fenton4v(dict(CFG, duration=iters * 1.0))          # 4v: one iteration = 10 * 0.1 ms
    m.define()
    return m


def test_run_drains_one_batch_behind_aligned_to_the_persistent_batches(fake):
    m = _fenton(300)
    m.record_frames(10)
    for _ in m.run(None):
        pass
    fetches = [c for c in m._ctx.calls if c[0] == 'fetch']
    # at k = 128, 192, 256: the frames of k <= 64, 128, 192 (k = 1, 11, ..) -- all in launched work
    assert [(c[1], c[3]) for c in fetches] == [(7, 128), (6, 192), (7, 256)]
    assert all(c[1] == c[2] for c in fetches)
    launches = [c for c in m._ctx.calls if c[0] == 'launch']
    assert [c[1] for c in launches] == [64, 128, 192, 256]    # no batch was cut by a fetch
    iters, cube = m.frames()
    assert list(iters) == list(range(1, 300, 10)) and cube.shape == (30, 30, 40)
    assert m._ctx.calls[-1][0] == 'fetch'                      # the rest: fetched (and launched) by frames()
    for k, frame in zip(iters, cube):
        assert np.array_equal(frame, m._ctx._plane(int(k)))


@pytest.mark.parametrize('every', [1, 10, 100])
@pytest.mark.parametrize('first', [0, 1, 37])
def test_the_default_capacity_never_loses_a_frame(fake, every, first):
    m = _fenton(1000)
    m.record_frames(every, first=first)
    assert m._frames['capacity'] == 2 * (-(-64 // every) + 1)
    for _ in m.run(None):
        pass
    iters, cube = m.frames()
    want = list(range(first, 1001, every))
    assert list(iters) == want, (every, first)
    assert cube.shape[0] == len(want)


def test_a_small_ring_loses_the_oldest_frames_and_shows_the_gap(fake):
    m = _fenton(300)
    m.record_frames(1, capacity=4)
    for _ in m.run(None):
        pass
    iters, _ = m.frames()
    assert list(iters[-4:]) == [297, 298, 299, 300]
    assert np.any(np.diff(iters.astype(np.int64)) > 1)


@pytest.mark.parametrize('cls', [BeelerReuter, Courtemanche, Fenton4v])
def test_frames_normalise_the_potential_exactly_like_image(fake, cls):
    m = cls(dict(CFG, duration=5.0))
    m.define()
    m.record_frames(1, first=0)
    got_k, got = m.frames()
    assert list(got_k) == [0]
    # image() of the same plane, through the model's own expression
    m._ctx.state[m._pot_name] = m._ctx._plane(0)
    want = m.image()
    assert got[0].dtype == want.dtype
    assert np.array_equal(got[0].view(np.uint32), np.asarray(want, np.float32).view(np.uint32))
    # another variable is returned raw
    m.record_frames(1, first=0, name=m._ctx.var_names[1], stride=3)
    _, raw = m.frames()
    assert raw.shape == (1, 10, 14) and np.array_equal(raw[0], m._ctx._plane(0)[::3, ::3])


def test_frames_argument_errors_and_stop(fake):
    m = _fenton(10)
    with pytest.raises(AssertionError):
        m.frames()
    for bad in (dict(every=0), dict(every=1, stride=0), dict(every=1, first=-1)):
        with pytest.raises(ValueError):
            m.record_frames(**bad)
    m.record_frames(3)
    m.stop_frames()
    assert ('frames_stop',) in m._ctx.calls
    with pytest.raises(AssertionError):
        m.frames()


def test_frame_entry_points_validate_without_a_gpu():
    L = _capi.lib()
    r, c = C.c_int(), C.c_int()
    n = C.c_size_t()
    it = (C.c_uint64 * 4)()
    buf = (C.c_float * 4)()
    assert L.fib_frames_watch(None, 0, 1, 10, 1, 8) == -1
    assert L.fib_frames_stop(None) == -1
    assert L.fib_frames_shape(None, C.byref(r), C.byref(c)) == -1
    assert L.fib_frames_fetch(None, buf, it, 4, C.byref(n)) == -1
    assert L.fib_frames_fetch(None, None, None, 0, None) == -1
    assert 'NULL' in L.fib_last_error().decode()
