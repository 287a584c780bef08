"""CPU: the host side of pacing (IonicModel.pace / stop_pacing, the checkpoint manifest's `pacing` records) against a
fake context that schedules and fires entries the way include/fib_b200.h fib_pace_add describes, and the new entry
points' argument checks without a GPU."""
import ctypes as C
import json
import os

import pytest

from fib_tf_b200 import _capi
from fib_tf_b200 import checkpoint as ck
from fib_tf_b200.fenton import Fenton4v
from test_checkpoint_cpu import CFG, CheckpointContext, fake  # noqa: F401  (fake: the fixture)

PCFG = dict(CFG, duration=20)          # 20 run() iterations (dt_per_step 10, dt 0.1)


class PacingContext(CheckpointContext):
    """CheckpointContext plus the pacing contract: an entry fires after the ODE iterations k = first + j * every
    counted from its pace_add, at most 4 entries, finished entries dropped.  `fired` lists (ctx iteration, rect)
    of every stimulus, by pacing and by stimulate() alike."""

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.paces, self.next_id, self.fired = {}, 0, []

    def pace_add(self, r0, r1, c0, c1, value, floor_v, first, every=0, count=1):
        if first < 1 or count < 0 or (count != 1 and every < 1):
            raise _capi.FibError('fib_pace_add: bad schedule')
        if len(self.paces) >= _capi.PACE_MAX:
            raise _capi.FibError('fib_pace_add: at most 4 pacing entries')
        pid, self.next_id = self.next_id, self.next_id + 1
        self.paces[pid] = {'rect': (r0, r1, c0, c1), 'at': self.iters + first, 'every': every if count != 1 else 1,
                           'count': count}
        self.calls.append(('pace_add', (r0, r1, c0, c1), value, floor_v, first, every, count))
        return pid

    def pace_remove(self, pace_id=-1):
        if pace_id >= self.next_id:
            raise _capi.FibError('fib_pace_remove: no such entry')
        for k in list(self.paces):
            if pace_id < 0 or k == pace_id:
                del self.paces[k]

    def step(self, op=0, n_iter=1):
        for _ in range(n_iter):
            super().step(op, 1)
            if op != _capi.OP_ODE:
                continue
            n = self.iters
            for pid, p in list(self.paces.items()):
                d = n - p['at']
                if d >= 0 and d % p['every'] == 0 and (p['count'] == 0 or d // p['every'] < p['count']):
                    self.fired.append((n, p['rect']))
                if p['count'] and n >= p['at'] + (p['count'] - 1) * p['every']:
                    del self.paces[pid]

    def stimulate(self, var, r0, r1, c0, c1, value, floor_v):
        self.fired.append((self.iters, (r0, r1, c0, c1)))


@pytest.fixture
def pacing(fake, monkeypatch):  # noqa: F811
    monkeypatch.setattr(_capi, 'Context', PacingContext)


def _model(cfg=PCFG):
    m = Fenton4v(dict(cfg))
    m.define()
    m.add_pace_op('s2', 'luq', 1.0)
    m.add_pace_op('s1', 'left', 1.0)
    return m


def _driver_fires(at, every, count, runs=1):
    """(iteration, rect) after which `for i in run(): if i == at + j * every: fire_op('s2')` fires."""
    m = _model()
    beats = {at + j * every for j in range(count)}
    for _ in range(runs):
        for i in m.run():
            if i in beats:
                m.fire_op('s2')
    return m._ctx.fired


@pytest.mark.parametrize('at,every,count', [(0, 0, 1), (4, 0, 1), (3, 5, 3), (2, 1, 6), (7, 4, 3)])
def test_pace_fires_after_the_iteration_fire_op_would(pacing, at, every, count):
    m = _model()
    m.pace('s2', at, every, count)
    assert m._ctx.calls[-1][4] == at + 1                 # first: k = at + 1 - iterations, iterations = 0
    for _ in m.run():
        pass
    assert m._ctx.fired == _driver_fires(at, every, count)
    assert len(m._ctx.fired) == count and not m._ctx.paces


def test_pace_counts_absolute_iterations_across_runs(pacing):
    m = _model()
    for _ in m.run():
        pass
    assert m.iterations == 20
    m.pace('s2', 24, 3, 4)                              # after iterations 25, 28, 31, 34
    assert m._ctx.calls[-1][4] == 5
    for _ in m.run():
        pass
    assert [n for n, _ in m._ctx.fired] == [25, 28, 31, 34]


def test_count_zero_paces_until_stopped(pacing):
    m = _model()
    m.pace('s2', 1, 4, 0)
    m.pace('s1', 0, 0, 1)
    for i in m.run():
        if i == 12:
            m.stop_pacing('s2')
    assert m._ctx.fired == [(1, (0, 37, 0, 5)), (2, (1, 18, 1, 12)), (6, (1, 18, 1, 12)), (10, (1, 18, 1, 12))]
    assert m._pacing == [] and not m._ctx.paces


def test_stop_pacing_removes_every_schedule(pacing):
    m = _model()
    m.pace('s2', 1, 2, 0)
    m.pace('s1', 3, 2, 0)
    m.stop_pacing()
    for _ in m.run():
        pass
    assert m._ctx.fired == [] and m._pacing == []


def test_pace_validation(pacing):
    m = _model()
    m._ops['slow'] = ('call', lambda: None)
    with pytest.raises(ValueError):
        m.pace('slow', 3)                                # not an add_pace_op op
    with pytest.raises(ValueError):
        m.pace('nope', 3)
    with pytest.raises(ValueError):
        m.pace('s2', 3, every=0, count=2)
    with pytest.raises(ValueError):
        m.pace('s2', 3, every=2, count=-1)
    for i in m.run():
        if i == 4:
            break
    assert m.iterations == 5
    with pytest.raises(ValueError):
        m.pace('s2', 4)                                  # iteration 5 has been stepped
    m.pace('s2', 5)                                      # iteration 6 has not
    with pytest.raises(AssertionError):
        Fenton4v(dict(PCFG)).pace('s2', 1)               # before define()


def test_finished_schedules_free_their_slots(pacing):
    m = _model()
    for j in range(4):
        m.pace('s2', j, 0, 1)
    with pytest.raises(_capi.FibError):
        m.pace('s1', 10, 1, 2)                           # a fifth entry
    for i in m.run():
        if i == 5:
            m.pace('s1', 10, 1, 2)                       # the four have fired: room again
            assert len(m._pacing) == 1
    assert [n for n, _ in m._ctx.fired] == [1, 2, 3, 4, 11, 12]


def test_pacing_state_records():
    e = {'name': 's1', 'rect': [0, 5, 0, 9], 'value': 1.0, 'floor': 0.0, 'next': 10, 'every': 4, 'count': 5, 'id': 2}
    # beats after 10, 14, 18, 22, 26
    assert ck.pacing_state([e], 9)[0] == {k: v for k, v in e.items() if k != 'id'}
    assert ck.pacing_state([e], 10)[0]['next'] == 14 and ck.pacing_state([e], 10)[0]['count'] == 4
    assert ck.pacing_state([e], 13)[0]['next'] == 14 and ck.pacing_state([e], 13)[0]['count'] == 4
    assert ck.pacing_state([e], 22)[0]['next'] == 26 and ck.pacing_state([e], 22)[0]['count'] == 1
    assert ck.pacing_state([e], 26) == []
    forever = dict(e, count=0)
    assert ck.pacing_state([forever], 1000)[0]['count'] == 0 and ck.pacing_state([forever], 1000)[0]['next'] == 1002
    once = dict(e, every=0, count=1)
    assert ck.pacing_state([once], 9)[0]['next'] == 10 and ck.pacing_state([once], 10) == []


@pytest.mark.parametrize('stop_at', [6, 9, 12])
def test_restore_continues_the_train(pacing, tmp_path, stop_at):
    """Checkpoint mid-train, restore into a new model: the beats follow the same absolute iterations, remaining
    beats included."""
    whole = _model()
    whole.pace('s2', 3, 3, 5)                            # after 4, 7, 10, 13, 16
    whole.pace('s1', 8, 0, 1)                            # after 9
    for _ in whole.run():
        pass
    want = whole._ctx.fired

    m = _model(dict(PCFG, duration=stop_at))
    m.pace('s2', 3, 3, 5)
    m.pace('s1', 8, 0, 1)
    for _ in m.run():
        pass
    m.checkpoint(str(tmp_path / 'ck')).wait()
    got = list(m._ctx.fired)
    man = ck.load_manifest(str(tmp_path / 'ck'))
    assert man['iterations'] == stop_at
    assert all(p['next'] > stop_at for p in man['pacing'])
    with open(os.path.join(str(tmp_path / 'ck'), ck.MANIFEST)) as f:
        assert json.load(f)['pacing'] == man['pacing']

    r = Fenton4v(dict(PCFG, duration=20 - stop_at))
    r.restore(str(tmp_path / 'ck'))
    r.add_pace_op('s2', 'luq', 1.0)
    r.add_pace_op('s1', 'left', 1.0)
    assert r.iterations == stop_at
    adds = [c for c in r._ctx.calls if c[0] == 'pace_add']
    assert len(adds) == len(man['pacing'])
    assert r._ctx.calls.index(adds[-1]) < min(r._ctx.calls.index(c) for c in r._ctx.calls if c[0] == 'rect')
    for _ in r.run():
        pass
    got += [(n + stop_at, rect) for n, rect in r._ctx.fired]
    assert got == want
    r.stop_pacing('s2')                                  # the restored schedules carry their entry ids
    assert not r._ctx.paces


def test_a_manifest_without_pacing_restores_as_before(pacing, tmp_path):
    m = _model()
    for i in m.run():
        if i == 4:
            break
    m.checkpoint(str(tmp_path / 'ck')).wait()
    fn = os.path.join(str(tmp_path / 'ck'), ck.MANIFEST)
    with open(fn) as f:
        man = json.load(f)
    assert man['pacing'] == []
    del man['pacing']
    ck.write_manifest(str(tmp_path / 'ck'), man)
    r = Fenton4v(dict(PCFG))
    r.restore(str(tmp_path / 'ck'))
    assert r._pacing == [] and not [c for c in r._ctx.calls if c[0] == 'pace_add']


def test_resume_pacing_refuses_a_beat_in_the_past():
    class Ctx:
        def pace_add(self, *a):
            raise AssertionError('not reached')
    with pytest.raises(ck.CheckpointError):
        ck.resume_pacing(Ctx(), [{'name': 's', 'rect': [0, 1, 0, 1], 'value': 1.0, 'floor': 0.0, 'next': 5,
                                   'every': 1, 'count': 0}], 5)


def test_pace_entry_points_reject_null_and_bad_arguments():
    L = _capi.lib()
    i = C.c_int()
    assert L.fib_pace_add(None, 0, 1, 0, 1, 1.0, 0.0, 1, 1, 1, C.byref(i)) == -1
    assert 'NULL' in L.fib_last_error().decode()
    assert L.fib_pace_remove(None, 0) == -1
    assert 'NULL' in L.fib_last_error().decode()
    assert 'fib_pace_add' in _capi.EXPORTS and 'fib_pace_remove' in _capi.EXPORTS
    assert _capi.ABI_VERSION == 6 == L.fib_version()

