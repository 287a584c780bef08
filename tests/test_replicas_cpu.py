"""CPU: the host side of replicas (include/fib_b200.h "Replicas", config['replicas']) against a fake context that
records the calls: config validation, the tall-grid reshaping of reads and writes, the replica= arguments of the
stimuli, pacing and holes, and the checkpoint manifest's replicas / per-replica diff."""
import json
import os

import numpy as np
import pytest

from fib_tf_b200 import _capi
from fib_tf_b200 import checkpoint as ck
from fib_tf_b200.br import BeelerReuter
from fib_tf_b200.court import Courtemanche
from fib_tf_b200.fenton import Fenton4v

B, H, W = 3, 7, 12


class ReplicaContext:
    """A batched context the way the library addresses it: one grid of replicas * height rows."""
    NAMES = {_capi.FENTON4V: ['U', 'V', 'W', 'S'], _capi.BR: ['V', 'C', 'M', 'H', 'J', 'D', 'F', 'XI'],
             _capi.COURT: ['V', '_Na_i_', '_m_', '_h_', '_j_', '_K_i_', '_oa_', '_oi_', '_ua_', '_ui_', '_xr_', '_xs_',
                           '_Ca_i_', '_d_', '_f_', '_f_Ca_', '_Ca_rel_', '_u_', '_v_', '_w_', '_Ca_up_']}
    STEPS = {_capi.FENTON4V: 10, _capi.BR: 5, _capi.COURT: 1}
    made = []

    def __init__(self, model, height, width, dt, diff, flags=0, device=0, row0=0, rows=0, steps_per_launch=0,
                 replicas=1):
        self.model, self.height, self.width, self.dt, self.diff, self.flags = model, height, width, dt, diff, flags
        self.replicas = replicas
        self.replica_diff = [diff] * replicas
        self.row0, self.rows = 0, height * replicas
        self.steps_per_launch = steps_per_launch
        self.var_names = list(self.NAMES[model])
        self.nvars, self.dt_per_step = len(self.var_names), self.STEPS[model]
        self.state, self.calls, self.phase = {}, [], None
        ReplicaContext.made.append(self)

    def set_state(self, var, host):
        a = np.asarray(host, dtype=np.float32)
        assert a.shape == (self.rows, self.width)
        self.state[var] = a.copy()

    def get_state(self, var, out=None):
        return self.state[var].copy()

    def set_phase(self, rows, first_row=0):
        self.phase = (np.array(rows), first_row)

    def set_replica_diff(self, diff):
        self.replica_diff = [float(d) for d in diff]
        self.calls.append(('set_replica_diff', list(diff)))

    def set_table(self, table, data):
        pass

    def build_lut(self):
        pass

    def stimulate(self, *a, **kw):
        self.calls.append(('stimulate', a, kw))

    def pace_add(self, *a, **kw):
        self.calls.append(('pace_add', a, kw))
        return len([c for c in self.calls if c[0] == 'pace_add']) - 1

    def step(self, op=0, n_iter=1):
        self.calls.append(('step', op, n_iter))

    def activation_get(self, which):
        return np.full((self.rows, self.width), float(which), np.float32)

    def sync(self):
        pass

    def close(self):
        pass


@pytest.fixture
def fake(monkeypatch):
    ReplicaContext.made = []
    monkeypatch.setattr(_capi, 'Context', ReplicaContext)
    return ReplicaContext


def cfg(**kw):
    c = {'width': W, 'height': H, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 10, 'timeline': False,
         'timeline_name': 'unused', 'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False,
         'replicas': B}
    c.update(kw)
    return c


def test_config_validation():
    with pytest.raises(ValueError, match='replicas'):
        Fenton4v(cfg(replicas=0))
    with pytest.raises(ValueError, match='diff holds 2 values for 3 replicas'):
        Fenton4v(cfg(diff=[1.0, 2.0]))
    with pytest.raises(ValueError, match='distributed'):
        Fenton4v(cfg(distributed=True))
    assert Fenton4v(cfg(diff=[1.0, 2.0, 3.0])).replica_diff == [1.0, 2.0, 3.0]
    assert Fenton4v(cfg()).replica_diff == [1.5] * B
    one = Fenton4v(cfg(replicas=1))
    assert one.replicas == 1 and one._rows == H


def test_context_and_initial_state(fake):
    m = Fenton4v(cfg(diff=[1.0, 1.25, 1.5]))
    m.define()
    ctx = fake.made[-1]
    assert ctx.replicas == B and ctx.rows == B * H and ctx.diff == 1.0
    assert ('set_replica_diff', [1.0, 1.25, 1.5]) in ctx.calls
    # the S1 column covers every replica's rows
    assert np.all(ctx.state['U'][:, 1] == 1.0) and np.all(ctx.state['U'][:, 2] == 0.0)
    # equal coefficients: nothing to upload beyond fib_config.diff
    Fenton4v(cfg()).define()
    assert not [c for c in fake.made[-1].calls if c[0] == 'set_replica_diff']
    # unbatched models keep the old constructor call (no replicas keyword)
    Fenton4v(cfg(replicas=1)).define()
    assert fake.made[-1].replicas == 1


def test_reads_and_writes_gain_a_replica_axis(fake):
    m = BeelerReuter(cfg())
    m.define()
    ctx = fake.made[-1]
    tall = np.arange(B * H * W, dtype=np.float32).reshape(B * H, W)
    ctx.state['V'] = tall.copy()
    assert m.pot().eval().shape == (B, H, W)
    assert np.array_equal(m.pot().eval(), tall.reshape(B, H, W))
    assert m.image().shape == (B, H, W)
    per = np.stack([np.full((H, W), b, np.float32) for b in range(B)])
    m.pot().assign(per)
    assert np.array_equal(ctx.state['V'], per.reshape(B * H, W))
    m.pot().assign(np.full((H, W), 7.0, np.float32))            # one plane for every replica
    assert np.all(ctx.state['V'] == 7.0)
    with pytest.raises(ValueError):
        m.pot().assign(np.zeros((B + 1, H, W), np.float32))
    maps = m.activation_maps()
    assert maps['first'].shape == (B, H, W)


def test_court_define_state_broadcasts(fake):
    m = Courtemanche(cfg(lut=False))
    plane = {n: np.full((H, W), i, np.float32) for i, n in enumerate(ReplicaContext.NAMES[_capi.COURT])}
    m.define(state=plane)
    ctx = fake.made[-1]
    assert ctx.state['_m_'].shape == (B * H, W) and np.all(ctx.state['_m_'] == 2)
    batched = {n: np.stack([v + b for b in range(B)]) for n, v in plane.items()}
    m2 = Courtemanche(cfg(lut=False))
    m2.define(state=batched)
    assert np.array_equal(fake.made[-1].state['V'].reshape(B, H, W)[:, 0, 0], np.arange(B))


def test_holes_per_replica(fake):
    m = Fenton4v(cfg())
    m.add_hole_to_phase_field(6, 3, 2, replica=1)
    m.add_hole_to_phase_field(6, 0, 2)                        # every replica, touching the top border
    ph = m.phase
    assert ph.shape == (B, H, W)
    one = Fenton4v(cfg(replicas=1))
    one.add_hole_to_phase_field(6, 0, 2)
    both = Fenton4v(cfg(replicas=1))
    both.add_hole_to_phase_field(6, 3, 2)
    both.add_hole_to_phase_field(6, 0, 2)
    assert np.array_equal(ph[0], one.phase) and np.array_equal(ph[2], one.phase)
    assert np.array_equal(ph[1], both.phase)
    with pytest.raises(ValueError):
        m.add_hole_to_phase_field(1, 1, 1, replica=B)
    m.define()
    rows, first = fake.made[-1].phase
    assert first == 0 and np.array_equal(rows, ph.reshape(B * H, W))


def test_stimuli_and_pacing_take_a_replica(fake):
    m = Fenton4v(cfg())
    m.define()
    ctx = fake.made[-1]
    m.add_pace_op('s2', 'luq', 1.0)
    m.fire_op('s2')
    m.fire_op('s2', replica=2)
    stims = [c for c in ctx.calls if c[0] == 'stimulate']
    assert stims[0][2] == {} and stims[1][2] == {'replica': 2}
    assert stims[0][1][1:5] == (1, H // 2, 1, W // 2)          # replica-local rows
    with pytest.raises(ValueError):
        m.fire_op('s2', replica=B)
    m.pace('s2', 4, every=3, count=2, replica=1)
    m.pace('s2', 5)
    paces = [c for c in ctx.calls if c[0] == 'pace_add']
    assert paces[0][2] == {'replica': 1} and paces[1][2] == {}
    st = ck.pacing_state(m._pacing, 0)
    assert st[0]['replica'] == 1 and 'replica' not in st[1]
    fresh = ReplicaContext(_capi.FENTON4V, H, W, 0.1, 1.5, replicas=B)
    ck.resume_pacing(fresh, st, 0)
    assert [c[2] for c in fresh.calls if c[0] == 'pace_add'] == [{'replica': 1}, {}]


def test_refusals(fake):
    m = Fenton4v(cfg())
    m.define()
    with pytest.raises(ValueError, match='replicas'):
        m.masked_image_mean(0)
    with pytest.raises(ValueError, match='replicas'):
        m.excitable_fraction()
    with pytest.raises(ValueError, match='activation maps'):
        next(m.run(im=object()))
    m.cl_observer = lambda i, cl: None
    with pytest.raises(ValueError):
        next(m.run())


def test_manifest_records_replicas_and_diff(tmp_path):
    ctx = ReplicaContext(_capi.BR, H, W, 0.1, 1.5, replicas=B)
    ctx.replica_diff = [0.5, 1.0, 1.5]
    info = {'act_armed': False, 'fr_armed': False, 'iterations': 3}
    shard = {'rows': [0, B * H], 'files': {v: ck.shard_file(v, 0, B * H) for v in ctx.var_names}}
    man = ck.manifest(ctx, info, [shard])
    assert man['config']['replicas'] == B and man['config']['diff'] == [0.5, 1.0, 1.5]
    ck.write_manifest(str(tmp_path), man)
    back = ck.load_manifest(str(tmp_path))
    assert back['config'] == json.loads(json.dumps(man['config']))
    ck.check_compatible(back, ctx)
    other = ReplicaContext(_capi.BR, H, W, 0.1, 1.5, replicas=B)
    other.replica_diff = [0.5, 1.0, 1.25]
    with pytest.raises(ValueError, match='diff'):
        ck.check_compatible(back, other)
    with pytest.raises(ValueError, match='replicas'):
        ck.check_compatible(back, ReplicaContext(_capi.BR, H, W, 0.1, 1.5, replicas=B + 1))
    with pytest.raises(ValueError, match='replicas'):
        ck.check_compatible(back, ReplicaContext(_capi.BR, H, W, 0.1, 1.5))
    # an unbatched checkpoint keeps today's manifest, and refuses a batched model
    single = ck.manifest(ReplicaContext(_capi.BR, H, W, 0.1, 1.5), info, [dict(shard, rows=[0, H])])
    assert 'replicas' not in single['config'] and single['config']['diff'] == 1.5
    with pytest.raises(ValueError, match='replicas'):
        ck.check_compatible(single, ctx)
    # read_rows covers the tall grid
    for v in ctx.var_names:
        np.save(os.path.join(str(tmp_path), shard['files'][v]),
                np.arange(B * H * W, dtype=np.float32).reshape(B * H, W))
    rows = ck.read_rows(str(tmp_path), 'V', H, 2 * H, back)
    assert np.array_equal(rows, np.arange(B * H * W, dtype=np.float32).reshape(B * H, W)[H:2 * H])
