"""CPU: the host side of the per-replica observers (include/fib_b200.h, fib_replica_sums, fib_replica_count_below,
fib_replica_probe_watch) against a fake batched context that computes the sums in NumPy from its state: run() with a
replica_cl_observer drains one batch behind and finds the crossings of every replica on their own, masks broadcast
over the replicas, and masked_image_means / excitable_fractions / weighted_means normalise exactly as image() does."""
import numpy as np
import pytest

from fib_tf_b200 import _capi
from fib_tf_b200.br import BeelerReuter
from fib_tf_b200.fenton import Fenton4v
from test_replicas_cpu import ReplicaContext

B, H, W = 3, 24, 12


class ObservedContext(ReplicaContext):
    """ReplicaContext plus the replica observers; the probe records come from `script` (one [B] row per
    iteration) when set, else from the state."""
    script = None

    def __init__(self, *a, **kw):
        super().__init__(*a, **kw)
        self.weights, self.watch, self.ring = {}, None, []

    def set_phase(self, rows, first_row=0):
        self.phase = np.array(rows, dtype=np.float32)

    def set_weights(self, slot, rows, first_row=0):
        a = np.asarray(rows, dtype=np.float32)
        assert a.shape == (self.rows, self.width) and first_row == 0
        self.weights[slot] = a.copy()

    def step(self, op=0, n_iter=1):
        super().step(op, n_iter)
        for _ in range(n_iter if self.watch and op == 0 else 0):
            var, row, col = self.watch
            rec = (self.script.pop(0) if self.script else
                   self.state[var].reshape(self.replicas, self.height, self.width)[:, row, col])
            self.ring.append(np.asarray(rec, dtype=np.float32))

    def replica_probe_watch(self, var, row, col):
        self.calls.append(('replica_watch', var, row, col))
        self.watch, self.ring = ((var, row, col) if row >= 0 else None), []
        return 4096

    def replica_probe_fetch(self, max_records=None):
        self.calls.append(('replica_fetch', max_records))
        recs = self.ring[:max_records]
        del self.ring[:len(recs)]
        return np.asarray(recs, dtype=np.float32).reshape(len(recs), self.replicas)

    def _per_replica(self, a):
        return np.asarray(a, dtype=np.float64).reshape(self.replicas, -1)

    def replica_sums(self, var, slot=-1):
        w = self.phase if slot < 0 else self.weights[slot]
        w = np.ones((self.rows, self.width)) if w is None else w
        x, w = self._per_replica(self.state[var]), self._per_replica(w)
        return (w * x).sum(axis=1), w.sum(axis=1)

    def replica_count_below(self, var, sub, div, cutoff, w_min):
        w = self.phase if self.phase is not None else np.ones((self.rows, self.width), np.float32)
        img = (self.state[var] - np.float32(sub)) / np.float32(div)
        keep = w.reshape(self.replicas, -1) > np.float32(w_min)
        below = keep & (img.reshape(self.replicas, -1) < np.float32(cutoff))
        return below.sum(axis=1), keep.sum(axis=1)


@pytest.fixture
def fake(monkeypatch):
    ObservedContext.made, ObservedContext.script = [], None
    monkeypatch.setattr(_capi, 'Context', ObservedContext)
    return ObservedContext


def cfg(**kw):
    c = {'width': W, 'height': H, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 40, 'timeline': False,
         'timeline_name': 'unused', 'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False,
         'replicas': B, 'probe_batch': 8}
    c.update(kw)
    return c


def _crossings(trace, weight=1.0):
    """The reference's crossing rule on one replica's raw 4v trace: (i, cl) of each upward pass through 0.5."""
    out, v0, last = [], 0.0, 0
    for i, v in enumerate(trace):
        v1 = float(v) * weight
        if v1 >= 0.5 and v0 < 0.5:
            out.append((i, (i - last) * 1.0))
            last = i
        v0 = v1
    return out


def test_run_drains_one_batch_behind_and_crosses_per_replica(fake):
    m = Fenton4v(cfg())
    m.add_hole_to_phase_field(W // 2, 20, 3, replica=2)      # replica 2's probe cell is inside its hole
    m.define()
    n = m.millisecond_to_step(m.duration)
    rng = np.random.default_rng(1)
    traces = rng.uniform(0, 1, (n, B)).astype(np.float32)
    fake.script = [t for t in traces]
    seen, fetched_at = [], []
    m.replica_cl_observer = lambda i, b, cl: seen.append((i, b, cl))
    for i in m.run():
        fetched_at.append(sum(c[0] == 'replica_fetch' for c in m._ctx.calls))
    ctx = m._ctx
    assert ctx.calls[0] == ('replica_watch', 'U', 20, W // 2) and ctx.calls[-1] == ('replica_watch', 'U', -1, -1)
    fetches = [c for c in ctx.calls if c[0] == 'replica_fetch']
    # first fetch once two batches are unread, then one batch at a time, the rest at the end
    assert fetched_at.index(1) == 2 * 8 and all(f[1] == 8 for f in fetches[:-1])
    assert sum(f[1] for f in fetches) == n
    weight = m.phase[2, 20, W // 2]
    assert weight < 0.5
    expected = sorted([(i, b, cl) for b in range(B) for i, cl in _crossings(traces[:, b], weight if b == 2 else 1.0)])
    assert seen == expected                    # in order of i, then replica
    assert any(b == 0 for _, b, _ in seen) and any(b == 1 for _, b, _ in seen) and not any(b == 2 for _, b, _ in seen)


def test_run_refusals(fake):
    m = Fenton4v(cfg())
    m.define()
    m.replica_cl_observer = lambda i, b, cl: None
    m.cl_observer = lambda i, cl: None
    with pytest.raises(ValueError):
        next(m.run())
    one = Fenton4v(cfg(replicas=1))
    one.define()
    one.replica_cl_observer = lambda i, b, cl: None
    one.cl_observer = lambda i, cl: None
    with pytest.raises(ValueError, match='replica_cl_observer'):
        next(one.run())
    one.cl_observer = None
    with pytest.raises(ValueError, match='replica_cl_observer'):
        next(one.run(im=object()))
    one._nranks = 2                     # as a sharded model sees itself
    for call in (lambda: one.masked_image_means(0), one.excitable_fractions, lambda: one.weighted_means('U')):
        with pytest.raises(ValueError, match='unsharded'):
            call()


def test_masks_broadcast_over_replicas(fake):
    m = BeelerReuter(cfg())
    m.define()
    rng = np.random.default_rng(2)
    one = rng.uniform(0, 1, (H, W)).astype(np.float32)
    each = rng.uniform(0, 1, (B, H, W)).astype(np.float32)
    assert m.add_probe_mask(one) == 0 and m.add_probe_mask(each) == 1
    assert np.array_equal(m._ctx.weights[0], np.tile(one, (B, 1)))
    assert np.array_equal(m._ctx.weights[1], each.reshape(B * H, W))
    with pytest.raises(ValueError):
        m.add_probe_mask(np.ones((B + 1, H, W), np.float32))
    u = Fenton4v(cfg(replicas=1))
    u.define()
    assert u.add_probe_mask(one) == 0 and np.array_equal(u._ctx.weights[0], one)


@pytest.mark.parametrize('cls', [Fenton4v, BeelerReuter])
def test_normalisations_equal_the_image_expressions(fake, cls):
    m = cls(cfg())
    m.add_hole_to_phase_field(W // 2, H // 2, 4, replica=1)
    m.define()
    rng = np.random.default_rng(3)
    lo, hi = float(m.min_v), float(m.max_v)
    for name in m._ctx.var_names:
        m._ctx.state[name] = rng.uniform(lo, hi, (B * H, W)).astype(np.float32)
    mask = rng.uniform(0, 1, (B, H, W)).astype(np.float32)
    slot = m.add_probe_mask(mask)
    # image()'s expression in float64 (image() itself rounds it to float32)
    v = m._ctx.state[m._pot_name].reshape(B, H, W).astype(np.float64)
    img = v if cls is Fenton4v else (v - m.min_v) / (m.max_v - m.min_v)
    np.testing.assert_allclose(img, m.image(), rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(m.masked_image_means(slot), [np.mean(img[b] * mask[b]) for b in range(B)],
                               rtol=1e-12, atol=1e-15)
    phase = m.phase
    rho = [np.sum(m.image()[b][phase[b] > 1e-3] < 0.2) / np.sum(phase[b] > 1e-3) for b in range(B)]
    assert np.array_equal(m.excitable_fractions(0.2, 1e-3), rho)
    name = m._ctx.var_names[1]
    means = [np.average(m._ctx.state[name].reshape(B, H, W)[b].astype(np.float64), weights=phase[b]) for b in range(B)]
    np.testing.assert_allclose(m.weighted_means(name), means, rtol=1e-12)
    assert m.masked_image_means(slot).dtype == np.float64 and m.excitable_fractions().shape == (B,)
