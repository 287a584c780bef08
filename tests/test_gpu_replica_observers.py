"""GPU: per-replica observers (include/fib_b200.h, fib_replica_sums, fib_replica_count_below,
fib_replica_probe_watch / fib_replica_probe_fetch; IonicModel.masked_image_means, excitable_fractions, weighted_means,
replica_cl_observer).

The check throughout: what replica b of a batched context observes equals what its unbatched twin -- its own diff,
hole and S2 iteration, as in test_gpu_replicas.py -- observes with the scalar calls: probe records bit for bit
(including iterations with a fire_op(replica=b) or a pace(replica=b) beat), threshold counts exactly, sums within
1e-12 relative (double sums in a varying order).  Then egm.py's and court_ultra.py's protocols as ensembles, the
persistent kernel with B = 1, the capacity rule and overflow at 1024 x 128^2, and the refusals."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_replicas import B, BASE, FAMILIES, _make, _run, _same_bits

pytestmark = pytest.mark.gpu

PROW = 20


@pytest.fixture(scope='module')
def capi(cuda_device):
    from fib_tf_b200 import _capi
    return _capi


def _pace_at(b):
    return 13 + 2 * b


def _norm(m):
    """(sub, div) of image() for count_below."""
    from fib_tf_b200 import _capi
    return (0.0, 1.0) if m.MODEL_ID == _capi.FENTON4V else (float(m.min_v), float(m.max_v - m.min_v))


def _close(a, b, rtol=1e-12):
    return abs(a - b) <= rtol * max(abs(a), abs(b)) + 1e-300


@pytest.mark.parametrize('kind,H,W,extra,slow,kernel', FAMILIES,
                         ids=['%s-%dx%d-%s' % (f[0], f[1], f[2], '-'.join(sorted(f[3])) or 'plain') for f in FAMILIES])
def test_replica_observers_equal_the_twins(capi, kind, H, W, extra, slow, kernel):
    iters = 24
    bat = _make(kind, H, W, extra)
    singles = [_make(kind, H, W, extra, replica=b) for b in range(B)]
    pot = bat._pot_name
    assert bat._ctx.replica_probe_watch(pot, PROW, W // 2) == capi.PROBE_RING
    for b, s in enumerate(singles):
        s._ctx.probe_watch(pot, PROW, W // 2)
        bat.pace('s2', _pace_at(b), replica=b)
        s.pace('s2', _pace_at(b))
    kernels = _run(bat, iters, None, slow)
    assert any(kernel in k and k.endswith(',Z=%d' % B) for k in kernels), kernels
    for b, s in enumerate(singles):
        _run(s, iters, b, slow)
    rec = bat._ctx.replica_probe_fetch()
    assert rec.shape == (iters, B)
    for b, s in enumerate(singles):
        assert _same_bits(rec[:, b], s._ctx.probe_fetch()), b
    assert not _same_bits(rec[:, 0], rec[:, 1])
    # threshold counts, exactly
    sub, div = _norm(bat)
    below, total = bat._ctx.replica_count_below(pot, sub, div, 0.2, 1e-3)
    for b, s in enumerate(singles):
        assert (below[b], total[b]) == s._ctx.count_below(pot, sub, div, 0.2, 1e-3), b
    # phase-weighted and masked sums, against the twin and against float64 NumPy
    rng = np.random.default_rng(5)
    mask = rng.uniform(0, 1, (B, H, W)).astype(np.float32)
    slot = bat.add_probe_mask(mask)
    for b, s in enumerate(singles):
        assert s.add_probe_mask(mask[b]) == slot
    phase = bat.phase.astype(np.float64)
    for var in (pot, bat._ctx.var_names[1]):
        x = bat._ctx.get_state(var).reshape(B, H, W).astype(np.float64)
        pw, pn = bat._ctx.replica_sums(var)
        mw, mn = bat._ctx.replica_sums(var, slot)
        for b, s in enumerate(singles):
            sw, sn = s._ctx.weighted_sum(var)
            tw, tn = s._ctx.masked_sum(var, slot)
            assert _close(pw[b], sw) and _close(pn[b], sn), (var, b)
            assert _close(mw[b], tw) and _close(mn[b], tn), (var, b)
            assert _close(pw[b], np.sum(phase[b] * x[b])) and _close(pn[b], np.sum(phase[b])), (var, b)
            assert _close(mw[b], np.sum(mask[b] * x[b])) and _close(mn[b], np.sum(mask[b].astype(np.float64))), b
    for m in [bat] + singles:
        m.close()


def test_egm_protocol_as_an_ensemble(capi):
    """egm.py's loop (BR, a hole, S2, two Gaussian masks sampled every millisecond) at 128^2 for 60 ms, three
    diffs in one context: each replica's masked_image_means trace equals its twin's masked_image_mean trace."""
    from fib_tf_b200.br import BeelerReuter
    from fib_tf_b200.egm import create_mask
    diffs = [1.0, 0.7, 1.3]
    cfg = {'width': 128, 'height': 128, 'dt': 0.1, 'dt_per_plot': 10, 'duration': 60, 'skip': False,
           'cheby': True, 'timeline': False, 'timeline_name': 'x', 'save_graph': False}

    def drive(model, mean):
        model.add_hole_to_phase_field(40, 64, 12)
        model.define()
        model.add_pace_op('s2', 'luq', 10.0)
        s2 = model.millisecond_to_step(20)
        m1 = model.add_probe_mask(create_mask(model, 75 + 15, 64, 5))
        m2 = model.add_probe_mask(create_mask(model, 75 - 15, 64, 5))
        every = max(int(10 / model.dt_per_step), 1)
        trace = []
        for i in model.run(None, block=False):
            if i == s2:
                model.fire_op('s2')
            if i % every == 0:
                trace.append([mean(m1), mean(m2)])
        model.close()
        return np.asarray(trace)

    bat = BeelerReuter(dict(cfg, replicas=B, diff=diffs))
    got = drive(bat, bat.masked_image_means)                 # [samples, 2, B]
    assert got.shape[1:] == (2, B)
    for b, d in enumerate(diffs):
        m = BeelerReuter(dict(cfg, diff=d))
        want = drive(m, m.masked_image_mean)
        np.testing.assert_allclose(got[:, :, b], want, rtol=1e-12, atol=1e-15)
    assert got[:, 0, 0].min() < 0.2 * got[:, 0, 0].max()    # the wave crossed the masks
    assert not np.allclose(got[:, 0, 0], got[:, 0, 1])


def test_court_ultra_run_small_as_an_ensemble(capi):
    """court_ultra.py's run_small loop (holes incl. neg=True, 'slow' every 10th iteration, S2) at 128^2: the
    replica_cl_observer (i, cl) sequences equal the twins' cl_observer sequences, excitable_fractions equals
    excitable_fraction and weighted_means the twins' weighted_sum means."""
    from fib_tf_b200.court_ultra import Courtemanche
    diffs = [1.5, 1.0, 1.25]
    cfg = {'width': 128, 'height': 128, 'dt': 0.1, 'dt_per_plot': 10, 'duration': 250, 'skip': False,
           'cheby': True, 'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'ultra_slow': False}

    def drive(model, s2s, observe, rho):
        model.add_hole_to_phase_field(model.width // 2, model.height // 2, 10)
        model.add_hole_to_phase_field(model.width // 2, model.height // 2, model.width // 2 - 6, neg=True)
        model.define()
        model.add_pace_op('s2', 'luq', 10.0)
        observe(model)
        rhos = []
        for i in model.run(None, block=False):
            if i % 10 == 0:
                model.fire_op('slow')
            for b, s2 in enumerate(s2s):
                if i == s2:
                    model.fire_op('s2', **({'replica': b} if model.replicas > 1 else {}))
            if i % 500 == 0:
                rhos.append(rho(model))
        return rhos

    s2s = [1200 + 150 * b for b in range(B)]
    seen = {b: [] for b in range(B)}

    def watch_all(m):
        m.replica_cl_observer = lambda i, b, cl: seen[b].append((i, cl))

    bat = Courtemanche(dict(cfg, replicas=B, diff=diffs))
    rho_b = drive(bat, s2s, watch_all, lambda m: m.excitable_fractions(0.2, 1e-3))
    means = bat.weighted_means('_Na_i_')
    for b, d in enumerate(diffs):
        log = []
        one = Courtemanche(dict(cfg, diff=d))

        def watch_one(m):
            m.cl_observer = lambda i, cl: log.append((i, cl))
        rho_1 = drive(one, [s2s[b]], watch_one, lambda m: m.excitable_fraction(0.2, 1e-3))
        assert seen[b] == log, b
        assert [r[b] for r in rho_b] == rho_1, b
        swx, sw = one._ctx.weighted_sum('_Na_i_')
        assert _close(means[b], swx / sw), b
        one.close()
    assert all(seen[b] for b in range(B)), seen
    bat.close()


def test_one_replica_on_the_persistent_kernel(capi):
    """BASELINE config 1 (4v 512^2, headless, persistent kernel): replica_cl_observer with B = 1 reports the
    cl_observer sequence with the same number of launches."""
    from fib_tf_b200.fenton import Fenton4v
    cfg = {'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 300,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False}

    def drive(replica):
        m = Fenton4v(cfg)
        m.define()
        m.add_pace_op('top', 'top', 1.0)
        seen = []
        if replica:
            m.replica_cl_observer = lambda i, b, cl: seen.append((i, cl))
        else:
            m.cl_observer = lambda i, cl: seen.append((i, cl))
        n0 = m._ctx.launch_count()
        for i in m.run(None, block=False):
            if i in (10, 200):
                m.fire_op('top')
        kern = capi.last_kernel()
        launches = m._ctx.launch_count() - n0
        m.close()
        return seen, launches, kern

    one, l_one, k_one = drive(False)
    rep, l_rep, k_rep = drive(True)
    assert 'persist' in k_one and 'persist' in k_rep, (k_one, k_rep)
    assert rep == one and len(one) >= 2, (rep, one)
    assert l_rep == l_one


def test_capacity_records_and_overflow_at_1024_replicas(capi):
    H = W = 128
    nrep = 1024
    c = capi.Context(capi.FENTON4V, H, W, 0.1, 1.5, replicas=nrep)
    rng = np.random.default_rng(7)
    c.set_state('U', rng.uniform(0, 1, (nrep * H, W)).astype(np.float32))
    assert c.replica_probe_watch('U', PROW, 77) == 4096                   # min(4096, max(256, 2^22 / 1024))
    want = []
    for _ in range(4):
        c.step(capi.OP_ODE, 1)
        want.append(c.get_state('U').reshape(nrep, H, W)[:, PROW, 77])
    assert capi.last_kernel().endswith(',Z=%d' % nrep)
    got = c.replica_probe_fetch(3)
    assert got.shape == (3, nrep) and _same_bits(got, np.asarray(want[:3]))
    extra = 4096 + 5
    c.step(capi.OP_ODE, extra)
    got = c.replica_probe_fetch(8192)
    assert got.shape == (4096, nrep)                                      # the oldest 1 + 5 records were lost
    assert _same_bits(got[-1], c.get_state('U').reshape(nrep, H, W)[:, PROW, 77])
    assert len(c.replica_probe_fetch()) == 0
    c.close()
    # the rule's other branch: 2^22 / 16384 = 256 records
    small = capi.Context(capi.FENTON4V, 16, 16, 0.1, 1.5, replicas=16384)
    small.set_state('U', rng.uniform(0, 1, (16384 * 16, 16)).astype(np.float32))
    assert small.replica_probe_watch('U', 3, 5) == 256
    small.step(capi.OP_ODE, 300)
    got = small.replica_probe_fetch(1000)
    assert got.shape == (256, 16384)
    assert _same_bits(got[-1], small.get_state('U').reshape(16384, 16, 16)[:, 3, 5])
    small.close()


def test_refusals(capi):
    H, W = 36, 64
    L = capi.lib()
    c = capi.Context(capi.BR, H, W, 0.1, 1.0, replicas=B)
    buf = np.zeros(2 * (B + 1))
    u64 = np.zeros(2 * (B + 1), np.uint64)
    p, q = buf.ctypes.data_as(C.c_void_p), u64.ctypes.data_as(C.c_void_p)
    assert L.fib_replica_sums(c._h, 0, -1, p, p, B + 1) == -1                        # FIB_E_ARG
    assert L.fib_replica_count_below(c._h, 0, 0.0, 1.0, 0.2, 1e-3, q, q, B - 1) == -1
    assert L.fib_replica_sums(c._h, 0, 2, p, p, B) == -4                             # FIB_E_STATE: empty slot
    with pytest.raises(capi.FibError, match='empty'):
        c.replica_sums('V', 2)
    for row, col in ((H, 0), (0, W)):
        with pytest.raises(capi.FibError, match='not in this'):
            c.replica_probe_watch('V', row, col)
    c.replica_probe_watch('V', H - 1, W - 1)
    n = C.c_size_t()
    assert L.fib_probe_fetch(c._h, None, 0, C.byref(n)) == -4                        # the other kind
    c.probe_watch('V', 2 * H + 1, 0)                                                  # replaces the replica watch
    assert L.fib_replica_probe_fetch(c._h, None, 0, C.byref(n)) == -4
    c.probe_watch('V', -1, -1)
    assert L.fib_probe_fetch(c._h, None, 0, C.byref(n)) == -4
    # the whole-context sums stay refused on a batched context
    with pytest.raises(capi.FibError, match='replicas'):
        c.weighted_sum('V')
    c.close()
    # unbatched: n == 1, the whole grid
    one = capi.Context(capi.BR, H, W, 0.1, 1.0)
    assert L.fib_replica_sums(one._h, 0, -1, p, p, 2) == -1
    wx, w = one.replica_sums('V')
    assert wx.shape == (1,) and _close(wx[0], one.weighted_sum('V')[0]) and w[0] == H * W
    one.close()
    # Python: a distributed model has the scalar forms only
    from fib_tf_b200.fenton import Fenton4v
    m = Fenton4v(dict(BASE, width=W, height=H, diff=1.5))
    m.define()
    m._nranks = 2
    for call in (lambda: m.masked_image_means(0), m.excitable_fractions, lambda: m.weighted_means('U')):
        with pytest.raises(ValueError, match='unsharded'):
            call()
    m._nranks = 1
    m.close()
