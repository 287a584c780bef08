"""GPU: (1) the op-level entry points of IonicModel's stencil helpers (fib_op_*; ionic.py:44-123)
against the oracle -- BIT-identical for the boundary, the Laplacian and the phase-field sums, which
are written in the reference's association order without FMA contraction (fib_stencil.cuh);
(2) the device-side observers of SURVEY 8(f1): the cycle-length probe ring and the threshold count
behind the excitable fraction rho; (3) the enqueue-only strip upload."""
import numpy as np
import pytest

from oracle import monodomain_np as onp

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def cuda(cuda_device):
    import cuda_adapter
    return cuda_adapter


@pytest.mark.parametrize('H,W', [(3, 3), (5, 9), (64, 97), (300, 513)])
def test_stencil_ops_are_bit_identical_to_the_oracle(cuda, H, W):
    from fib_tf_b200 import _capi
    rng = np.random.default_rng(H * 131 + W)
    X = rng.uniform(-85.0, 25.0, (H, W)).astype(np.float32)
    ph = onp.hole_phase(None, H, W, W // 2, H // 2, max(min(H, W) // 4, 1))
    ph = onp.hole_phase(ph, H, W, 0, H - 1, max(min(H, W) // 6, 1))
    X0 = onp.enforce_boundary(X)
    assert np.array_equal(_capi.op_enforce_boundary(X), X0)
    # laplace(X0): REFLECT pad + 9-point stencil, with and without the phase term
    assert np.array_equal(_capi.op_laplace(X0), onp.laplace(X0))
    # the step kernels never materialise X0: their collapsed clamp map on the raw plane is the same thing
    assert np.array_equal(_capi.op_laplace(X, mode=1), onp.laplace(X0))
    # phase term: sums and products are exact replicas, the final division is the 2-ulp SFU one
    want = onp.laplace(X0, ph)
    got = _capi.op_laplace(X0, ph)
    term = onp.phase_term(np.pad(X0, 1, mode='reflect'), ph)
    assert np.all(np.abs(got.astype(np.float64) - want) <= 4 * np.spacing(np.abs(term)) + np.spacing(np.abs(want)))
    assert np.array_equal(_capi.op_laplace(X, ph, mode=1), got)
    assert np.all(np.abs(_capi.op_laplace(X0, ph, mode=2).astype(np.float64) - term) <= 4 * np.spacing(np.abs(term)))


def test_model_level_helpers_mirror_the_reference_methods(cuda):
    """IonicModel.enforce_boundary / laplace / phase_field / rush_larsen exist with the reference's
    signatures (ionic.py:44-123) and agree with the oracle."""
    from fib_tf_b200.br import BeelerReuter
    cfg = {'width': 90, 'height': 70, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False, 'cheby': False}
    m = BeelerReuter(cfg)
    m.add_hole_to_phase_field(40, 30, 9)
    rng = np.random.default_rng(3)
    X = rng.uniform(-85.0, 25.0, (70, 90)).astype(np.float32)
    X0 = m.enforce_boundary(X)
    assert np.array_equal(X0, onp.enforce_boundary(X))
    lap = m.laplace(X0)
    want = onp.laplace(X0, m.phase)
    term = onp.phase_term(np.pad(X0, 1, mode='reflect'), m.phase)
    # the sums and products are exact replicas; the term's final division is the 2-ulp SFU one
    assert np.all(np.abs(lap.astype(np.float64) - want) <= 4 * np.spacing(np.abs(term)) + np.spacing(np.abs(want)))
    pf = m.phase_field(np.pad(X0, 1, mode='reflect'))
    assert np.all(np.abs(pf.astype(np.float64) - term) <= 4 * np.spacing(np.abs(term)))
    g = rng.uniform(1e-3, 0.998, X.shape).astype(np.float32)
    gi = rng.uniform(0.0, 1.0, X.shape).astype(np.float32)
    tau = rng.uniform(0.05, 500.0, X.shape).astype(np.float32)
    # the edges of x = -dt/tau (rl_edge_inputs): tau < 0, tau -> 0+, +-0, +-inf, very large tau, |dt/tau|
    # straddling the 0.125 switch of the expm1 polynomial, g == g_inf with an infinite exponent (0 * inf
    # = NaN, which the clip turns into its upper bound)
    from test_gpu_math_layer import rl_edge_inputs
    n = g.size
    g, gi, tau = (np.concatenate([a.ravel(), b]) for a, b in zip((g, gi, tau), rl_edge_inputs()))
    with np.errstate(all='ignore'):
        want = onp.rush_larsen(g, gi, tau, 0.1)
        want64 = onp.rush_larsen(g.astype(np.float64), gi.astype(np.float64), tau.astype(np.float64), 0.1)
        e32 = np.expm1(np.float32(-0.1) / tau)
    got = m.rush_larsen(g, gi, tau, 0.1)
    assert onp.rel_err(got[:n], want64[:n], 1e-3) <= 2e-6
    # the edges: where e = expm1(-dt/tau) overflows fp32 (0 * inf = NaN for g == g_inf, which the clip
    # turns into its upper bound) the fp32 oracle is the reference; elsewhere float64, with the error of
    # m_expm1_neg (fib_math.cuh: < 13 ulp, < 8 + x ulp for x = -dt/tau > 1) carried by |g - g_inf|
    inf = ~np.isfinite(e32[n:])
    assert onp.rel_err(got[n:][inf], want[n:][inf], 1e-3) == 0.0
    x = -0.1 / tau[n:][~inf].astype(np.float64)
    bar = (2e-6 * np.maximum(np.abs(want64[n:][~inf]), 1e-3) + np.abs(g - gi)[n:][~inf].astype(np.float64) *
           np.where(x > 1, 8 + x, 13) * np.spacing(np.abs(e32[n:][~inf])))
    assert np.all(np.abs(got[n:][~inf] - want64[n:][~inf]) <= bar)
    from fib_tf_b200 import _capi
    strict = _capi.op_rush_larsen(g, gi, tau, 0.1, strict=True)
    assert np.all(np.abs(strict[:n].astype(np.float64) - want[:n]) <= 2 * np.spacing(np.abs(want[:n])))   # expm1f: 1 ulp
    # at the edges that ulp of e is carried by |g - g_inf|, which can exceed the result (cancellation)
    ulp_e = np.nan_to_num(np.spacing(np.abs(e32[n:])), nan=0.0)
    assert np.all(np.abs(strict[n:].astype(np.float64) - want[n:]) <=
                  2 * np.spacing(np.abs(want[n:])) + np.abs(g - gi)[n:].astype(np.float64) * ulp_e)
    m.close()


def test_device_probe_ring_reproduces_the_per_iteration_probe(cuda):
    """run(None) with a cl_observer: the probe cell is recorded on the device after every iteration
    (a node of the iteration graph) and fetched in batches.  The observer must be called with exactly
    the (iteration, cycle length) pairs of the reference's per-iteration host probe (probe_batch=1),
    including a stimulus that covers the probe cell between iterations; launches per iteration:
    the step kernels + ONE record kernel, and no per-iteration synchronisation."""
    from fib_tf_b200.fenton import Fenton4v

    def drive(**kw):
        cfg = {'width': 96, 'height': 64, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 420,
               'timeline': False, 'timeline_name': 'x', 'save_graph': False}
        cfg.update(kw)
        m = Fenton4v(cfg)
        m.add_hole_to_phase_field(70, 40, 6)
        m.define()
        m.add_pace_op('top', 'top', 1.0)
        seen = []
        m.cl_observer = lambda i, cl: seen.append((i, cl))
        n0 = m._ctx.launch_count()
        for i in m.run(None, block=False):
            if i == 330:
                m.fire_op('top')                # rows 0..4 only: a second wave towards the probe row 20
        launches = m._ctx.launch_count() - n0
        u = m._State['U'].eval()
        m.close()
        return seen, launches, u

    ring, l_ring, u_ring = drive()
    every, l_every, u_every = drive(probe_batch=1)
    assert ring == every and len(ring) >= 2, (ring, every)
    assert np.array_equal(u_ring, u_every)
    assert l_ring <= l_every          # batched read-back lets the persistent path batch its launches too
    # the raw ring API: values in order, wrap-around, loss of the oldest
    from fib_tf_b200 import _capi
    c = _capi.Context(_capi.FENTON4V, 8, 8, 0.1, 1.0)
    for v in c.var_names:
        c.set_state(v, np.full((8, 8), 0.25, np.float32))
    c.probe_watch('U', 3, 4)
    vals = []
    for k in range(5):
        c.step(0, 1)
        vals.append(c.probe('U', 3, 4))
    got = c.probe_fetch()
    assert np.array_equal(got, np.float32(vals))
    c.set_state('U', np.full((8, 8), 0.75, np.float32))     # a host write updates the LAST record
    c.step(0, 1)
    c.set_state('U', np.full((8, 8), 0.5, np.float32))
    assert np.array_equal(c.probe_fetch(), np.float32([0.5]))
    c.step(0, _capi.PROBE_RING + 10)
    got = c.probe_fetch()
    assert got.size == _capi.PROBE_RING and got[-1] == c.probe('U', 3, 4)
    c.close()


def test_excitable_fraction_is_the_host_formula(cuda):
    """rho = np.sum(image[phase > 1e-3] < 0.2) / np.sum(phase > 1e-3) (court_ultra.py:504-509) as one
    reduction on the device."""
    from fib_tf_b200.court_ultra import Courtemanche
    cfg = {'width': 120, 'height': 80, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'ultra_slow': False}
    for hole in (True, False):
        m = Courtemanche(cfg)
        if hole:
            m.add_hole_to_phase_field(60, 40, 12)
            m.add_hole_to_phase_field(60, 40, 55, neg=True)
        m.define()
        m._ctx.step(0, 40)
        image = m.image()
        phase = m.phase if hole else np.ones_like(image)
        for cutoff in (0.2, 0.5, 0.9):
            want = np.sum(image[phase > 1e-3] < cutoff) / np.sum(phase > 1e-3)
            assert m.excitable_fraction(cutoff, 1e-3) == want, (hole, cutoff)
        m.close()


def test_async_strip_upload_equals_synchronous_upload(cuda):
    from fib_tf_b200 import _capi
    H, W = 300, 257
    rng = np.random.default_rng(11)
    a = _capi.Context(_capi.BR, H, W, 0.1, 0.809)
    b = _capi.Context(_capi.BR, H, W, 0.1, 0.809)
    bufs = []
    for v in a.var_names:
        plane = rng.uniform(0.01, 0.9, (H, W)).astype(np.float32)
        if v == 'V':
            plane = plane * 100 - 85
        a.set_state(v, plane)
        for r0 in range(0, H, 64):
            blk = _capi.pinned_empty((min(64, H - r0), W))
            blk[:] = plane[r0:r0 + 64]
            b.set_rect_async(v, r0, 0, blk)
            bufs.append(blk)
    with pytest.raises(_capi.FibError):
        b.set_rect_async('V', 0, 0, np.zeros((4, W), np.float32))      # pageable memory is refused
    a.step(0, 3)
    b.step(0, 3)
    for v in a.var_names:
        assert np.array_equal(a.get_state(v), b.get_state(v)), v
    b.sync()
    for blk in bufs:
        _capi.pinned_free(blk)
    with pytest.raises(_capi.FibError):
        a.get_state('V', out=np.zeros((H, W), np.float16))
    with pytest.raises(_capi.FibError):
        a.get_state('V', out=np.zeros((W, H), np.float32).T)
    a.close()
    b.close()
