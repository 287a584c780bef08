"""GPU: the kernel flavours the BENCHMARKED configurations actually launch -- two cells per thread,
marching depth 2 (BASELINE configs 3 and 4, the 4096^2 roofline points) -- against the ORACLE.

launch_step (csrc/fib_kernels.cuh) switches to one cell per thread on grids of <= 320 Ki cells, so
the golden fixtures (<= 56 x 40) and the 512^2 live-oracle runs only ever see that small flavour.
Here:
  * every BR flag combination (exact, skip, cheby, cheby+skip, cheby_strict) on 1024 x 512 and the
    Courtemanche variants (multi-rate fast + slow ops, ultra, ultra + ultra-slow gate, each of them
    with the lookup table, and chronic-AF remodelling off) on 768 x 512, with a hole and a stimulus,
    100 / 50 time steps against the NumPy oracle run on the same inputs.  The oracle's table flavour
    (oracle.monodomain_np.court_lookup) reads the table the device built;
  * where oracle/_ref can be built: the tabulated flavour also against the reference's own compiled
    courtemanche.h on a 2200-column version of the table-row experiment;
  * every golden fixture replayed with FIB_SMALL_CELLS=0 (a subprocess: the switch is read once per
    process), which forces the wide flavours onto the reference-generated data.
Each test asserts, through fib_last_kernel, WHICH instantiation ran."""
import contextlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import golden_names, load_fixture
from oracle import monodomain_np as onp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
METAS = [load_fixture(n)[0] for n in golden_names() if 'long' not in n]


@pytest.fixture(scope='module')
def cuda(cuda_device):
    import cuda_adapter
    return cuda_adapter


def base_config(**kw):
    cfg = {'dt': 0.1, 'dt_per_plot': 10, 'duration': 10, 'timeline': False, 'timeline_name': 'x',
           'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False}
    cfg.update(kw)
    return cfg


def compare(kind, cfg, gpu, ref, jit, wide=None):
    """Bar per variable: oracle.monodomain_np.tolerance (flat 1e-5 / named waivers), but never tighter than
    3x the drift of the ulp-jittered oracle `jit` in this very scenario (see onp.ulp_jitter), nor than 3x the
    distance of `wide` (if given: the oracle with its V-only intermediates in float64) -- the oracle's own
    rounding, as the fixtures' `rounding` term."""
    report = []
    for v in ref.state:
        fl = onp.var_floor(kind, v)
        e = onp.rel_err(gpu.state[v], ref.state[v], fl)
        tol = max(onp.tolerance(kind, cfg, v, *onp.model_uncertainty(METAS, kind, cfg, v)),
                  3.0 * onp.rel_err(jit.state[v], ref.state[v], fl),
                  3.0 * onp.rel_err(wide.state[v], ref.state[v], fl) if wide is not None else 0.0)
        report.append((v, e, tol))
    bad = [(v, '%.3e > %.3e' % (e, t)) for v, e, t in report if not e <= t]
    assert not bad, (kind, {k: cfg.get(k) for k in ('cheby', 'skip', 'cheby_strict', 'lut', 'ultra_slow', 'chronic')},
                     bad)
    return report


@pytest.mark.parametrize('flags,kernels', [
    (dict(cheby=False, skip=False), ('BeelerReuter<exact,slow>',)),
    (dict(cheby=False, skip=True), ('BeelerReuter<exact,slow>', 'BeelerReuter<exact,fast>')),
    (dict(cheby=True, skip=False), ('BeelerReuter<cheby,slow>',)),
    (dict(cheby=True, skip=True), ('BeelerReuter<cheby,slow>', 'BeelerReuter<cheby,fast>')),
    (dict(cheby=True, skip=True, cheby_strict=True), ('BeelerReuter<strict,slow>', 'BeelerReuter<strict,fast>')),
])
def test_beeler_reuter_wide_flavour_against_the_oracle(cuda, flags, kernels):
    """BASELINE config 3's flavour: 1024 x 512 = 512 Ki cells, hole, S2 half way, 20 iterations =
    100 time steps, every state variable against the oracle."""
    from fib_tf_b200 import _capi
    cfg = base_config(width=1024, height=512, diff=0.809, **flags)
    ref, jit, gpu = onp.OracleModel('br', cfg), onp.OracleModel('br', cfg), cuda.CudaModel('br', cfg, graph=False)
    for m in (ref, jit, gpu):
        m.add_hole(300, 200, 40)
        m.define()
        m.add_pace('s2', 'luq', 10.0)
    rng = np.random.default_rng(2)
    for i in range(20):
        for m in (ref, jit, gpu):
            m.iterate()
            if i == 9:
                m.fire('s2')
        if i < 19:
            onp.ulp_jitter(jit.state, rng)
    # which instantiation ran: two cells per thread, marching depth 2, with the phase field
    last = _capi.last_kernel()
    assert 'VEC=2,R=2' in last and 'PHASE=1' in last and kernels[-1] in last, last
    compare('br', cfg, gpu, ref, jit)
    gpu.close()


@pytest.mark.parametrize('kind,extra,steps,kernel', [
    ('court', {}, 50, 'Courtemanche<fast>,VEC=2'),
    ('court', {'lut': True}, 50, 'Courtemanche<fast,lut>,VEC=2,R=2'),
    ('court_ultra', {}, 50, 'Courtemanche<all>'),
    ('court_ultra', {'ultra_slow': True}, 50, 'Courtemanche<all,us>'),
    ('court_ultra', {'lut': True}, 50, 'Courtemanche<all,lut>,VEC=2,R=2'),
    ('court_ultra', {'lut': True, 'ultra_slow': True}, 50, 'Courtemanche<all,lut,us>,VEC=2,R=2'),
    ('court', {'chronic': False}, 50, 'Courtemanche<fast>,VEC=2'),
    ('court_ultra', {'chronic': False}, 50, 'Courtemanche<all>,VEC=2'),
])
def test_courtemanche_wide_flavours_against_the_oracle(cuda, kind, extra, steps, kernel):
    """BASELINE config 4's flavours on 768 x 512 = 384 Ki cells: the multi-rate loop ('slow' every 10th
    iteration), the all-states variant, the ultra-slow gate, the lookup table and chronic-AF remodelling
    switched off; hole, S2 half way, `steps` iterations.  The oracle's table flavour reads the table the
    device built (test_gpu_court_lut.py tests that table on its own)."""
    from fib_tf_b200 import _capi
    cfg = base_config(width=768, height=512, diff=0.809 if kind == 'court' else 1.5, **extra)
    gpu = cuda.CudaModel(kind, cfg, graph=False)
    gpu.add_hole(300, 200, 40)
    gpu.define()
    table = gpu.m._ctx.get_table(_capi.TABLE_COURT_LUT, (150, 30)) if extra.get('lut') else None
    ref, jit = onp.OracleModel(kind, cfg, table=table), onp.OracleModel(kind, cfg, table=table)
    # direct flavours: the oracle's fp32 calc_inter has no correct digit right next to its removable
    # singularities (test_gpu_parity.py::test_courtemanche_removable_singularities), which a wave crosses;
    # `wide` measures that: measured with chronic=False, court_ultra, _xr_: 1.5e-5 away from the fp32 oracle,
    # 8.6e-7 in the cells that never came within 0.5 mV of a singular voltage
    wide = onp.OracleModel(kind, cfg) if table is None else None
    oracles = [m for m in (ref, jit, wide) if m is not None]
    for m in oracles:
        m.add_hole(300, 200, 40)
        m.define()
    models = [gpu] + oracles
    for m in models:
        m.add_pace('s2', 'luq', 10.0)

    def step(m):
        if m is wide:
            with float64_intermediates():
                return m.iterate()
        return m.iterate()

    gpu.iterate()
    assert kernel in _capi.last_kernel() and 'PHASE=1' in _capi.last_kernel(), _capi.last_kernel()
    rng = np.random.default_rng(3)
    for m in oracles:
        step(m)
    for i in range(1, steps):
        onp.ulp_jitter(jit.state, rng)
        for m in models:
            if kind == 'court' and (i - 1) % 10 == 0:
                if m is wide:
                    with float64_intermediates():
                        m.fire('slow')
                else:
                    m.fire('slow')
                if m is gpu and i == 1:
                    slow = kernel.split(',VEC')[0].replace('<fast', '<slow')
                    assert slow + ',VEC=2' in _capi.last_kernel(), (slow, _capi.last_kernel())
            if i == steps // 2:
                m.fire('s2')
            step(m)
    compare(kind, cfg, gpu, ref, jit, wide)
    gpu.close()


@contextlib.contextmanager
def float64_intermediates():
    """onp.court_inter evaluated in float64 (then rounded to fp32) inside the block."""
    fp32 = onp.court_inter

    def wide(V, ultra=False):
        with np.errstate(all='ignore'):
            q = fp32(np.asarray(V, np.float64), ultra)
        return {k: np.asarray(a, np.float32) for k, a in q.items()}
    onp.court_inter = wide
    try:
        yield
    finally:
        onp.court_inter = fp32


def test_lut_wide_flavour_against_the_compiled_reference_header(cuda):
    """The tabulated flavour BASELINE config 4 launches (two cells per thread, marching depth 2)
    against the reference's own courtemanche.h (oracle/_ref): the experiment of
    test_gpu_parity.py::test_lut_path_against_the_compiled_reference_header on 150 table rows x 2200
    state perturbations = 335 Ki cells (above the small-grid switch), diff = 0, no gate clip.
    One step: |new_cuda - new_ref| <= 1e-5 * max(|increment|, 1e-3 * floor) + 1 ulp(state);
    5 steps: 1e-3 in the rel_err metric (the truncating lookup is discontinuous in V)."""
    from fib_tf_b200 import _capi
    from oracle import cpu_port
    ref = cpu_port.court_ref()
    if ref is None:
        pytest.skip('oracle/_ref was not built')
    table = np.zeros([150, 30], np.float32)
    ref.ref_init_table(table)
    HI, WI, dt = 150, 2200, 0.1
    cell0 = np.zeros(21, np.float32)
    ref.ref_init_cell(cell0, 0)
    f = (0.55 + 0.9 * np.arange(WI, dtype=np.float64) / WI).astype(np.float32)       # 0.55 .. 1.45
    init = np.empty([HI, WI, 21], np.float32)
    init[:, :, 1:] = cell0[None, None, 1:] * f[None, :, None]
    gates = [2, 3, 4, 6, 7, 8, 9, 10, 11, 13, 14, 15, 17, 18, 19]      # enum States
    init[:, :, gates] = np.clip(init[:, :, gates], 1e-4, 0.9999)
    # voltages strictly inside a row of the truncating lookup i = int(V + 100)
    init[:, :, 0] = (np.arange(HI, dtype=np.float32) - 100.0)[:, None] + \
        (0.2 + 0.6 * (np.arange(WI) % 7) / 7.0).astype(np.float32)[None, :]
    padded = np.pad(init, ((1, 1), (1, 1), (0, 0)), mode='symmetric')
    H, W = padded.shape[:2]

    def cuda_run(steps):
        ctx = _capi.Context(_capi.COURT_ULTRA, H, W, dt, 0.0, flags=_capi.F_LUT | _capi.F_NO_CLIP | _capi.F_NO_GRAPH)
        ctx.set_table(_capi.TABLE_COURT_LUT, table)
        for k, name in enumerate(ctx.var_names):
            ctx.set_state(name, padded[:, :, k])
        ctx.step(_capi.OP_ODE, steps)
        out = np.stack([ctx.get_state(n) for n in ctx.var_names], axis=2)
        names, kern = list(ctx.var_names), _capi.last_kernel()
        ctx.close()
        return out[1:-1, 1:-1], names, kern

    def ref_run(steps):
        st = init.reshape(-1, 21).copy()           # (ref_euler_batch advances its argument in place)
        inc = np.zeros_like(st)
        ref.ref_euler_batch(st, inc, st.shape[0], steps, dt, table, 1)
        return st.reshape(init.shape), inc.reshape(init.shape)

    got, names, kern = cuda_run(1)
    assert 'Courtemanche<all,lut>,VEC=2,R=2' in kern, kern
    want, inc = ref_run(1)
    for k, name in enumerate(names):
        fl = onp.var_floor('court_ultra', name)
        tol = 1e-5 * np.maximum(np.abs(inc[:, :, k]), 1e-3 * fl) + np.spacing(np.abs(want[:, :, k]))
        bad = np.abs(got[:, :, k].astype(np.float64) - want[:, :, k]) > tol
        assert not bad.any(), (name, int(bad.sum()), float(np.abs(got[:, :, k] - want[:, :, k]).max()))
    # 5 steps (measured: V max 1.9e-4, _m_ 1.1e-3 in the rel_err metric).  The lookup truncates V to a table
    # row, and these perturbed states move by millivolts per step: a cell that crosses an integer voltage
    # within the ~1e-4 mV by which two fp32 implementations differ reads different rows for one step.
    # With 330 000 cells a handful of such cells is certain, so the bar is on the population: at most
    # 0.1 % of the cells off by more than 1e-3, and the typical cell within 2e-5.
    got, names, _ = cuda_run(5)
    want, _ = ref_run(5)
    for k, name in enumerate(names):
        fl = onp.var_floor('court_ultra', name)
        err = np.abs(got[:, :, k].astype(np.float64) - want[:, :, k]) / np.maximum(np.abs(want[:, :, k]), fl)
        assert np.isfinite(err).all(), name
        assert (err > 1e-3).mean() <= 1e-3, (name, float((err > 1e-3).mean()))
        assert np.median(err) <= 2e-5, (name, float(np.median(err)))


@pytest.mark.parametrize('strict', [False, True])
def test_fixtures_on_the_wide_flavours(cuda, strict):
    """Every golden fixture (the reference's own output) with FIB_SMALL_CELLS=0: the wide flavours on
    the reference-generated data, same bars as test_gpu_parity.py.  (--strict: the BR cheby fixtures
    with the reference's operation order.)"""
    env = dict(os.environ, FIB_SMALL_CELLS='0', FIB_PERSIST='0')     # wide step kernels, not the persistent one
    cmd = [sys.executable, os.path.join(ROOT, 'tests', 'gpu_parity_report.py'), '--assert'] + (['--strict'] if strict else [])
    r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=900)
    tail = '\n'.join((r.stdout + r.stderr).splitlines()[-40:])
    assert r.returncode == 0, tail
    assert 'VEC=2' in r.stdout and 'failures against the applied bar: 0' in r.stdout, tail


@pytest.mark.parametrize('name', [n for n in golden_names() if n.startswith('br_cheby') and 'long' not in n])
def test_cheby_strict_order_against_the_reference_fixture(cuda, name):
    """config['cheby_strict']: the polynomial gates in the reference's own operation order
    (br.py:215,289-301,327-331; FIB_F_CHEBY_STRICT).  What is left to differ is the last bit of expm1f /
    expf (CUDA libm vs glibc), i.e. exactly the fixtures' `noise` experiment -- and that alone moves the
    reference by 2-4e-5 on M, H, D.  So the strict flavour cannot reach 1e-5 either (measured 1.0e-5 ...
    4.5e-5 on br_cheby: profiles/r2_parity_report_strict.txt); it is held to the same bars as the
    default and must be strictly closer to the reference than Horner on the gate with the largest error."""
    meta, arr = load_fixture(name)
    errs = {}
    for strict in (False, True):
        m2 = dict(meta, config=dict(meta['config'], cheby_strict=strict))
        worst = {}

        def check(i, m):
            for v in meta['vars']:
                key = 's%d__%s' % (i, v)
                e = onp.rel_err(m.state[v], arr[key], onp.var_floor('br', v))
                tol = onp.parity_tolerance(m2, key)
                assert e <= tol, '%s %s strict=%s: rel_err %.3e > tol %.3e' % (name, key, strict, e, tol)
                worst[v] = max(worst.get(v, 0.0), e)

        m, _ = onp.run_fixture(m2, check, model_factory=cuda.CudaModel)
        m.close()
        errs[strict] = worst
    v = max(errs[False], key=errs[False].get)
    assert errs[True][v] < errs[False][v], (v, errs[True][v], errs[False][v])


DUMP = """
import sys, numpy as np
sys.path.insert(0, %r); sys.path.insert(0, %r)
from cuda_adapter import CudaModel
from fib_tf_b200 import _capi
out = {}
cfg = {'width': 200, 'height': 120, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809, 'duration': 1, 'timeline': False,
       'timeline_name': 'x', 'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False, 'graph': False}
for tag, kind, extra in (('br_exact', 'br', {}), ('br_cheby_skip', 'br', {'cheby': True, 'skip': True}),
                         ('br_strict', 'br', {'cheby': True, 'cheby_strict': True}),
                         ('court', 'court', {}), ('court_ultra_us', 'court_ultra', {'ultra_slow': True, 'diff': 1.5}),
                         ('court_lut', 'court', {'lut': True}),
                         ('court_ultra_lut_us', 'court_ultra', {'lut': True, 'ultra_slow': True, 'diff': 1.5})):
    m = CudaModel(kind, dict(cfg, **extra))
    m.add_hole(90, 60, 17)
    m.define()
    m.add_pace('s2', 'luq', 10.0)
    for i in range(8):
        m.iterate()
        if kind == 'court' and i %% 4 == 0:
            m.fire('slow')
        if i == 3:
            m.fire('s2')
    out[tag + '/kernel'] = np.array(_capi.last_kernel())
    for v in m.m._ctx.var_names:
        out[tag + '/' + v] = m.state[v]
    m.close()
np.savez(sys.argv[1], **out)
"""


def test_packed_pairs_are_bit_identical_to_scalar_cells(cuda, tmp_path):
    """Packed fp32 (fma/mul/add.rn.f32x2, csrc/fib_math.cuh) rounds every lane exactly like the scalar
    instruction and the library is built with -fmad=false, so the two-cells-per-thread flavours (one f2
    pair) must reproduce the one-cell-per-thread flavours BIT FOR BIT: the same run with the small-grid
    switch at its default (scalar cells) and at 0 (pairs), in two subprocesses (the switch is read once)."""
    script = DUMP % (ROOT, os.path.join(ROOT, 'tests'))
    files = []
    for small in (None, '0'):
        env = dict(os.environ, FIB_PERSIST='0')
        if small is not None:
            env['FIB_SMALL_CELLS'] = small
        f = str(tmp_path / ('dump_%s.npz' % small))
        r = subprocess.run([sys.executable, '-c', script, f], env=env, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        files.append(np.load(f))
    a, b = files
    assert 'VEC=1' in str(a['br_exact/kernel']) and 'VEC=2' in str(b['br_exact/kernel'])
    assert 'VEC=2' in str(b['court_ultra_us/kernel']) and 'VEC=2' in str(b['br_strict/kernel'])
    assert 'Courtemanche<fast,lut>,VEC=1' in str(a['court_lut/kernel'])
    assert 'Courtemanche<fast,lut>,VEC=2' in str(b['court_lut/kernel'])
    assert 'Courtemanche<all,lut,us>,VEC=1' in str(a['court_ultra_lut_us/kernel'])
    assert 'Courtemanche<all,lut,us>,VEC=2' in str(b['court_ultra_lut_us/kernel'])
    for k in a.files:
        if not k.endswith('/kernel'):
            assert np.array_equal(a[k], b[k], equal_nan=True), k
