"""GPU: the CUDA path (through the C ABI, via the drop-in Python API) against
  (1) the golden fixtures = the UNMODIFIED reference executed under oracle/tfshim.py,
  (2) the NumPy oracle run live on the same seeded inputs at 512^2,
  (3) size-independent properties at the full benchmark sizes.

Tolerance (written here, used everywhere below): for every state variable and snapshot,
    rel_err = max |cuda - ref| / max(|ref|, floor(var))  <=  1e-5            (BASELINE.json's bar)
(floor: 0.1 % of the variable's range; the full range for the accumulating voltage V of BR /
Courtemanche -- see oracle.monodomain_np.var_floor; a NaN / Inf pattern that differs from the
reference's is an infinite error).  The ONLY exceptions are the variables named in
oracle.monodomain_np.WAIVERS -- the gates driven by the degree-8 polynomial fits of BR `cheby`
(M, H, J, D, XI), D / XI of the exact-gate `skip` schedule and the Courtemanche release gates
_u_ / _v_ -- for which the reference's OWN fp32 result moves by more than 1e-5 when only its math
library is swapped (`noise`, recorded per plane in the fixtures by oracle/make_golden.py with
oracle/tfshim.ALT_LIBM) or against float64 (`rounding`, tfshim.WIDE).  Those are held to
min(cap, max(1e-5, 3 * that uncertainty)) with a hard cap per flavour.  The measured error of every
variable against the flat bar is committed in profiles/r2_parity_report.txt."""
import numpy as np
import pytest

from conftest import golden_names, load_fixture
from oracle import monodomain_np as onp

pytestmark = pytest.mark.gpu

SHORT = [n for n in golden_names() if 'long' not in n]
LONG = [n for n in golden_names() if 'long' in n]


@pytest.fixture(scope='module')
def cuda(cuda_device):
    import cuda_adapter
    return cuda_adapter


@pytest.mark.parametrize('name', SHORT)
def test_per_step_parity_with_reference_fixture(cuda, name):
    meta, arr = load_fixture(name)
    seen = []

    def check(i, m):
        for v in meta['vars']:
            key = 's%d__%s' % (i, v)
            e = onp.rel_err(m.state[v], arr[key], onp.var_floor(meta['model'], v))
            tol = onp.parity_tolerance(meta, key)
            assert e <= tol, '%s %s: rel_err %.3e > tol %.3e' % (name, key, e, tol)
        seen.append(i)

    m, _ = onp.run_fixture(meta, check, model_factory=cuda.CudaModel)
    m.close()
    assert seen == meta['snaps']


def crossings(trace, level, dt_iter):
    """Linear-interpolated times (ms) at which the trace crosses `level` upwards / downwards."""
    t = np.asarray(trace, dtype=np.float64)
    up, dn = [], []
    for i in range(1, len(t)):
        if t[i - 1] < level <= t[i]:
            up.append((i - 1 + (level - t[i - 1]) / (t[i] - t[i - 1])) * dt_iter)
        if t[i - 1] >= level > t[i]:
            dn.append((i - 1 + (t[i - 1] - level) / (t[i - 1] - t[i])) * dt_iter)
    return up, dn


@pytest.mark.parametrize('name', LONG)
def test_long_horizon_apd_and_activation_time(cuda, name):
    """One full action potential on a strip: activation time at the probe (conduction velocity)
    and action-potential duration must match the reference within 1 % (BASELINE.json)."""
    meta, arr = load_fixture(name)
    m, trace = onp.run_fixture(meta, None, model_factory=cuda.CudaModel)
    m.close()
    lo, hi = onp.OracleModel.RANGE[meta['model']]
    level = lo + 0.3 * (hi - lo) if meta['model'] != 'fenton4v' else 0.3
    dt_iter = meta['dt_per_step'] * meta['config']['dt']
    up_r, dn_r = crossings(arr['probe'], level, dt_iter)
    up_c, dn_c = crossings(trace, level, dt_iter)
    assert len(up_r) >= 1 and len(dn_r) >= 1 and len(up_c) == len(up_r) and len(dn_c) == len(dn_r)
    assert abs(up_c[0] - up_r[0]) <= 0.01 * up_r[0]                     # activation time -> CV
    apd_r, apd_c = dn_r[0] - up_r[0], dn_c[0] - up_c[0]
    assert abs(apd_c - apd_r) <= 0.01 * apd_r, (apd_c, apd_r)
    # and the whole trace stays close in absolute terms (1 % of the voltage range)
    assert np.max(np.abs(trace - arr['probe'])) <= 0.01 * (hi - lo)


METAS = [load_fixture(n)[0] for n in SHORT]


def live_tolerance(kind, cfg, var, drift=0.0):
    """Bar for a run that has no fixture of its own: 1e-5 (for a waived variable the rule of
    oracle.monodomain_np.tolerance with the worst uncertainty the fixtures of that flavour recorded),
    but never tighter than 3x `drift` = how far the ORACLE ITSELF moves in this very scenario when
    every cell is jittered by +-1 ulp after every iteration (onp.ulp_jitter): a stimulus into
    refractory tissue or a steep wave front amplifies one ulp per step to 1e-5 ... 2e-4 in the
    Courtemanche gates, and no second fp32 implementation can be closer to the oracle than that."""
    return max(onp.tolerance(kind, cfg, var, *onp.model_uncertainty(METAS, kind, cfg, var)), 3.0 * drift)


@pytest.mark.parametrize('kind,cfg,iters', [
    ('fenton4v', dict(diff=1.5), 10),
    ('br', dict(diff=0.809, cheby=True, skip=False), 20),
    ('br', dict(diff=0.809, cheby=False, skip=True), 20),
    ('court', dict(diff=0.809, width=256, height=256), 100),
    ('court_ultra', dict(diff=1.5, width=256, height=256, ultra_slow=True), 100),
    ('court', dict(diff=0.809, width=256, height=256, lut=True), 100),
    ('court_ultra', dict(diff=1.5, width=256, height=256, lut=True, ultra_slow=True), 100),
    ('court', dict(diff=0.809, width=256, height=256, chronic=False), 100),
])
def test_100_steps_against_live_oracle(cuda, kind, cfg, iters):
    """BASELINE configs 1-2 (512^2 with the shipped holes) and Courtemanche at 256^2 (one cell per
    thread), also with the lookup table and without chronic-AF remodelling: 100 time steps, every
    state variable, against the oracle run here on the same inputs (the oracle's table flavour reads
    the table the device built)."""
    from fib_tf_b200 import _capi
    base = {'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'duration': 10,
            'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False,
            'cheby': False, 'ultra_slow': False}
    base.update(cfg)
    W = base['width']
    gpu = cuda.CudaModel(kind, base)
    gpu.add_hole(W // 2, W // 2, 30 * W // 512)
    gpu.define()
    table = gpu.m._ctx.get_table(_capi.TABLE_COURT_LUT, (150, 30)) if cfg.get('lut') else None
    ref, jit = onp.OracleModel(kind, base, table=table), onp.OracleModel(kind, base, table=table)
    for m in (ref, jit):
        m.add_hole(W // 2, W // 2, 30 * W // 512)
        m.define()
    for m in (ref, jit, gpu):
        m.add_pace('s2', 'luq', 1.0 if kind == 'fenton4v' else 10.0)
    rng = np.random.default_rng(1)
    for i in range(iters):
        for m in (ref, jit, gpu):
            m.iterate()
            if kind == 'court' and i % 10 == 0:
                m.fire('slow')
            if i == iters // 2:
                m.fire('s2')
        if i == 0 and kind.startswith('court'):
            last = _capi.last_kernel()
            assert 'VEC=1' in last and ('lut' in last) == bool(cfg.get('lut')), last
        if i + 1 < iters:
            onp.ulp_jitter(jit.state, rng)
    for v in ref.state:
        fl = onp.var_floor(kind, v)
        e = onp.rel_err(gpu.state[v], ref.state[v], fl)
        tol = live_tolerance(kind, base, v, onp.rel_err(jit.state[v], ref.state[v], fl))
        assert e <= tol, '%s %s: rel_err %.3e > %.3e' % (kind, v, e, tol)
    gpu.close()


@pytest.mark.parametrize('kind,extra', [('fenton4v', {}), ('br', {'cheby': True, 'skip': True}),
                                        ('court', {}), ('court_ultra', {'ultra_slow': True}),
                                        # large enough for the wide kernel flavours and deeper marching
                                        ('br', {'cheby': True, 'width': 1300, 'height': 900}),
                                        ('fenton4v', {'width': 1100, 'height': 1000}),
                                        ('court', {'lut': True}), ('court_ultra', {'lut': True, 'ultra_slow': True})])
def test_row_shards_are_bit_identical_to_the_unsharded_run(cuda, kind, extra):
    """Emulates R row shards in one process (fib_step_group, device-to-device halo rows) and
    requires BIT-IDENTICAL planes: sharding must not change arithmetic; seams are interior."""
    from fib_tf_b200 import _capi
    from fib_tf_b200.sharding import partition_rows
    cfg = {'width': 72, 'height': 45, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.1, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False,
           'cheby': False, 'ultra_slow': False}
    cfg.update(extra)
    whole = cuda.CudaModel(kind, cfg)
    whole.add_hole(30, 20, 7)
    whole.define()
    m = whole.m
    c0 = m._ctx
    W0 = cfg['width']
    flags = m._flags() if hasattr(m, '_flags') else (
        (_capi.F_CHEBY if cfg['cheby'] else 0) | (_capi.F_SKIP if cfg['skip'] else 0)
        if kind == 'br' else 0)
    parts = partition_rows(cfg['height'], 4)
    shards = [_capi.Context(m.MODEL_ID, cfg['height'], cfg['width'], cfg['dt'], cfg['diff'],
                            flags=flags | _capi.F_NO_GRAPH, row0=r0, rows=n) for r0, n in parts]
    for s, (r0, n) in zip(shards, parts):
        for v in c0.var_names:
            s.set_state(v, c0.get_state(v)[r0:r0 + n])
        s.set_phase(m.phase, 0)
        if kind == 'br':
            s.set_table(_capi.TABLE_BR_CHEBY, m.chebyshev_table())
        if flags & _capi.F_LUT:
            s.build_lut()
    for it in range(6):
        c0.step(_capi.OP_ODE, 1)
        _capi.step_group(shards, _capi.OP_ODE, 1)
        if kind == 'court' and it % 2 == 0:
            c0.step(_capi.OP_SLOW, 1)
            _capi.step_group(shards, _capi.OP_SLOW, 1)
        if it == 2:     # a stimulus crossing the seams
            args = (c0.var_names[0], 5, 40, 3, 30, float(m.max_v) * 0.5, float(m.min_v))
            c0.stimulate(*args)
            for s in shards:
                s.stimulate(*args)
    for v in c0.var_names:
        full = c0.get_state(v)
        got = np.concatenate([s.get_state(v) for s in shards], axis=0)
        assert np.array_equal(full, got), 'variable %s differs between sharded and unsharded' % v
    for s in shards:
        s.close()
    whole.close()


def test_cuda_graph_replay_is_bit_identical_to_direct_launches(cuda):
    cfg = {'width': 100, 'height': 64, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': True,
           'cheby': True, 'ultra_slow': False}
    a, b = cuda.CudaModel('br', cfg), cuda.CudaModel('br', cfg, graph=False)
    for m in (a, b):
        m.add_hole(40, 30, 8)
        m.define()
        for _ in range(7):
            m.iterate()
    for v in a.m._ctx.var_names:
        assert np.array_equal(a.state[v], b.state[v]), v
    a.close()
    b.close()


def test_planar_wave_property_at_4096(cuda):
    """Size-independent property at the benchmark size: with the y-uniform S1 initial state every
    row of a 4096-wide grid evolves identically, and equals the oracle's 5-row strip of the same
    width within the parity tolerance."""
    cfg = {'width': 4096, 'height': 4096, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False}
    gpu = cuda.CudaModel('fenton4v', cfg)
    gpu.define()
    ref = onp.OracleModel('fenton4v', dict(cfg, height=5))
    ref.define()
    for _ in range(5):
        gpu.iterate()
        ref.iterate()
    for v in ('U', 'V', 'W', 'S'):
        a = gpu.state[v]
        assert np.array_equal(a, np.broadcast_to(a[0], a.shape)), 'rows differ for %s' % v
        assert onp.rel_err(a[:5], ref.state[v], 1e-3) <= 1e-5
    gpu.close()


def test_planar_wave_property_at_the_bench_size_32768(cuda):
    """The same property at the size the bench line is quoted on (32768^2, 20 GiB of state): rows
    sampled across the grid are identical to each other and match the oracle's 5-row strip."""
    N = 32768
    cfg = {'width': N, 'height': N, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False}
    gpu = cuda.CudaModel('fenton4v', cfg)
    gpu.define()
    ref = onp.OracleModel('fenton4v', dict(cfg, height=5))
    ref.define()
    for _ in range(2):
        gpu.iterate()
        ref.iterate()
    ctx = gpu.m._ctx
    for v in ('U', 'V', 'W', 'S'):
        rows = [ctx.get_rect(v, r, r + 1, 0, N)[0] for r in (0, 1, 2, 4097, 16384, N - 2, N - 1)]
        for a in rows[1:]:
            assert np.array_equal(a, rows[0]), v
        assert onp.rel_err(rows[0], ref.state[v][2], 1e-3) <= 1e-5, v
    assert gpu.m.nonfinite_cells() == {}
    gpu.close()


def test_uniform_rest_state_stays_uniform_at_4096(cuda):
    """A uniform field has a Laplacian of exactly 0 in fp32 (4c + 2c - 6c), so a uniform BR state
    must stay exactly uniform at any size."""
    cfg = {'width': 4096, 'height': 4096, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809,
           'duration': 1, 'timeline': False, 'timeline_name': 'x', 'save_graph': False,
           'skip': False, 'cheby': True}
    gpu = cuda.CudaModel('br', cfg)
    gpu.define(False)
    for _ in range(4):
        gpu.iterate()
    for v in gpu.m._ctx.var_names:
        a = gpu.state[v]
        assert a.min() == a.max(), v
    gpu.close()


def test_empty_and_edge_geometries(cuda):
    """Smallest legal grid (3x3), a width that is not a multiple of the vector width, a stimulus
    with an empty rectangle, and an n_iter of 0."""
    for H, W in ((3, 3), (3, 7), (9, 5), (17, 33)):
        cfg = {'width': W, 'height': H, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.0, 'duration': 1,
               'timeline': False, 'timeline_name': 'x', 'save_graph': False}
        ref, gpu = onp.OracleModel('fenton4v', cfg), cuda.CudaModel('fenton4v', cfg)
        for m in (ref, gpu):
            m.define()
            m.iterate()
        gpu.m._ctx.step(0, 0)
        gpu.m._ctx.stimulate('U', 0, 0, 0, 0, 1.0, 0.0)
        ref.state['U'] = np.maximum(ref.state['U'], np.float32(0.0))
        for v in ('U', 'V', 'W', 'S'):
            assert onp.rel_err(gpu.state[v], ref.state[v], 1e-3) <= 1e-5, (H, W, v)
        gpu.close()


def test_lut_path_against_the_compiled_reference_header(cuda):
    """courtemanche.h compiled on the host (oracle/_ref): deriv<Courtemanche> with its 150x30 table
    and forward Euler state += dt*rate (SURVEY.md 8c item 2), against the CUDA LUT flavour with the
    SAME table uploaded, the native no-clip gate rule and diff = 0 (every cell an independent ODE).

    (1) ONE step from 150 x 8 different states: every table row (voltages at half-integers, safely
        inside a row of the truncating lookup) x 8 perturbations of the gates / concentrations.
        Bar: |new_cuda - new_ref| <= 1e-5 * max(|increment|, 1e-3 * floor) + 1 ulp(state).
    (2) 30 steps from the same states: the lookup is discontinuous in V, so a 1-ulp difference just
        below an integer voltage reads another table row; bar 1e-3 in the rel_err metric."""
    from fib_tf_b200 import _capi
    from oracle import cpu_port
    ref = cpu_port.court_ref()
    if ref is None:
        pytest.skip('oracle/_ref was not built')
    table = np.zeros([150, 30], np.float32)
    ref.ref_init_table(table)
    HI, WI, dt = 150, 8, 0.1
    cell0 = np.zeros(21, np.float32)
    ref.ref_init_cell(cell0, 0)
    init = np.zeros([HI, WI, 21], np.float32)
    for r in range(HI):
        for c in range(WI):
            st = cell0.copy()
            f = np.float32(0.55 + 0.13 * c)
            st[1:] = st[1:] * f
            gates = [2, 3, 4, 6, 7, 8, 9, 10, 11, 13, 14, 15, 17, 18, 19]      # enum States
            st[gates] = np.clip(st[gates], 1e-4, 0.9999)
            st[0] = r - 100 + 0.5
            init[r, c] = st
    # one ring of SYMMETRIC padding around the 150 x 8 experiment, so that the kernel's
    # enforce_boundary (border ring := neighbouring interior cell) changes nothing
    init = np.pad(init, ((1, 1), (1, 1), (0, 0)), mode='symmetric')
    H, W = init.shape[:2]

    def cuda_run(steps):
        ctx = _capi.Context(_capi.COURT_ULTRA, H, W, dt, 0.0, flags=_capi.F_LUT | _capi.F_NO_CLIP)
        ctx.set_table(_capi.TABLE_COURT_LUT, table)
        for k, name in enumerate(ctx.var_names):
            ctx.set_state(name, init[:, :, k])
        ctx.step(_capi.OP_ODE, steps)
        out = np.stack([ctx.get_state(n) for n in ctx.var_names], axis=2)
        names = list(ctx.var_names)
        ctx.close()
        return out, names

    def ref_run(steps):
        out = init.copy()
        rate = np.zeros(21, np.float32)
        inc = np.zeros_like(out)
        for r in range(H):
            for c in range(W):
                st = out[r, c].copy()
                for _ in range(steps):
                    ref.ref_deriv(st, rate, dt, table, 1)
                    inc[r, c] = np.float32(dt) * rate
                    st = (st + np.float32(dt) * rate).astype(np.float32)
                out[r, c] = st
        return out, inc

    got, names = cuda_run(1)
    want, inc = ref_run(1)
    for k, name in enumerate(names):
        fl = onp.var_floor('court_ultra', name)
        tol = 1e-5 * np.maximum(np.abs(inc[:, :, k]), 1e-3 * fl) + np.spacing(np.abs(want[:, :, k]))
        bad = np.abs(got[:, :, k].astype(np.float64) - want[:, :, k]) > tol
        assert not bad.any(), (name, int(bad.sum()), float(np.abs(got[:, :, k] - want[:, :, k]).max()))
    got, names = cuda_run(30)
    want, _ = ref_run(30)
    for k, name in enumerate(names):
        e = onp.rel_err(got[:, :, k], want[:, :, k], onp.var_floor('court_ultra', name))
        assert e <= 1e-3, (name, e)


def test_run_generator_observers_and_masked_means(cuda):
    """The drop-in driver loop: run() yields, fire_op between iterations, the headless cycle-length
    probe, keep_state, a Screen stand-in, and the on-device pseudo-EGM reduction against NumPy."""
    from fib_tf_b200.br import BeelerReuter
    from fib_tf_b200.egm import create_mask
    from fib_tf_b200.screen import Screen
    cfg = {'width': 64, 'height': 64, 'dt': 0.1, 'dt_per_plot': 5, 'diff': 0.809, 'duration': 30,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False, 'cheby': True}
    m = BeelerReuter(cfg)
    m.add_hole_to_phase_field(50, 50, 7)
    m.define()
    m.add_pace_op('s2', 'top', 10.0)
    slot = m.add_probe_mask(create_mask(m, 24, 30, 6))
    seen, spikes = [], []
    m.cl_observer = lambda i, cl: spikes.append((i, cl))
    im = Screen(m.height, m.width, 'test')
    for i in m.run(im, block=False):
        seen.append(i)
        if i == 3:
            m.fire_op('s2')
    assert seen == list(range(m.samples)) and m.samples == 60
    assert im.frames_shown == 60 and im.last.shape == (64, 64)
    assert len(spikes) == 1 and 30 < spikes[0][0] < 60      # the S1 wave reaches [20, W//2] at ~24 ms
    img = m.image()
    want = float(np.mean(img * create_mask(m, 24, 30, 6)))
    got = m.masked_image_mean(slot)
    assert abs(got - want) <= 1e-5 * abs(want) + 1e-9
    # phase-weighted mean (court_ultra.py:466-480)
    swx, sw = m._ctx.weighted_sum('M')
    mm = m._State['M'].eval()
    assert abs(swx / sw - np.average(mm, weights=m.phase)) <= 1e-5
    m.close()


def test_checkpoint_restart_and_timeline(cuda, tmp_path):
    """run(keep_state=True) -> model.state dict -> np.save / np.load -> define(state=...)
    (ionic.py:226-229, court.py:49-56, court_ultra.py:511,518): the restarted run must continue
    bit-identically; config['timeline'] writes a chrome trace and advances the state once more
    (ionic.py:231-241)."""
    import json as _json
    from fib_tf_b200.court import Courtemanche
    cfg = {'width': 40, 'height': 24, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809, 'duration': 2,
           'timeline': False, 'timeline_name': str(tmp_path / 'trace.json'), 'save_graph': False}

    def drive(m, **kw):
        for i in m.run(None, block=False, **kw):
            if i % 10 == 0:
                m.fire_op('slow')

    whole = Courtemanche(dict(cfg, duration=4))
    whole.add_hole_to_phase_field(20, 12, 4)
    whole.define()
    drive(whole)
    a = Courtemanche(cfg)
    a.add_hole_to_phase_field(20, 12, 4)
    a.define()
    drive(a, keep_state=True)
    np.save(str(tmp_path / 'state_small'), a.state)
    state = np.load(str(tmp_path / 'state_small.npy'), allow_pickle=True).item(0)
    assert sorted(state) == sorted(a._ctx.var_names)
    b = Courtemanche(dict(cfg, timeline=True))
    b.add_hole_to_phase_field(20, 12, 4)
    b.define(s1=False, state=state)
    drive(b)
    trace = _json.load(open(cfg['timeline_name']))
    assert trace['traceEvents'][0]['dur'] > 0
    # b ran 20 + 1 traced iterations after the restart: advance `whole` by the same extra step
    whole._ctx.step(0, 1)
    for v in whole._ctx.var_names:
        assert np.array_equal(whole._State[v].eval(), b._State[v].eval()), v
    for m in (whole, a, b):
        m.close()


@pytest.mark.parametrize('module,frames', [('fib_tf_b200.fenton', 100), ('fib_tf_b200.br', 100)])
def test_reference_driver_blocks_run_unchanged(cuda, module, frames, tmp_path, monkeypatch):
    """The `__main__` blocks of the drop-in modules are the reference's own driver loops
    (fenton.py:155-187, br.py:347-382: 512^2, 1000 ms, hole, S2 at 210/300 ms, a frame into
    cube.npy every 10 ms).  They must run headless and leave a re-entrant wave behind."""
    import runpy
    monkeypatch.chdir(tmp_path)
    runpy.run_module(module, run_name='__main__')
    cube = np.load(str(tmp_path / 'cube.npy'), mmap_mode='r')
    assert cube.shape == (frames, 512, 512)
    last = np.asarray(cube[-1])
    assert np.isfinite(last).all() and 0.0 <= last.min() and last.max() <= 1.0 + 1e-6
    # activity persists long after S1 (10 ms) and S2 died out only if the S1-S2 protocol produced a
    # spiral: an excited region (image > 0.5) is still present in the last frames
    assert (np.asarray(cube[-10:]) > 0.5).mean() > 0.01


@pytest.mark.parametrize('ultra', [False, True])
def test_courtemanche_driver_loops_stay_finite(cuda, ultra):
    """The driver loops of court.py:582-636 / court_ultra.py:489-512 (holes incl. neg=True, S2,
    'slow' every 10th iteration, 'trend', cl_observer, keep_state) for 600 ms at 256^2: finite
    state, a propagated S1 wave, gates inside their clip range."""
    from functools import partial
    from fib_tf_b200 import court, court_ultra
    cfg = {'width': 256, 'height': 256, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5 if ultra else 0.809,
           'duration': 600, 'skip': False, 'cheby': True, 'timeline': False,
           'timeline_name': 'unused.json', 'save_graph': False, 'ultra_slow': ultra}
    mod = court_ultra if ultra else court
    m = mod.Courtemanche(cfg)
    m.add_hole_to_phase_field(128, 128, 15)
    m.add_hole_to_phase_field(128, 128, 122, neg=True)
    m.define()
    m.add_pace_op('s2', 'luq', 10.0)
    log = []
    m.cl_observer = partial(court_ultra.cl_observer, m, log, 0) if ultra else \
        (lambda i, cl: log.append((i, cl)))
    s2 = m.millisecond_to_step(300)
    trend = []
    for i in m.run(None, keep_state=True, block=False):
        if i % 10 == 0:
            m.fire_op('slow')
            m.fire_op('trend')
            trend.append(m._Trend.eval())
        if i == s2:
            m.fire_op('s2')
    trend = np.asarray(trend)
    assert np.isfinite(trend).all() and trend[:, 0].max() > -20.0        # the wave passed the probe
    assert sorted(m.state) == sorted(m._ctx.var_names)
    for name, a in m.state.items():
        assert np.isfinite(a).all(), name
    for g in ('_m_', '_h_', '_j_', '_d_', '_f_', '_u_', '_v_', '_w_'):
        assert 1e-5 <= m.state[g].min() and m.state[g].max() <= 0.99999 + 1e-7, g
    q = m.calc_inter(-50.0)
    assert abs(q['m_inf'] - 0.268253) < 1e-5 and abs(q['i_NaCab'] - 102066.71) < 1.0   # SURVEY B.4
    m.close()


def test_async_frame_grab_equals_synchronous_read(cuda):
    from fib_tf_b200 import _capi
    from fib_tf_b200.br import BeelerReuter
    cfg = {'width': 300, 'height': 200, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False, 'cheby': True}
    m = BeelerReuter(cfg)
    m.define()
    m._ctx.step(0, 7)
    want = m.image()
    buf = _capi.pinned_empty((200, 300))
    m.image_async(buf)
    m._ctx.step(0, 9)                  # keeps stepping while the frame travels
    got = m.image_wait()
    assert np.array_equal(got, want)
    m.image_async(buf)                 # staging buffer is reused safely
    assert np.array_equal(m.image_wait(), m.image())
    _capi.pinned_free(buf)
    assert m.nonfinite_cells() == {}
    bad = m._State['M'].eval()
    bad[5, 7] = np.nan
    bad[9, 1] = np.inf
    m._State['M'].assign(bad)
    assert m.nonfinite_cells() == {'M': 2}
    m.close()


@pytest.mark.parametrize('name', SHORT)
def test_cuda_is_as_close_to_exact_arithmetic_as_the_reference(cuda, name):
    """Independent of any tolerance on |cuda - ref|: the fixtures keep the float64 evaluation of the
    reference graph (fp32 parameters and inputs, double arithmetic) for the last snapshot.  The
    CUDA planes must be as close to it as the reference's own fp32 run is (factor 2.5, floor 1e-5
    in the rel_err metric)."""
    meta, arr = load_fixture(name)
    last = max(meta['snaps'])
    out = {}

    def grab(i, m):
        if i == last:
            for v in meta['vars']:
                out[v] = m.state[v]

    m, _ = onp.run_fixture(meta, grab, model_factory=cuda.CudaModel)
    m.close()
    for v in meta['vars']:
        fl = onp.var_floor(meta['model'], v)
        truth = arr['wide__' + v]
        e_ref = onp.rel_err(arr['s%d__%s' % (last, v)], truth, fl)
        e_cuda = onp.rel_err(out[v], truth, fl)
        assert e_cuda <= max(1e-5, 2.5 * e_ref), '%s %s: cuda %.2e vs reference %.2e from exact' % (
            name, v, e_cuda, e_ref)


@pytest.mark.parametrize('flags', [dict(cheby=False, skip=False), dict(cheby=False, skip=True),
                                   dict(cheby=True, skip=False)])
def test_beeler_reuter_removable_singularities(cuda, flags):
    """br.py:150-151 and the alpha_m of br.py:52 are 0/0 at V == -23.0 and V == -47.0 exactly; the
    reference's GPU clip turns the NaN into the upper bound (fib_common.cuh: clip_tf).  The kernel
    evaluates both terms through an expm1 polynomial within ~3 mV of the singular points and reuses
    exponentials across gates, so this test plants cells exactly on, next to and around the switch
    points (|0.04 (V+23)|, |0.1 (V+47)| = 0.125), plus a sweep over the whole clipped voltage range,
    in a diffusion-free grid (every cell an independent ODE) and requires the first iteration (5
    time steps) to agree with the oracle.  Cells within 0.3 mV of a singular point (but not on it)
    are skipped: there the reference's own fp32 cancellation is worse than 1e-5."""
    H, W = 34, 131
    cfg = {'width': W, 'height': H, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.0, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False}
    cfg.update(flags)
    deltas = [0.0, 0.5, -0.5, 1.0, -1.0, 1.2, -1.3, 3.0, -3.0, 3.12, -3.12, 3.13, -3.13, 3.2, -3.2, 6.0, -6.0]
    special = np.float32([s + d for s in (-23.0, -47.0) for d in deltas])
    rng = np.random.default_rng(5)
    V = rng.uniform(-85.0, 25.0, size=(H, W)).astype(np.float32)
    V.flat[:4 * special.size] = np.tile(special, 4)
    rng.shuffle(V.reshape(-1))
    near = np.zeros_like(V, bool)
    for s in (-23.0, -47.0):
        near |= (np.abs(V - np.float32(s)) < 0.3) & (V != np.float32(s))
    assert (V == np.float32(-23.0)).sum() >= 4 and (V == np.float32(-47.0)).sum() >= 4
    state = {'V': V, 'C': rng.uniform(5e-5, 5e-3, (H, W)).astype(np.float32)}
    for g in ('M', 'H', 'J', 'D', 'F', 'XI'):
        state[g] = rng.uniform(1e-3, 0.998, (H, W)).astype(np.float32)
    ref, gpu = onp.OracleModel('br', cfg), cuda.CudaModel('br', cfg)
    ref.define(s1=False)
    gpu.define(s1=False)
    for k, a in state.items():
        ref.state[k] = a.copy()
        gpu.m._State[k].assign(a)
    with np.errstate(all='ignore'):
        ref.iterate()
    gpu.iterate()
    inner = np.zeros((H, W), bool)
    inner[1:-1, 1:-1] = True                      # the border ring is overwritten by enforce_boundary
    keep = inner & ~near
    # random states over the WHOLE voltage range, including where the polynomial fits are worst
    # (tau_h < 0 below -83.85 mV) and the cells that took the NaN -> clip path: exact gates measured
    # worst 2.3e-5 (C of those cells, 5 steps later), hence 5e-5; polynomial gates: the waiver caps
    for v in ref.state:
        got, want = gpu.state[v], ref.state[v]
        assert np.isfinite(got[inner]).all() and np.isfinite(want[inner]).all(), v
        e = onp.rel_err(got[keep], want[keep], onp.var_floor('br', v))
        tol = max(5e-5, live_tolerance('br', cfg, v))
        assert e <= tol, '%s %s: rel_err %.3e > %.3e' % (flags, v, e, tol)
    # the cells planted ON the singular points took the reference's NaN -> upper clip bound path
    on23 = inner & (V == np.float32(-23.0))
    assert on23.any() and (gpu.state['V'][on23] > 15.0).all() and (ref.state['V'][on23] > 15.0).all()
    gpu.close()


def test_courtemanche_removable_singularities(cuda):
    """court.py:316-327,398-413: tau_d, tau_w and the alpha/beta of xr and xs are x/(e^y - 1) shapes
    guarded only at x == 0 exactly.  One ulp next to a singular voltage the reference's own fp32
    result is noise (its e^y - 1 has no correct digit; for V one ulp above 3.3328 mV it is exactly
    0, i.e. tau_xr = 0 and xr jumps to its steady state), so those cells are checked against the
    SAME formulas evaluated in float64, where the kernel (expm1 polynomial behind a warp vote,
    model_court.cuh) must be accurate; all other cells are checked against the fp32 oracle."""
    H, W, dt = 20, 66, 0.1
    cfg = {'width': W, 'height': H, 'dt': dt, 'dt_per_plot': 10, 'diff': 0.0, 'duration': 1,
           'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'ultra_slow': False}
    sing = np.float32([-10.0001, 7.9, -14.1, 3.3328, 19.9])
    vals = []
    for s in sing:
        for k in (0, 1, -1, 2, -2, 3, -3, 10, -10, 1000, -1000, 30000, -30000):
            v = np.float32(s)
            for _ in range(abs(k)):
                v = np.nextafter(v, np.float32(np.inf if k > 0 else -np.inf), dtype=np.float32)
            vals.append(v)
    vals = np.float32(vals)
    rng = np.random.default_rng(7)
    V = rng.uniform(-90.0, 40.0, size=(H, W)).astype(np.float32)
    V.flat[:4 * vals.size] = np.tile(vals, 4)
    rng.shuffle(V.reshape(-1))
    gates = ('_m_', '_h_', '_j_', '_oa_', '_oi_', '_ua_', '_ui_', '_xr_', '_xs_', '_d_', '_f_', '_f_Ca_',
             '_u_', '_v_', '_w_')
    ref, gpu = onp.OracleModel('court_ultra', cfg), cuda.CudaModel('court_ultra', cfg)
    ref.define(s1=False)
    gpu.define(s1=False)
    init = {k: a.copy() for k, a in ref.state.items()}
    init['V'] = V
    for g in gates:
        init[g] = rng.uniform(1e-3, 0.998, (H, W)).astype(np.float32)
    for k, a in init.items():
        ref.state[k] = a.copy()
        gpu.m._State[k].assign(a)
    with np.errstate(all='ignore'):
        ref.iterate()
    gpu.iterate()
    inner = np.zeros((H, W), bool)
    inner[1:-1, 1:-1] = True
    near = np.zeros((H, W), bool)
    for s in sing:
        near |= np.abs(V - s) < 0.5
    assert (near & inner).sum() >= 100
    for v in ref.state:
        got, want = gpu.state[v], ref.state[v]
        assert np.isfinite(got).all(), v
        keep = inner & ~near
        e = onp.rel_err(got[keep], want[keep], onp.var_floor('court_ultra', v))
        assert e <= 5e-5, (v, e)
    # every cell, near-singular ones included, against float64: g + (g - g_inf) expm1(-dt / tau)
    with np.errstate(all='ignore'):
        q = onp.court_inter(V.astype(np.float64))
    for g, inf, tau in (('_d_', 'd_infinity', 'tau_d'), ('_w_', 'w_infinity', 'tau_w'),
                        ('_xr_', 'xr_infinity', 'tau_xr'), ('_xs_', 'xs_infinity', 'tau_xs')):
        g0 = init[g].astype(np.float64)
        exact = np.clip(g0 + (g0 - q[inf]) * np.expm1(-dt / q[tau]), 1e-5, 0.99999)
        e = onp.rel_err(gpu.state[g][inner], exact[inner], onp.var_floor('court_ultra', g))
        assert e <= 2e-5, (g, e)
    gpu.close()


@pytest.mark.parametrize('hole', [False, True])
@pytest.mark.parametrize('H,W,nshards', [(3, 4, 1), (7, 8, 1), (45, 72, 4), (64, 128, 2), (130, 244, 3),
                                         (300, 500, 1), (1000, 1100, 4)])
def test_two_steps_per_launch_is_bit_identical(cuda, H, W, nshards, hole):
    """Temporal blocking (csrc/fib_fused.cuh): steps_per_launch=2 must reproduce the one-step
    kernels BIT FOR BIT -- unsharded (CUDA-graph replay and direct launches) and as row shards
    exchanging two halo rows of all four planes -- from a random state (non-trivial border ring),
    with a stimulus crossing the seams half way, without and with a phase field (two holes, one of
    them across a shard seam and one touching the border)."""
    from fib_tf_b200 import _capi
    from fib_tf_b200.sharding import partition_rows
    dt, diff = 0.1, 1.5
    rng = np.random.default_rng(H * 1000 + W)
    init = {'U': rng.uniform(0.0, 1.0, (H, W)), 'V': rng.uniform(0.0, 1.0, (H, W)),
            'W': rng.uniform(0.0, 1.0, (H, W)), 'S': rng.uniform(0.0, 1.0, (H, W))}
    init = {k: v.astype(np.float32) for k, v in init.items()}
    init['U'][H // 3:H // 2 + 1, W // 4:W // 2] = 0.95          # a depolarised patch

    phase = None
    if hole:
        yy, xx = np.mgrid[0:H, 0:W]
        phase = np.ones((H, W))
        for cy, cx, rad in ((H / 2.0, W / 2.0, max(min(H, W) / 6.0, 1.0)), (0.0, W * 0.8, max(min(H, W) / 8.0, 1.0))):
            phase *= 0.5 * (np.tanh(0.1 * (np.hypot(yy - cy, xx - cx) - rad) * 10.0) + 1.0)
        phase = np.maximum(phase, 1e-5).astype(np.float32)          # ionic.py:104-105

    def make(steps_per_launch, flags=0, parts=((0, 0),)):
        out = [_capi.Context(_capi.FENTON4V, H, W, dt, diff, flags=flags, row0=r0, rows=n,
                             steps_per_launch=steps_per_launch) for r0, n in parts]
        for s, (r0, n) in zip(out, parts):
            for v, a in init.items():
                s.set_state(v, a if n == 0 else a[r0:r0 + n])
            if phase is not None:
                s.set_phase(phase, 0)
        return out

    stim = ('U', 1, max(H - 1, 2), 1, max(W // 2, 2), 0.6, 0.0)
    ref, = make(1)
    fused, = make(2)
    direct, = make(2, flags=_capi.F_NO_GRAPH)
    parts = [p for p in partition_rows(H, nshards)]
    shards = make(2, flags=_capi.F_NO_GRAPH, parts=parts) if nshards > 1 else []
    for it in range(4):
        for c in (ref, fused, direct):
            c.step(_capi.OP_ODE, 1)
        if shards:
            _capi.step_group(shards, _capi.OP_ODE, 1)
        if it == 1:
            for c in [ref, fused, direct] + shards:
                c.stimulate(*stim)
    for v in ref.var_names:
        want = ref.get_state(v)
        assert np.isfinite(want).all()
        assert np.array_equal(fused.get_state(v), want), 'graph replay, %s' % v
        assert np.array_equal(direct.get_state(v), want), 'direct launches, %s' % v
        if shards:
            got = np.concatenate([s.get_state(v) for s in shards], axis=0)
            assert np.array_equal(got, want), 'row shards, %s' % v
    # probes and reductions read the fused layout correctly
    assert fused.probe('W', H // 2, W // 2) == ref.probe('W', H // 2, W // 2)
    a, b = fused.weighted_sum('V'), ref.weighted_sum('V')
    # (double-precision atomics: the summation order, hence the last bits, vary from run to run)
    assert abs(a[0] - b[0]) <= 1e-9 * abs(b[0]) and abs(a[1] - b[1]) <= 1e-9 * abs(b[1])
    for c in [ref, fused, direct] + shards:
        c.close()
