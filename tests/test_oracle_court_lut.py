"""CPU: the NumPy oracle's Courtemanche lookup-table flavour (oracle.monodomain_np court_lut_table /
court_lookup / court_solve(table=...)) and its chronic-off and no-clip switches.  No GPU and no built
library needed.

The table flavour is the exact cell with the 30 voltage-only intermediates read from row
clamp(int(fp32(V) + 100), 0, 149) of a [150, 30] table whose row k is calc_inter(k - 100)
(courtemanche.h:105-134, 354-357, 473-479).  These tests pin the column order to the header's
known-answer vector, the row rule at its edges, and show that the lookup is really used."""
import numpy as np
import pytest

from oracle import monodomain_np as onp
from test_oracle_cport import KAT_M50

F32 = np.float32


def test_table_row_50_is_the_reference_known_answer():
    """Row 50 (V = -50 mV) against calc_inter(-50) of the reference's own header, column by column:
    the column order comes from outside the project."""
    tab = onp.court_lut_table()
    assert tab.shape == (150, 30) and tab.dtype == np.float32
    for k, name in enumerate(onp.COURT_LUT_COLUMNS):
        assert np.isclose(tab[50, k], KAT_M50[k], rtol=6e-6, atol=5e-7), (k, name, tab[50, k], KAT_M50[k])


def test_table_rows_are_calc_inter_at_integer_voltages():
    tab = onp.court_lut_table()
    for k in (0, 1, 49, 50, 60, 99, 100, 110, 149):
        q = onp.court_inter(np.array([k - 100], np.float32))
        want = np.array([q[n][0] for n in onp.COURT_LUT_COLUMNS], np.float32)
        assert np.array_equal(tab[k], want), k


def test_device_binding_uses_the_same_column_order():
    from fib_tf_b200 import _capi            # imports without the shared library
    assert tuple(_capi.INTER_NAMES[:30]) == onp.COURT_LUT_COLUMNS
    assert tuple(_capi.INTER_NAMES[30:]) == ('us_infinity', 'tau_us')


def f32_next(x, direction):
    return np.nextafter(F32(x), F32(direction))


# planted voltage -> row of the truncating lookup (the sum V + 100 is rounded to fp32 first)
PLANTED = [
    (F32(-100.0), 0), (f32_next(-100.0, -np.inf), 0), (F32(-100.5), 0), (F32(-101.0), 0), (F32(-130.0), 0),
    (F32(49.0), 149), (f32_next(50.0, -np.inf), 149), (F32(50.0), 149), (F32(80.0), 149),
    (F32(-0.0), 100), (F32(-1e-6), 100), (F32(-4e-6), 99),
    (f32_next(-50.0, np.inf), 50), (f32_next(-50.0, -np.inf), 49),
    (F32(-50.0), 50), (F32(-50.5), 49), (F32(-49.5), 50), (F32(0.0), 100), (F32(0.999), 100),
]


def test_lookup_selects_the_planted_rows():
    V = np.array([v for v, _ in PLANTED], np.float32)
    rows = onp.court_lut_row(V)
    assert rows.tolist() == [r for _, r in PLANTED]
    # in real arithmetic -1e-6 + 100 is below 100: the fp32 sum is what the kernels truncate
    assert int(np.trunc(np.float64(F32(-1e-6)) + 100.0)) == 99
    tab = onp.court_lut_table()
    q = onp.court_lookup(V.reshape(1, -1), tab)
    for k, name in enumerate(onp.COURT_LUT_COLUMNS):
        assert q[name].shape == (1, V.size)
        assert np.array_equal(q[name][0], tab[[r for _, r in PLANTED], k]), name
    # a table with distinct rows: the value read IS the row
    marked = np.repeat(np.arange(150, dtype=np.float32)[:, None], 30, axis=1)
    marked += np.arange(30, dtype=np.float32)[None, :] / 100
    q = onp.court_lookup(V, marked)
    for k, name in enumerate(onp.COURT_LUT_COLUMNS):
        assert np.array_equal(q[name], np.float32([r + k / 100 for _, r in PLANTED])), name


def _planted_state(V, ultra_slow, rng):
    """Resting state with every other plane perturbed (factor 0.55 ... 1.45, gates in [1e-4, 0.9999]),
    V as given, one ring of SYMMETRIC padding so that enforce_boundary changes nothing."""
    H, W = V.shape
    st = onp.court_init(H, W, s1=False, ultra_slow=ultra_slow)
    gates = ('_m_', '_h_', '_j_', '_oa_', '_oi_', '_ua_', '_ui_', '_xr_', '_xs_', '_d_', '_f_', '_f_Ca_',
             '_u_', '_v_', '_w_', '_us_')
    for k in st:
        if k == 'V':
            continue
        st[k] = (st[k] * rng.uniform(0.55, 1.45, (H, W))).astype(np.float32)
        if k in gates:
            st[k] = np.clip(st[k], F32(1e-4), F32(0.9999))
    st['V'] = V.astype(np.float32)
    return {k: np.pad(a, 1, mode='symmetric') for k, a in st.items()}


SOLVES = [
    pytest.param(dict(multirate=True), id='court-fast-and-slow'),
    pytest.param(dict(multirate=False), id='court_ultra'),
    pytest.param(dict(multirate=False, ultra_slow=True), id='court_ultra-us'),
]


@pytest.mark.parametrize('chronic', [True, False])
@pytest.mark.parametrize('kw', SOLVES)
def test_lut_step_equals_exact_step_at_integer_voltages(kw, chronic):
    """Where V is an integer in [-100, 49] the table row IS calc_inter(V), so one step of the table
    flavour equals one step of the exact model bit for bit (court's fast op assigns V, _Na_i_, _m_,
    _h_ of this solve and its 'slow' op the other 17: all of them are compared).  At -50.5 mV the
    two must differ: the table flavour really reads the table."""
    rng = np.random.default_rng(11)
    us = bool(kw.get('ultra_slow'))
    V = (np.arange(150, dtype=np.float32) - 100).reshape(10, 15)
    S = _planted_state(V, us, rng)
    tab = onp.court_lut_table()
    with np.errstate(all='ignore'):
        exact = onp.court_solve(S, 0.1, 0.0, chronic=chronic, **kw)
        lut = onp.court_solve(S, 0.1, 0.0, chronic=chronic, table=tab, **kw)
    assert sorted(exact) == sorted(lut) and ('_us_' in exact) == us
    for k in exact:
        assert np.array_equal(exact[k], lut[k]), k
    S = _planted_state(np.full((10, 15), -50.5, np.float32), us, rng)
    with np.errstate(all='ignore'):
        exact = onp.court_solve(S, 0.1, 0.0, chronic=chronic, **kw)
        lut = onp.court_solve(S, 0.1, 0.0, chronic=chronic, table=tab, **kw)
    for k in ('V', '_m_', '_h_', '_j_', '_d_', '_xr_'):
        assert not np.array_equal(exact[k][1:-1, 1:-1], lut[k][1:-1, 1:-1]), k
    if us:      # the us gate is computed directly in both flavours
        assert np.array_equal(exact['_us_'], lut['_us_'])


@pytest.mark.parametrize('kw', SOLVES)
def test_chronic_and_clip_switches_change_what_they_should(kw):
    """chronic=False changes i_to, i_Kur, i_Ca_L (court.py:193-194,218) and nothing voltage-only;
    clip=False only changes gates that leave [1e-5, 0.99999]."""
    rng = np.random.default_rng(12)
    V = np.linspace(-90.0, 40.0, 12 * 9, dtype=np.float32).reshape(12, 9)
    S = _planted_state(V, bool(kw.get('ultra_slow')), rng)
    with np.errstate(all='ignore'):
        on = onp.court_solve(S, 0.1, 0.0, **kw)
        off = onp.court_solve(S, 0.1, 0.0, chronic=False, **kw)
        noclip = onp.court_solve(S, 0.1, 0.0, clip=False, **kw)
    for k in ('V', '_Ca_i_'):             # (K_i and Na_i move by less than an ulp in one step)
        assert not np.array_equal(on[k], off[k]), k
    for k in ('_m_', '_h_', '_d_', '_oa_'):           # gates: the current state's currents do not enter
        assert np.array_equal(on[k], off[k]), k
    for k in on:
        inside = (noclip[k] >= F32(1e-5)) & (noclip[k] <= F32(0.99999))
        assert np.array_equal(on[k][inside], noclip[k][inside]), k
    g = S['_m_'][:1, :1]
    assert onp.rush_larsen(g, F32(2.0), F32(0.01), 0.1)[0, 0] == F32(0.99999)
    assert onp.rush_larsen(g, F32(2.0), F32(0.01), 0.1, clip=False)[0, 0] > F32(1.5)


def test_oracle_model_reads_lut_and_chronic_from_the_config():
    cfg = {'width': 9, 'height': 7, 'dt': 0.1, 'diff': 0.0, 'ultra_slow': True}
    runs = {}
    for key, extra in (('exact', {}), ('lut', {'lut': True}), ('chronic_off', {'chronic': False}),
                       ('lut_table', {'lut': True})):
        m = onp.OracleModel('court_ultra', dict(cfg, **extra),
                            table=onp.court_lut_table() + 1 if key == 'lut_table' else None)
        m.define(s1=False)
        m.state['V'][...] = -50.5
        m.iterate()
        runs[key] = m.state
    assert not np.array_equal(runs['exact']['_m_'], runs['lut']['_m_'])
    assert not np.array_equal(runs['lut']['_m_'], runs['lut_table']['_m_'])       # the given table is used
    assert not np.array_equal(runs['exact']['V'], runs['chronic_off']['V'])
    assert np.array_equal(runs['exact']['_m_'], runs['chronic_off']['_m_'])
    # and the multi-rate model's 'slow' op takes the same switches
    for kind in ('court',):
        a, b = (onp.OracleModel(kind, dict(cfg, **e)) for e in ({}, {'lut': True, 'chronic': False}))
        for m in (a, b):
            m.define(s1=False)
            m.state['V'][...] = -50.5
            m.fire('slow')
        assert not np.array_equal(a.state['_j_'], b.state['_j_'])
        assert not np.array_equal(a.state['_Ca_i_'], b.state['_Ca_i_'])
