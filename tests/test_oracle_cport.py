"""CPU: (1) the plain-C/OpenMP port (bench.py's CPU baseline) against the golden fixtures;
(2) the compiled reference header oracle/_ref (courtemanche.h) against the known-answer vector
of SURVEY.md Appendix B.4 and against the NumPy oracle's calc_inter."""
import numpy as np
import pytest

from conftest import golden_names, load_fixture
from oracle import cpu_port
from oracle import monodomain_np as onp

PORTED = [n for n in golden_names() if n.startswith(('fenton_', 'br_')) and 'long' not in n]


@pytest.mark.parametrize('name', PORTED)
def test_c_port_matches_reference_fixture(name):
    meta, arr = load_fixture(name)

    def check(i, m):
        for v in meta['vars']:
            key = 's%d__%s' % (i, v)
            e = onp.rel_err(m.state[v], arr[key], onp.var_floor(meta['model'], v))
            assert e <= onp.parity_tolerance(meta, key), (name, key, e)

    onp.run_fixture(meta, check, model_factory=cpu_port.CPortModel)


# g++ 13.3 -O2 build of the reference's generate_table.cpp: calc_inter(V = -50), 30 columns
KAT_M50 = [0.006693, 0.960396, 0.345409, 0.711940, 387.911591, 0.995004, 0.268253, 0.021009,
           0.020188, 4.309348, 79.754211, 4.309348, 1464.123657, 253.195618, 200.473541, 0.097097,
           12.825628, 23.367565, 0.156622, 0.786152, 0.113842, 0.995673, 0.003978, 0.063673,
           0.005335, 0.720790, 0.010301, 102066.710938, 0.981871, 2.431505]
# courtemanche.h:105-134 column order -> names used by court.py's calc_inter dict
NAMES = onp.COURT_LUT_COLUMNS


def test_numpy_oracle_reproduces_the_reference_known_answer():
    """The NumPy oracle's calc_inter(V = -50) against the vector above, with nothing compiled: the two
    bars of the next test added (printing with %f, then oracle vs header)."""
    mine = onp.court_inter(np.array([-50.0], np.float32))
    assert np.allclose([float(mine[n][0]) for n in NAMES], KAT_M50, rtol=6e-6, atol=5e-7)


def test_reference_header_known_answer_and_numpy_oracle_agree():
    ref = cpu_port.court_ref()
    if ref is None:
        pytest.skip('oracle/_ref not built (no /root/reference here)')
    q = np.zeros(30, np.float32)
    ref.ref_calc_inter(-50.0, q)
    assert np.allclose(q, KAT_M50, rtol=2e-6, atol=5e-7)         # printed with %f: 6 decimals
    mine = onp.court_inter(np.array([-50.0], np.float32))
    for k, n in enumerate(NAMES):
        assert abs(float(mine[n][0]) - q[k]) <= 4e-6 * abs(q[k]), n
    # whole table: NumPy oracle vs the reference header on the LUT grid V = -100..49
    tab = np.zeros([150, 30], np.float32)
    ref.ref_init_table(tab)
    v = np.arange(150, dtype=np.float32) - 100
    mine = onp.court_inter(v)
    for k, n in enumerate(NAMES):
        col = np.asarray(mine[n], np.float64)
        ok = np.abs(col - tab[:, k]) <= 2e-5 * np.abs(tab[:, k]) + 1e-30
        # known, documented differences between court.py and courtemanche.h:
        #  * alpha_h / alpha_j are exactly 0 in the header and V*1e-20 in court.py above -40 mV
        #  * tau_d: the header switches to the limit formula AT V = -10 (courtemanche.h:179-182),
        #    court.py evaluates the regular formula at V + 10.0001 (court.py:306) -> 9e-4 apart
        if n in ('h_inf', 'j_inf'):
            ok |= (v >= -40.0) & (np.abs(col) < 1e-15)
        if n == 'tau_d':
            ok |= (v == -10.0) & (np.abs(col - tab[:, k]) <= 2e-3 * tab[:, k])
        assert ok.all(), (n, np.where(~ok)[0][:5])
