"""CPU: the activation-map contract of include/fib_b200.h (fib_activation_watch), restated in NumPy
(oracle/activation_np.py), against the float64 event rule the spiral statistics use (events() of
test_spiral_statistics.py) and against the conduction-velocity measurement of test_cv_table.py; and the
new entry points' argument checks without a GPU."""
import ctypes as C

import numpy as np
import pytest

import cv_common as cv
from fib_tf_b200 import _capi
from oracle import monodomain_np as onp
from oracle.activation_np import ActivationMapNP
from test_spiral_statistics import events


def _traces():
    """[samples, cells] fp32: one synthetic trace per column, each padded with its last value."""
    n = 1200
    i = np.arange(n)
    cols = [
        0.5 + 0.6 * np.sin(2 * np.pi * i / 37.3 + 0.3),                         # a sine
        np.r_[0.0, 0.25, 0.5, 0.75, 1.0, 0.5, 0.25, 0.0, 0.5, 0.5, 1.0],      # a ramp landing on the level
        np.full(20, 0.5),                                                      # flat at the level
        np.r_[1.0, 0.9, 0.4, 0.1, 0.0],                                        # a down-crossing first
        np.r_[0.0, 1.0, 1.0],                                                  # a crossing in iteration 1
        np.r_[0.0, np.nan, 1.0, 0.0, 1.0, np.nan, 0.0, 0.2, 0.9],              # NaN samples
        (i % 7) / 6.0 * 1.3 - 0.1,                                             # many beats (171 saw teeth)
        0.5 + 0.5 * np.cos(2 * np.pi * i / 5.1),                               # many fast beats
    ]
    out = np.empty((n, len(cols)), np.float32)
    for k, c in enumerate(cols):
        c = np.asarray(c, np.float32)
        out[:len(c), k] = c
        out[len(c):, k] = c[-1]
    return out


def _run(traces, up, down):
    m = ActivationMapNP(traces[0], up, down)
    for s in traces[1:]:
        m.update(s)
    return m


def _close(t32, t64):
    t32 = np.float64(t32)
    return abs(t32 - t64) <= 2 * np.spacing(np.float32(abs(t64)))


@pytest.mark.parametrize('up,down', [(0.5, 0.5), (0.625, 0.375), (0.25, 0.75)])
def test_oracle_maps_equal_the_float64_event_lists(up, down):
    tr = _traces()
    m = _run(tr, up, down)
    for k in range(tr.shape[1]):
        ups, _ = events(tr[:, k], up, 1.0)
        _, dns = events(tr[:, k], down, 1.0)
        assert m.count[k] == len(ups), (k, m.count[k], len(ups))
        for plane, want in ((m.first, ups[0] if len(ups) else None), (m.last, ups[-1] if len(ups) else None),
                            (m.prev, ups[-2] if len(ups) > 1 else None), (m.repol, dns[-1] if len(dns) else None)):
            if want is None:
                assert np.isnan(plane[k]), (k, plane[k])
            else:
                assert _close(plane[k], want), (k, plane[k], want)
    assert m.count[6] > 150 and m.count[7] > 200                     # the many-beat traces
    assert m.count[2] == 0 and np.isnan(m.repol[2])                  # flat at the level: no event


def test_oracle_edge_cases_by_hand():
    tr = _traces()
    m = _run(tr, 0.5, 0.5)
    # the ramp: up-crossings ending exactly on the level count (iterations 2 and 8 end at 0.5)
    assert m.first[1] == 2.0 and m.last[1] == 8.0 and m.prev[1] == 2.0 and m.count[1] == 2
    assert m.repol[1] == 5.0                                         # 0.5 -> 0.25: 0.5 >= 0.5 > 0.25
    # a down-crossing with no activation before it
    assert m.count[3] == 0 and np.isnan(m.first[3]) and 1.0 < m.repol[3] < 2.0
    # a crossing in iteration 1: t = 0 + 0.5 / 1
    assert m.first[4] == 0.5 and m.count[4] == 1
    # NaN samples: 0 -> nan and nan -> 1 produce nothing; 1 -> 0 (iteration 3) and 0 -> 1 (iteration 4) do
    assert m.count[5] == 2 and m.first[5] == 3.5 and m.repol[5] == 2.5


def _cv_pair(kind, diff):
    """measure_cv on the CPU oracle's strip, and the same run's CV from the oracle's LAST map."""
    width = 420 if kind == 'fenton4v' else 300
    c1, c2 = (150, 350) if kind == 'fenton4v' else (100, 240)
    level = 0.5 if kind == 'fenton4v' else -30.0
    m = onp.OracleModel(kind, cv.strip_config(diff, width))
    m.define()
    dt_iter = m.dt_per_step * 0.1
    amap = ActivationMapNP(m.pot(), level, level)

    def read_row(mm):
        p = mm.pot()
        amap.update(p)
        return p[2]
    got = cv.measure_cv(m, level, c1, c2, dt_iter, 4000, read_row)
    lat = amap.last[2].astype(np.float64) * dt_iter
    return got, (c2 - c1) / (lat[c2] - lat[c1])


@pytest.mark.parametrize('kind,diff', [('fenton4v', 1.0), ('br', 1.0)])
def test_cv_from_the_oracle_map_equals_measure_cv(kind, diff):
    got, from_map = _cv_pair(kind, diff)
    assert abs(from_map - got) <= 1e-6 * got, (from_map, got)


def test_activation_entry_points_reject_a_null_context():
    L = _capi.lib()
    buf = (C.c_float * 4)()
    assert L.fib_activation_watch(None, 0.5, 0.5) == -1
    assert L.fib_activation_stop(None) == -1
    assert L.fib_activation_get(None, _capi.ACT_LAST, buf, 4) == -1
    assert 'NULL' in L.fib_last_error().decode()
