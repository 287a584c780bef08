"""
fib_tf_b200.court_ultra -- drop-in for the reference's court_ultra.py: the Courtemanche model
with ALL states advanced every step with dt (court_ultra.py:107-111, 127-128; fire_op('slow')
is an empty op) and, with config['ultra_slow']=True, a 22nd state `_us_`: the ultra-slow Na
inactivation gate that scales i_Na (court_ultra.py:81-82, 198-199, 221-222, 445-450).
Exposes `_Inter[name].eval()` like the reference (court_ultra.py:114, 476-480).
"""
from functools import partial

import numpy as np

from . import _capi
from .court import INITIAL_STATE, Courtemanche as _MultiRate


class _InterVar:
    def __init__(self, model, col):
        self._model, self._col = model, col

    def eval(self):
        m = self._model
        v = m._ctx.get_state('V')
        q = m._ctx.court_inter(v.ravel())[:, self._col].reshape(v.shape)
        return m._gather(q)


class Courtemanche(_MultiRate):
    MODEL_ID = _capi.COURT_ULTRA
    _multirate = False

    def _initial_names(self):
        if self.ultra_slow:
            return INITIAL_STATE + (('_us_', 0.72),)    # steady state at 500 ms
        return INITIAL_STATE

    def _flags(self):
        return _MultiRate._flags(self) | (_capi.F_ULTRA_SLOW if self.ultra_slow else 0)

    def _create(self):
        ctx = _MultiRate._create(self)
        self._ops['slow'] = ('call', lambda: None)      # court_ultra.py:108: empty group
        self._Inter = {name: _InterVar(self, k) for k, name in enumerate(_capi.INTER_NAMES)}
        return ctx

    def _update_trend(self):
        """court_ultra.py:117-120: only Trend[0] := V[width//2, height//8]."""
        self._Trend.value[0] = self._probe('V', self.width // 2, self.height // 8)

    def δt(self, name):
        return self.dt

    def calc_inter(self, V, mod=np):
        out = _MultiRate.calc_inter(self, V, mod)
        scalar = np.ndim(V) == 0
        v = np.atleast_1d(np.asarray(V, dtype=np.float32))
        q = self._inter_context().court_inter(v.ravel())
        for k in (30, 31):
            col = q[:, k].reshape(v.shape)
            out[_capi.INTER_NAMES[k]] = float(col[0]) if scalar else col
        return out


def cl_observer(m, cyclelengths, i0, i, cl):
    """court_ultra.py:465-486, with the phase-weighted means reduced on the device."""
    def mean(name):
        swx, sw = m._ctx.weighted_sum(name)
        return swx / sw
    row = [i0 + i, cl, mean('_Na_i_'), mean('_f_Ca_')]
    if m.ultra_slow:
        w = m.phase if m.phase is not None else None
        row += [mean('_us_'), float(np.average(m._Inter['us_infinity'].eval(), weights=w)),
                float(np.average(m._Inter['tau_us'].eval(), weights=w))]
    cyclelengths.append(row)
    print('\t'.join('%.5g' % x for x in row))


def run_small(config, im, cyclelengths, radius=50, i0=0):
    m = Courtemanche(config)
    m.add_hole_to_phase_field(m.width // 2, m.height // 2, radius)
    m.add_hole_to_phase_field(m.width // 2, m.height // 2, m.width // 2 - 6, neg=True)
    m.define()
    m.add_pace_op('s2', 'luq', 10.0)
    m.cl_observer = partial(cl_observer, m, cyclelengths, i0)
    s2 = m.millisecond_to_step(300)
    for i in m.run(im, keep_state=True, block=False):
        if i % 10 == 0:
            m.fire_op('slow')
        if i == s2:
            m.fire_op('s2')
        if i % 5000 == 0:
            # rho = np.sum(image[phase > 1e-3] < 0.2) / np.sum(phase > 1e-3), cutoff -55 mV
            # (court_ultra.py:504-509), as a threshold count on the device
            print('rho = %.4f' % m.excitable_fraction(0.2, 1e-3))
    np.save('state_small', m.state)
    return m.state


def run_large(config, im, cyclelengths, radius, i0=0):
    m = Courtemanche(config)
    m.add_hole_to_phase_field(m.width // 2, m.height // 2, radius)
    state = np.load('state_small.npy', allow_pickle=True).item(0)
    m.define(state=state)
    m.cl_observer = partial(cl_observer, m, cyclelengths, i0)
    for i in m.run(im, keep_state=True, block=False):
        if i % 10 == 0:
            m.fire_op('slow')
    np.save('state_large', m.state)
    return m.state


if __name__ == '__main__':
    config = {
        'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5,
        'duration': 10000, 'skip': False, 'cheby': True, 'timeline': False,
        'timeline_name': 'timeline_court.json', 'save_graph': False, 'ultra_slow': False
    }
    cyclelengths = []
    run_small(config, None, cyclelengths, radius=10)
