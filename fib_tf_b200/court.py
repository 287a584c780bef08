"""
fib_tf_b200.court -- drop-in for the reference's court.py: the modified Courtemanche-Ramirez-
Nattel 1998 human atrial model (21 state variables, "chronic AF" remodelling on by default).

Multi-rate by driver convention, exactly like the reference (court.py:94-103, 615-617):
  * run()'s op advances only V, _Na_i_, _m_, _h_ with dt         -> kernel mode COURT_FAST
  * fire_op('slow') advances the other 17 states with 10*dt, evaluated on the CURRENT state
    (drivers fire it every 10th iteration)                        -> kernel mode COURT_SLOW
With config['lut']=True the 30 voltage-only intermediates come from the 150x30 table of
courtemanche.h (truncating lookup), read from a transposed copy [30][160] that stays L1-resident (see csrc/model_court.cuh for the shared-memory A/B).
"""
import numpy as np

from . import _capi
from .ionic import DeviceVar, IonicModel

# state names and resting values in the reference's creation order (court.py:57-78)
INITIAL_STATE = (
    ('V', -81.18), ('_Na_i_', 1.117e+01), ('_m_', 2.98e-3), ('_h_', 9.649e-1), ('_j_', 9.775e-1),
    ('_K_i_', 1.39e+02), ('_oa_', 3.043e-2), ('_oi_', 9.992e-1), ('_ua_', 4.966e-3),
    ('_ui_', 9.986e-1), ('_xr_', 3.296e-5), ('_xs_', 1.869e-2), ('_Ca_i_', 1.013e-4),
    ('_d_', 1.367e-4), ('_f_', 9.996e-1), ('_f_Ca_', 7.755e-1), ('_Ca_rel_', 1.488),
    ('_u_', 0.0), ('_v_', 1.0), ('_w_', 0.9992), ('_Ca_up_', 1.488))


class _HostValue:
    """.eval()-able holder of a small host array (the reference's Trend variable)."""

    def __init__(self, n):
        self.value = np.zeros([n], dtype=np.float32)

    def eval(self):
        return self.value.copy()


class Courtemanche(IonicModel):
    MODEL_ID = _capi.COURT
    _pot_name = 'V'
    _multirate = True

    def __init__(self, props):
        super().__init__(props)
        self.min_v = -100.0     # mV
        self.max_v = 50.0       # mV
        self.depol = -81.0      # mV
        self.chronic = True
        self.fast_states = ['V', '_Na_i_', '_m_', '_h_']

    def init_state_variable(self, state, name, value):
        if name in state:
            print('Warning! The state variable arlready exists')
        state[name] = self._local_full(value)

    def _initial_names(self):
        return INITIAL_STATE

    def _flags(self):
        f = 0 if self.chronic else _capi.F_NO_CHRONIC
        if self.__dict__.get('lut'):
            f |= _capi.F_LUT
        return f

    def define(self, s1=True, state=None):
        """Resting state (court.py:57-78) or a saved `state` dict (court.py:49-56, 623-626);
        S1 = columns 0..24 of V set to 20 mV."""
        ctx = self._create()
        if state is None:
            state = {}
            for name, val in self._initial_names():
                self.init_state_variable(state, name, val)
            if s1:
                state['V'][:, :25] = 20.0
        else:   # a full-grid dict saved by run(keep_state=True): take this shard's rows ([H, W] for every
            # replica of a batched model, or [replicas, H, W])
            state = {k: self._own_rows(v) for k, v in state.items()}
        missing = [n for n in ctx.var_names if n not in state]
        if missing:
            raise KeyError('state is missing %s' % missing)
        for name in ctx.var_names:
            ctx.set_state(name, state[name])

    def _create(self):
        """The context, LUT, ops and handles of define(), without the initial state (define() and restore())."""
        IonicModel.define(self)
        if list(self.fast_states) != ['V', '_Na_i_', '_m_', '_h_']:
            raise NotImplementedError('the fast/slow split is compiled into the kernels: '
                                      "fast_states must stay ['V', '_Na_i_', '_m_', '_h_']")
        ctx = self._make_context(self._flags())
        if self.__dict__.get('lut'):
            ctx.build_lut()
        self.dt_per_step = 1
        self._ode_op = _capi.OP_ODE
        self._ops['slow'] = ('call', lambda: ctx.step(_capi.OP_SLOW, 1))
        self._ops['trend'] = ('call', self._update_trend)
        self._State = {n: DeviceVar(self, n) for n in ctx.var_names}
        self._V = self._State['V']
        self._Trend = _HostValue(2)
        return ctx

    def _update_trend(self):
        """court.py:107-112: Trend := (V, _Na_i_) at [width//2, 20] (row index from `width`)."""
        r, c = self.width // 2, 20
        self._Trend.value[0] = self._probe('V', r, c)
        self._Trend.value[1] = self._probe('_Na_i_', r, c)

    def euler(self, g, Rate, dt):
        return g + Rate * dt

    def δt(self, name):
        """Step of a state variable: dt for the fast states, 10*dt otherwise (court.py:118-122)."""
        if name in self.fast_states:
            return self.dt
        return self.dt * 10

    def calc_inter(self, V, mod=np):
        """The 30 voltage-only intermediates (court.py:273-429) for scalar or array V, evaluated
        by the same device function the step kernels use (fib_court_inter)."""
        scalar = np.ndim(V) == 0
        v = np.atleast_1d(np.asarray(V, dtype=np.float32))
        q = self._inter_context().court_inter(v.ravel())
        out = {}
        for k, name in enumerate(_capi.INTER_NAMES[:30]):
            col = q[:, k].reshape(v.shape)
            out[name] = float(col[0]) if scalar else col
        return out

    def _inter_context(self):
        if self._ctx is not None:
            return self._ctx
        if getattr(self, '_aux_ctx', None) is None:     # calc_inter before define()
            self._aux_ctx = _capi.Context(self.MODEL_ID, 3, 3, self.dt, self.replica_diff[0])
        return self._aux_ctx

    def pot(self):
        return self._V

    def image(self):
        """V mapped to 0..1 (court.py:574-580)."""
        v = self._V.eval()
        return (v - self.min_v) / (self.max_v - self.min_v)


def cl_observer(i, cl):
    print('Observer: %d:\t%d' % (i, cl))


if __name__ == '__main__':
    config = {
        'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809,
        'duration': 20000, 'skip': False, 'cheby': True, 'timeline': False,
        'timeline_name': 'timeline_court.json', 'save_graph': False
    }
    m1 = Courtemanche(config)
    m1.add_hole_to_phase_field(256, 256, 30)
    m1.add_hole_to_phase_field(256, 256, 250, neg=True)
    m1.define()
    m1.add_pace_op('s2', 'luq', 10.0)
    m1.cl_observer = cl_observer
    im = None
    s2 = m1.millisecond_to_step(350)
    data = []
    for i in m1.run(im, keep_state=True, block=False):
        if i % 10 == 0:
            m1.fire_op('slow')
            m1.fire_op('trend')
            data.append(m1._Trend.eval())
        if i == s2:
            m1.fire_op('s2')

    m2 = Courtemanche(config)
    m2.add_hole_to_phase_field(256, 256, 100)
    m2.add_hole_to_phase_field(256, 256, 250, neg=True)
    m2.define(state=m1.state)
    m2.cl_observer = cl_observer
    for i in m2.run(im):
        if i % 10 == 0:
            m2.fire_op('slow')
            m2.fire_op('trend')
            data.append(m2._Trend.eval())
    np.savetxt('vol_na_2.dat', np.asarray(data))
