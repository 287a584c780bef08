"""
fib_tf_b200.br -- drop-in for the reference's br.py: the modified 8-variable Beeler-Reuter model
(J Physiol 1977;268:177-210) with the reference's two optimisation flags:

  cheby  gate steady states / time constants from degree-8 polynomials fitted at define() time
         (br.py:207-252, 289-331); the 12x9 coefficient table is computed HERE on the host in
         fp64 exactly like the reference and handed to the kernel (FIB_TABLE_BR_CHEBY);
  skip   multi-rate: the slow gates xi, j, d, f advance once per 5 steps with 5*dt (br.py:96-107).
  cheby_strict (extra, optional)  the polynomial gates in the reference's exact operation order.

One run() iteration = 5 time steps = 5 launches of the fused kernel (one CUDA graph).
"""
import numpy as np
from numpy.polynomial.chebyshev import Chebyshev

from . import _capi
from .ionic import DeviceVar, IonicModel


class BeelerReuter(IonicModel):
    MODEL_ID = _capi.BR
    _pot_name = 'V'

    def __init__(self, props):
        super().__init__(props)
        self.min_v = -90.0    # mV
        self.max_v = 30.0     # mV
        self.depol = -84.6
        # alpha/beta coefficient rows (br.py:49-62); d and f rates are doubled (br.py:46-48)
        self.ab_coef = np.array(
            [[0.0005, 0.083, 50., 0.0, 0.0, 0.057, 1.0],        # ca_x1
             [0.0013, -0.06, 20., 0.0, 0.0, -0.04, 1.0],        # cb_x1
             [0.0000, 0.0, 47., -1.0, 47., -0.1, -1.0],         # ca_m
             [40., -0.056, 72., 0.0, 0.0, 0.0, 0.0],            # cb_m
             [0.126, -.25, 77., 0.0, 0.0, 0.0, 0.0],            # ca_h
             [1.7, 0.0, 22.5, 0.0, 0.0, -0.082, 1.0],           # cb_h
             [0.055, -.25, 78.0, 0.0, 0.0, -0.2, 1.0],          # ca_j
             [0.3, 0.0, 32., 0.0, 0.0, -0.1, 1.0],              # cb_j
             [2 * 0.095, -0.01, -5., 0.0, 0.0, -0.072, 1.0],    # ca_d
             [2 * 0.07, -0.017, 44., 0.0, 0.0, 0.05, 1.0],      # cb_d
             [2 * 0.012, -0.008, 28., 0.0, 0.0, 0.15, 1.0],     # ca_f
             [2 * 0.0065, -0.02, 30., 0.0, 0.0, -0.2, 1.0]],    # cb_f
            dtype=np.float32)

    def define(self, s1=True):
        """Initial state br.py:71-82; S1 = column 1 of V set to 10 mV."""
        ctx = self._create()
        init = {'V': -84.624, 'C': 1e-4, 'M': 0.01, 'H': 0.988, 'J': 0.975, 'D': 0.003,
                'F': 0.994, 'XI': 0.0001}
        for name, val in init.items():
            a = self._local_full(val)
            if s1 and name == 'V':
                a[:, 1] = 10.0
            ctx.set_state(name, a)

    def _create(self):
        """The context, table and handles of define(), without the initial state (define() and restore())."""
        IonicModel.define(self)
        flags = (_capi.F_CHEBY if self.cheby else 0) | (_capi.F_SKIP if self.skip else 0)
        # config['cheby_strict'] (optional, default False): evaluate the polynomial gates in the
        # reference's own fp32 operation order (br.py:215,289-301,327-331) instead of Horner's scheme;
        # slower, used to show how closely the reference's result is defined (DESIGN.md section 4)
        if self.cheby and self.__dict__.get('cheby_strict'):
            flags |= _capi.F_CHEBY_STRICT
        ctx = self._make_context(flags)
        if self.cheby:
            ctx.set_table(_capi.TABLE_BR_CHEBY, self.chebyshev_table())
        self.dt_per_step = ctx.dt_per_step      # 5 in both schedules (br.py:101,105)
        self._ode_op = _capi.OP_ODE
        self._State = {n: DeviceVar(self, n) for n in ctx.var_names}
        self._V = self._State['V']
        return ctx

    # ---- define()-time NumPy set-up, as in the reference -------------------------------------
    def calc_alpha_beta_np(self):
        """alpha and beta of the six gates sampled at 1001 voltages (br.py:275-287);
        columns: xi, m, h, j, d, f."""
        v = np.linspace(self.min_v, self.max_v, 1001)
        c = self.ab_coef
        x = np.outer(v, np.ones(c.shape[0]))
        y = ((c[:, 0] * np.exp(c[:, 1] * (x + c[:, 2])) + c[:, 3] * (x + c[:, 4])) /
             (np.exp(c[:, 5] * (x + c[:, 2])) + c[:, 6]))
        return v, y[..., ::2], y[..., 1::2]

    @staticmethod
    def monomial_basis(deg):
        """a[i, j] = coefficient of S_j = 2^(j-1) x^j in the Chebyshev polynomial T_i
        (br.py:317-324: T_i expanded in powers of x, column j divided by T_j's leading term)."""
        a = np.zeros([deg + 1, deg + 1], dtype=int)
        a[0, 0] = 1
        a[1, 1] = 1
        for i in range(2, deg + 1):
            a[i, 1:] += 2 * a[i - 1, :-1]
            a[i, :] -= a[i - 2, :]
        a //= np.diag(a)
        return a

    def chebyshev_table(self, deg=8):
        """float64 [12][deg+1]: row 2g = inf, 2g+1 = tau of gate g in (xi, m, h, j, d, f), as
        coefficients d_i of r = d_0 + sum d_i S_i (br.py:303-331)."""
        v, alpha, beta = self.calc_alpha_beta_np()
        basis = np.transpose(self.monomial_basis(deg))
        table = np.zeros([12, deg + 1])
        for g in range(6):
            total = alpha[:, g] + beta[:, g]
            table[2 * g] = np.matmul(basis, Chebyshev.fit(v, alpha[:, g] / total, deg).coef)
            table[2 * g + 1] = np.matmul(basis, Chebyshev.fit(v, 1.0 / total, deg).coef)
        return table

    def pot(self):
        return self._V

    def image(self):
        """V mapped to 0..1 (br.py:337-343)."""
        v = self._V.eval()
        return (v - self.min_v) / (self.max_v - self.min_v)


if __name__ == '__main__':
    config = {
        'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 0.809,
        'duration': 1000, 'skip': False, 'cheby': True, 'timeline': False,
        'timeline_name': 'timeline_br.json', 'save_graph': False
    }
    model = BeelerReuter(config)
    model.add_hole_to_phase_field(150, 200, 40)     # center=(150,200), radius=40
    model.define()
    model.add_pace_op('s2', 'luq', 10.0)
    im = None

    s2 = model.millisecond_to_step(300)     # 300 ms
    ds = model.millisecond_to_step(10)
    n = int(model.duration / 10.0)
    cube = np.zeros([n, model.height, model.width], dtype=np.float32)
    for i in model.run(im):
        if i == s2:
            model.fire_op('s2')
        if i % ds == 0:
            cube[i // ds, :, :] = model.image() * model.phase
    np.save('cube', cube)
