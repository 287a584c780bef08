"""Adapter that lets oracle.monodomain_np.run_fixture() drive the PRODUCT (fib_tf_b200 models,
i.e. the CUDA kernels through the C ABI) with the same schedule as the golden fixtures."""
from fib_tf_b200.br import BeelerReuter
from fib_tf_b200.court import Courtemanche
from fib_tf_b200.court_ultra import Courtemanche as CourtemancheUltra
from fib_tf_b200.fenton import Fenton4v

CLASSES = {'fenton4v': Fenton4v, 'br': BeelerReuter, 'court': Courtemanche,
           'court_ultra': CourtemancheUltra}


class _StateView:
    def __init__(self, model):
        self._m = model

    def __getitem__(self, name):
        return self._m._State[name].eval()


class CudaModel:
    def __init__(self, kind, config, **extra):
        cfg = dict(config)
        cfg.update(extra)
        self.kind = kind
        self.m = CLASSES[kind](cfg)
        if kind in ('court', 'court_ultra'):
            # court.py sets `chronic` in __init__ (the config cannot reach it); define() reads it
            self.m.chronic = bool(cfg.get('chronic', True))
        self.state = _StateView(self.m)

    def add_hole(self, x, y, radius, neg=False):
        self.m.add_hole_to_phase_field(x, y, radius, neg)

    def define(self, s1=True, state=None):
        if state is not None:
            self.m.define(s1, state)
        else:
            self.m.define(s1)

    def add_pace(self, name, loc, v):
        self.m.add_pace_op(name, loc, v)

    def fire(self, name):
        self.m.fire_op(name)

    def iterate(self):
        self.m._ctx.step(self.m.ode_op(0), 1)

    def pot(self):
        return self.m.pot().eval()

    def close(self):
        self.m.close()


from oracle.monodomain_np import rel_err, var_floor  # noqa: E402,F401  (re-exported)
