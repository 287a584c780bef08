"""
fib_tf_b200.fenton -- drop-in for the reference's fenton.py: the Cherry-Ehrlich-Nattel-Fenton
(4v) canine left-atrial model (Heart Rhythm 2007;4(12):1553-62).

Same class name, constructor, define(s1), pot(), image() and driver block as fenton.py:31-187.
The ten unrolled explicit-Euler steps of one run() iteration (fenton.py:133-138) are ten
launches of the fused sm_100a kernel (boundary + 9-point Laplacian + phase term + 4v reaction),
replayed as one CUDA graph.
"""
import os

import numpy as np

from . import _capi
from .ionic import DeviceVar, IonicModel


class Fenton4v(IonicModel):
    MODEL_ID = _capi.FENTON4V
    _pot_name = 'U'

    def __init__(self, props):
        IonicModel.__init__(self, props)
        self.min_v = 0.0
        self.max_v = 1.0
        self.depol = 0.0

    def define(self, s1=True):
        """Initial state U=0, V=W=1, S=0; S1 = column 1 of U set to 1 (fenton.py:116-123)."""
        ctx = self._create()
        init = {'U': 0.0, 'V': 1.0, 'W': 1.0, 'S': 0.0}
        for name, val in init.items():
            a = self._local_full(val)
            if s1 and name == 'U':
                a[:, 1] = 1.0
            ctx.set_state(name, a)

    def _create(self):
        """The context and handles of define(), without the initial state (define() and restore())."""
        IonicModel.define(self)
        self.steps_per_launch_used = self._steps_per_launch()
        ctx = self._make_context(steps_per_launch=self.steps_per_launch_used)
        self.dt_per_step = ctx.dt_per_step      # 10
        self._ode_op = _capi.OP_ODE
        self._State = {n: DeviceVar(self, n) for n in ctx.var_names}
        self._U = self._State['U']
        return ctx

    # grids from this many cells up run two time steps per launch by default: below it the state
    # (4 planes) is L2-resident and the one-step kernel is faster (2048^2: 242 vs 209 Gcell-steps/s);
    # above it the fused kernel wins (4096^2: 195 -> 261, 8192^2: 208 -> 306)
    FUSE_MIN_CELLS = 3072 * 3072
    # with a phase field the fused kernel runs one CTA per SM fewer (phi windows): 3072^2 is a tie
    # (175 vs 178), 4096^2 185 -> 204, 8192^2 198 -> 240
    FUSE_MIN_CELLS_PHASE = 4096 * 4096

    def _steps_per_launch(self):
        """Temporal blocking: two time steps per kernel launch (csrc/fib_fused.cuh), BIT-IDENTICAL
        to one step per launch.  Config key 'steps_per_launch' (1 or 2) or FIB_STEPS_PER_LAUNCH
        override the size-based default; it needs width % 4 == 0, otherwise one step per launch
        is used.  The choice depends on the global grid only (all replicas of a batched model), so every rank
        of a sharded run makes the same one."""
        want = self.__dict__.get('steps_per_launch')
        if want is None:
            want = os.environ.get('FIB_STEPS_PER_LAUNCH')
        if want is None:
            floor = self.FUSE_MIN_CELLS if self._phase_rows is None else self.FUSE_MIN_CELLS_PHASE
            want = 2 if self.height * self.width * self.replicas >= floor else 1
        able = self.width % 4 == 0 and \
            (self._nranks == 1 or self.height // self._nranks >= 2)
        return 2 if int(want) == 2 and able else 1

    def pot(self):
        return self._U

    def image(self):
        return self._U.eval()


if __name__ == '__main__':
    # the reference's driver (fenton.py:155-187): 512^2, hole, S1-S2 at 210 ms, a frame every 10 ms
    model = Fenton4v({'width': 512, 'height': 512, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5,
                      'duration': 1000, 'timeline': False, 'timeline_name': 'timeline_4v.json',
                      'save_graph': False})
    model.add_hole_to_phase_field(256, 256, 30)
    model.define()
    model.add_pace_op('s2', 'luq', 1.0)
    s2, every = model.millisecond_to_step(210), model.millisecond_to_step(10)
    cube = np.zeros([int(model.duration / 10.0), model.height, model.width], dtype=np.float32)
    for i in model.run(None):           # headless; pass a fib_tf_b200.screen.Screen to watch
        if i == s2:
            model.fire_op('s2')
        if i % every == 0:
            cube[i // every] = model.image() * model.phase
    np.save('cube', cube)
