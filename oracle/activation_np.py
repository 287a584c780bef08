"""The activation-map contract of include/fib_b200.h (fib_activation_watch) restated in NumPy fp32.

    m = ActivationMapNP(s0, up, down)      # s0: the plane when the map is armed
    m.update(s1); m.update(s2); ...        # the plane after each ODE iteration
    m.first, m.last, m.prev, m.repol, m.count

Times are in iterations since arming.  In iteration k (a = s[k-1], b = s[k]):
    activation      a < up <= b      t = (k-1) + (up - a) / (b - a)
    repolarisation  a >= down > b    t = (k-1) + (a - down) / (a - b)
NumPy rounds every fp32 operation once, like the device's __fsub_rn / __fdiv_rn / __fadd_rn, so the planes
equal the device's bit for bit.  Test-only: the product never imports this module.
"""
import numpy as np

F32 = np.float32


class ActivationMapNP:
    def __init__(self, s0, up, down):
        self.prev_sample = np.array(s0, dtype=F32, copy=True)
        self.up, self.down = F32(up), F32(down)
        shape = self.prev_sample.shape
        self.first = np.full(shape, np.nan, F32)
        self.last = np.full(shape, np.nan, F32)
        self.prev = np.full(shape, np.nan, F32)
        self.repol = np.full(shape, np.nan, F32)
        self.count = np.zeros(shape, F32)
        self.k = 0                     # samples taken since arming = k - 1 of the next one

    def planes(self):
        """The five maps in fib_act_map order (FIRST, LAST, PREV, REPOL, COUNT)."""
        return [self.first, self.last, self.prev, self.repol, self.count]

    def update(self, sample):
        a, b = self.prev_sample, np.asarray(sample, dtype=F32)
        assert b.shape == a.shape
        k1 = F32(self.k)
        with np.errstate(invalid='ignore', divide='ignore', over='ignore'):
            act = (a < self.up) & (self.up <= b)
            rep = (a >= self.down) & (self.down > b)
            t_act = k1 + (self.up - a) / (b - a)
            t_rep = k1 + (a - self.down) / (a - b)
        t_act, t_rep = t_act.astype(F32), t_rep.astype(F32)
        self.first = np.where(act & np.isnan(self.first), t_act, self.first)
        self.prev = np.where(act, self.last, self.prev)
        self.last = np.where(act, t_act, self.last)
        self.count = np.where(act, self.count + F32(1), self.count).astype(F32)
        self.repol = np.where(rep, t_rep, self.repol)
        self.prev_sample = b.copy()
        self.k += 1
