"""The arithmetic layer (fib_tf_b200/csrc/fib_math.cuh) and the voltage-only intermediates built on it,
function by function against float64.

tests/csrc/unit_harness.cu is a test-only library that includes the product headers unchanged and
evaluates their device functions elementwise over host arrays, as T = float and as packed T = f2 pairs.
It is compiled here with the library's own nvcc flags (fib_tf_b200.build.NVCC_FLAGS, -fmad=false) and
anchored to libfibb200.so: its court_inter_dev<true, false, float> and rush_larsen equal the library's
fib_court_inter and fib_op_rush_larsen bit for bit.

  * the SFU-based primitives (m_exp, m_exp_affine, m_expm1, m_expm1_neg, m_rcp, m_div, m_log, m_sqrt,
    m_half_1p_tanh) in ulps of the correctly rounded result, over the argument ranges of their call sites,
    log-spaced over the whole fp32 range, and at their edges (switches, overflow, underflow, +-0,
    subnormals, +-inf, NaN);
  * the packed-pair vocabulary: every operation on f2 equals the scalar one lane for lane;
  * court_inter_dev<US, RATES> (the direct Courtemanche kernels use RATES = true, where the tau slots hold
    1/tau and several rates are formed over a common denominator) against court_inter in float64,
    including the -40 mV switch, the alpha_m guard and the removable singularities, and independent of
    what the other lanes of the warp compute;
  * one update of the trimmed exact Beeler-Reuter gates (br_gates_exact) against Rush-Larsen in float64,
    br_inf_rate_exact against float64, and the Horner evaluation of the Chebyshev gates (br_poly8)
    against the reference's left-to-right sum.

Each GPU test runs once and prints what it measured (pytest -s); the numbers in the docstrings were
measured on a B200."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import monodomain_np as onp

F32, F64, U32 = np.float32, np.float64, np.uint32
FLT_MIN = F64(np.finfo(F32).tiny)
FLT_MAX = F32(np.finfo(F32).max)
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HARNESS_SRC = os.path.join(HERE, 'csrc', 'unit_harness.cu')

gpu = pytest.mark.gpu


def compile_harness(out_dir):
    """nvcc with the library's flags -> <out_dir>/libunit_harness.so (needs no GPU)."""
    from fib_tf_b200 import build
    out = os.path.join(str(out_dir), 'libunit_harness.so')
    subprocess.check_call([os.environ.get('NVCC', 'nvcc')] + build.NVCC_FLAGS +
                          ['-I', os.path.join(ROOT, 'fib_tf_b200', 'csrc'), '-o', out, HARNESS_SRC])
    return out


def test_harness_compiles_for_sm100a(tmp_path):
    """A header change that breaks the harness is caught without a GPU."""
    assert os.path.getsize(compile_harness(tmp_path)) > 0


# --------------------------------------------------------------------------------------------------
# the harness
# --------------------------------------------------------------------------------------------------
UNARY = ('exp', 'expm1', 'expm1_neg', 'rcp', 'log', 'sqrt', 'half_1p_tanh', 'neg', 'abs')
BINARY = ('add', 'sub', 'mul', 'div', 'min', 'max', 'sel_lt', 'sel_gt')


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f32(a):
    return np.ascontiguousarray(a, dtype=F32)


class Harness:
    def __init__(self, path):
        L = self.L = C.CDLL(path)
        P, N, I, F = C.c_void_p, C.c_size_t, C.c_int, C.c_float
        for name, args in (('ut_unary', [I, I, P, N, P]), ('ut_binary', [I, I, P, P, N, P]),
                           ('ut_fma', [I, P, P, P, N, P]), ('ut_exp_affine', [I, P, N, F, F, P]),
                           ('ut_court_inter', [I, I, I, P, N, P]), ('ut_rush_larsen', [I, P, P, P, N, F, P]),
                           ('ut_br_gates_exact', [I, P, P, N, F, F, P]), ('ut_br_inf_rate_exact', [P, N, P]),
                           ('ut_br_poly8', [I, P, P, N, P])):
            getattr(L, name).argtypes = args
            getattr(L, name).restype = I

    @staticmethod
    def _check(rc):
        assert rc == 0, 'unit_harness call failed (%d)' % rc

    def unary(self, fn, x, packed=False):
        x = _f32(x)
        out = np.empty_like(x)
        self._check(self.L.ut_unary(UNARY.index(fn), int(packed), _p(x), x.size, _p(out)))
        return out

    def binary(self, fn, x, y, packed=False):
        x, y = _f32(x), _f32(y)
        out = np.empty_like(x)
        self._check(self.L.ut_binary(BINARY.index(fn), int(packed), _p(x), _p(y), x.size, _p(out)))
        return out

    def fma(self, x, y, z, packed=False):
        x, y, z = _f32(x), _f32(y), _f32(z)
        out = np.empty_like(x)
        self._check(self.L.ut_fma(int(packed), _p(x), _p(y), _p(z), x.size, _p(out)))
        return out

    def exp_affine(self, x, c, add, packed=False):
        x = _f32(x)
        out = np.empty_like(x)
        self._check(self.L.ut_exp_affine(int(packed), _p(x), x.size, float(c), float(add), _p(out)))
        return out

    def court_inter(self, V, us, rates, packed=False):
        V = _f32(V)
        out = np.empty((V.size, 32), F32)
        self._check(self.L.ut_court_inter(int(us), int(rates), int(packed), _p(V), V.size, _p(out)))
        return out

    def rush_larsen(self, g, g_inf, tau, neg_dt, packed=False):
        g, gi, t = _f32(g), _f32(g_inf), _f32(tau)
        out = np.empty_like(g)
        self._check(self.L.ut_rush_larsen(int(packed), _p(g), _p(gi), _p(t), g.size, float(neg_dt), _p(out)))
        return out

    def br_gates_exact(self, V, s, neg_dt, neg_dt_slow, packed=False):
        V, s = _f32(V), _f32(s)
        out = np.empty_like(s)
        self._check(self.L.ut_br_gates_exact(int(packed), _p(V), _p(s), V.size, float(neg_dt), float(neg_dt_slow),
                                             _p(out)))
        return out

    def br_inf_rate_exact(self, V):
        V = _f32(V)
        out = np.empty((V.size, 12), F32)
        self._check(self.L.ut_br_inf_rate_exact(_p(V), V.size, _p(out)))
        return out

    def br_poly8(self, c, x, packed=False):
        c, x = _f32(c), _f32(x)
        out = np.empty_like(x)
        self._check(self.L.ut_br_poly8(int(packed), _p(c), _p(x), x.size, _p(out)))
        return out


@pytest.fixture(scope='module')
def ut(cuda_device, tmp_path_factory):
    return Harness(compile_harness(tmp_path_factory.mktemp('unit_harness')))


# --------------------------------------------------------------------------------------------------
# helpers
# --------------------------------------------------------------------------------------------------
def ulps_around(points, k=16):
    """Every fp32 point and the 2k fp32 values within k ulps of it."""
    p = _f32(points)
    out, up, dn = [p], p.copy(), p.copy()
    for _ in range(k):
        up = np.nextafter(up, F32(np.inf))
        dn = np.nextafter(dn, F32(-np.inf))
        out += [up, dn]
    return np.concatenate(out)


def same_bits(a, b):
    """Bit-identical, except that any NaN matches any NaN (the payload is not compared)."""
    a, b = _f32(a), _f32(b)
    return (a.view(U32) == b.view(U32)) | (np.isnan(a) & np.isnan(b))


def ulp_error(got, ref):
    """|got - ref| in ulps of fp32(ref), where fp32(ref) is finite and normal (NaN elsewhere)."""
    ref = np.asarray(ref, F64)
    r32 = np.abs(ref).astype(F32)
    ok = np.isfinite(r32) & (r32 >= FLT_MIN)
    err = np.full(ref.shape, np.nan)
    err[ok] = np.abs(got[ok].astype(F64) - ref[ok]) / np.spacing(r32[ok]).astype(F64)
    return err


def pairs_shuffled(x, seed):
    """x in a seeded random order, padded to an even length: the pairs of the packed flavour mix values
    from everywhere in x."""
    x = np.random.default_rng(seed).permutation(_f32(x))
    return x if x.size % 2 == 0 else np.append(x, x[0])


def log_sweep(n=400001, lo=2.0 ** -149, hi=FLT_MAX):
    """Both signs, log-spaced from the smallest subnormal to FLT_MAX."""
    m = np.geomspace(lo, F64(hi), n).astype(F32)
    return np.concatenate([m, -m])


EDGES = np.float32([0.0, -0.0, 1e-45, -1e-45, 1e-40, -1e-40, FLT_MIN, -FLT_MIN, 1.0, -1.0, FLT_MAX, -FLT_MAX,
                    np.inf, -np.inf, np.nan])


# --------------------------------------------------------------------------------------------------
# the anchor: the harness compiles these functions the way the library does
# --------------------------------------------------------------------------------------------------
def court_voltages():
    """~2^20 fp32 voltages in [-120, 80] mV, every integer and half-integer, and +-16 ulps around -40,
    the alpha_m guard (-47.131, -47.129), the six removable singularities (5 voltages) and the twelve
    voltages where a fix-up argument y of court_inter_dev has |y| = 0.03."""
    grid = np.linspace(-120.0, 80.0, 1 << 20).astype(F32)
    halves = (np.arange(-240, 161) * 0.5).astype(F32)
    return np.unique(np.concatenate([grid, halves, ulps_around(COURT_SPECIAL)]))


# (centre, |dy/dV|) of the six fix-up arguments y_k of court_inter_dev, fp32 scales as in the header
_Y = ((-10.0001, 1.0 / 6.24), (7.9, 0.2), (-14.1, 0.2), (3.3328, 1.0 / 5.1237), (19.9, 1.0 / 17.0), (19.9, 1.0 / 9.0))
SINGULAR_MV = (-10.0001, 7.9, -14.1, 3.3328, 19.9)        # tau_d, tau_w, alpha_xr, beta_xr, alpha/beta_xs
COURT_SINGULAR = np.float32(SINGULAR_MV)
COURT_Y003 = np.float32([c + s * 0.03 / F64(F32(k)) for c, k in _Y for s in (-1, 1)])
COURT_SPECIAL = np.concatenate([np.float32([-40.0, -47.131, -47.129]), COURT_SINGULAR, COURT_Y003])


def rl_edge_inputs():
    """Rush-Larsen inputs at the edges of m_expm1_neg's argument x = -dt/tau (dt = 0.1): tau < 0,
    tau -> 0+, tau = +-0, +-inf, very large tau, |dt/tau| straddling 0.125, and g == g_inf with an
    infinite exponent.  Returns (g, g_inf, tau) as fp32 arrays of one shape."""
    rng = np.random.default_rng(5)
    taus = np.concatenate([
        -np.geomspace(1e-4, 1e4, 60), np.geomspace(1e-30, 1e-3, 40), [1e-40, 1e-45, 0.0, -0.0, -1e-40],
        [np.inf, -np.inf, 1e30, 3e38, -3e38, 1e9], ulps_around([0.8, -0.8], 16)]).astype(F32)
    g = rng.uniform(1e-3, 0.998, (taus.size, 4)).astype(F32)
    gi = rng.uniform(0.0, 1.0, (taus.size, 4)).astype(F32)
    gi[:, 0] = g[:, 0]                      # g == g_inf: 0 * inf = NaN where the exponent is infinite
    return g.ravel(), gi.ravel(), np.repeat(taus, 4)


@gpu
def test_harness_matches_the_library_bit_for_bit(ut):
    """court_inter_dev<true, false, float> against fib_court_inter on the dense voltage sweep, rush_larsen
    against fib_op_rush_larsen on the edge inputs: the harness compiles these functions as the library does."""
    from fib_tf_b200 import _capi
    V = court_voltages()
    ctx = _capi.Context(_capi.COURT_ULTRA, 3, 3, 0.1, 0.0)
    lib = ctx.court_inter(V)
    ctx.close()
    assert same_bits(ut.court_inter(V, us=True, rates=False), lib).all()
    g, gi, tau = rl_edge_inputs()
    assert same_bits(ut.rush_larsen(g, gi, tau, F32(-0.1)), _capi.op_rush_larsen(g, gi, tau, 0.1)).all()


# --------------------------------------------------------------------------------------------------
# (a) the primitives against float64
# --------------------------------------------------------------------------------------------------
def _ref64(fn, x):
    x = np.asarray(x, F64)
    with np.errstate(all='ignore'):
        if fn == 'exp':
            return np.exp(x)
        if fn in ('expm1', 'expm1_neg'):
            return np.expm1(x)
        if fn == 'rcp':
            return 1.0 / x
        if fn == 'log':
            return np.log(x)
        if fn == 'sqrt':
            return np.sqrt(x)
        if fn == 'half_1p_tanh':
            return 1.0 / (1.0 + np.exp(-2.0 * x))       # = 0.5 (1 + tanh x), without the cancellation
    raise ValueError(fn)


# the overflow / underflow thresholds of e^x in fp32: ln(FLT_MAX), ln(FLT_MIN), ln(2^-150)
EXP_EDGES = np.float32([88.72283935546875, -87.33654475055310898657, -103.97207708399179])


def straddle(points, k=8):
    """Pairs (p - i ulp, p + i ulp), i = 1 ... k, flattened: the two lanes of each pair sit on opposite
    sides of p."""
    up, dn, out = _f32(points), _f32(points), []
    for _ in range(k):
        up, dn = np.nextafter(up, F32(np.inf)), np.nextafter(dn, F32(-np.inf))
        out.append(np.stack([dn, up], -1))
    return np.concatenate(out).ravel()



# Per function: the inputs (dense over the arguments the call sites form, the log sweep, the edges) and
# the regions with their bars in ulps of fp32(ref).  A region's mask sees (x, ref).
PRIMITIVES = {
    # every exponent the models form for V in [-120, 80] mV lies in [-60, 60] ((V + 79.23) * 0.311 and
    # 0.35 V of the Courtemanche j and h gates are the widest); valid for |x| <= 2^127 (below)
    'exp': (lambda: np.concatenate([np.linspace(-60, 60, 1 << 18), log_sweep(hi=2.0 ** 24),
                                    ulps_around(EXP_EDGES, 64)]),
            [('|x| <= 2^24', lambda x, r: np.abs(x) <= 2.0 ** 24, 3.0)]),
    # x = -dt/tau of the Rush-Larsen factor (any sign: tau < 0 happens), |y| < 0.03 of the
    # Courtemanche fix-up, c5 (v + c2) of the BR alpha_m
    'expm1': (lambda: np.concatenate([np.linspace(-2, 2, 1 << 18), log_sweep(hi=2.0 ** 24),
                                      ulps_around([0.125, -0.125, 0.03, -0.03], 16), ulps_around(EXP_EDGES, 64)]),
              [('|x| < 0.125 (polynomial)', lambda x, r: np.abs(x) < 0.125, 2.0),
               ('|x| >= 0.125', lambda x, r: np.abs(x) >= 0.125, 13.0)]),
    'expm1_neg': (lambda: np.concatenate([np.linspace(-2, 2, 1 << 18), log_sweep(),
                                          ulps_around([0.125, -0.125], 16), ulps_around(EXP_EDGES, 64)]),
                  [('|x| < 0.125 (polynomial)', lambda x, r: np.abs(x) < 0.125, 2.0),
                   ('x <= -0.125', lambda x, r: x <= -0.125, 13.0),
                   ('0.125 <= x <= 1', lambda x, r: (x >= 0.125) & (x <= 1.0), 10.0),
                   # uncompensated: fl(x log2e) carries a relative error of up to |x| 2^-24 into e^x
                   ('x > 1, in units of 8 + x', lambda x, r: x > 1.0, lambda x: 8.0 + x)]),
    'rcp': (lambda: np.concatenate([log_sweep(), np.linspace(0.5, 4.0, 1 << 16)]),
            [('normal x, normal 1/x', lambda x, r: (np.abs(x) >= FLT_MIN) & (np.abs(r) >= FLT_MIN), 1.0)]),
    # E_K, E_Na, E_Ca: log of 5.4 / K_i ~ 0.04, 140 / Na_i ~ 13, 1.8 / Ca_i ~ 1e4; BR log(C), C ~ 1e-7
    'log': (lambda: np.concatenate([np.geomspace(1e-9, 1e6, 1 << 18), log_sweep()[:400001],
                                    ulps_around([1.0], 64)]),
            [('x outside [0.5, 2]', lambda x, r: ((x < 0.5) | (x > 2.0)) & (x >= FLT_MIN), 3.5)]),
    # xs_inf = sqrt of a sigmoid, i_NaK: sqrt((10 / Na_i)^3)
    'sqrt': (lambda: np.concatenate([np.linspace(0, 2, 1 << 18), log_sweep()[:400001]]),
             [('normal x', lambda x, r: x >= FLT_MIN, 1.0)]),
    # the Fenton 4v sigmoids: (U - b) / c and k (U - u_csi), U in [0, 1.6]
    'half_1p_tanh': (lambda: np.concatenate([np.linspace(-20, 20, 1 << 18), log_sweep(hi=2.0 ** 23)]),
                     [('|z| <= 2^23', lambda x, r: np.abs(x) <= 2.0 ** 23, 4.5)]),
}

# (input, output) pairs the comments of fib_math.cuh state, beyond the ulp bars; NaN == NaN here.
# m_exp and what is built on it (m_expm1, m_exp_affine, m_half_1p_tanh) compute r = fma(x, log2e, -t)
# with t = fl(x log2e): for x = +-inf that is inf - inf = NaN, so they return NaN (no call site forms
# an infinite exponent from finite state; m_expm1_neg has no such step and returns -1 / +inf).
SPECIALS = {
    'exp': [(0.0, 1.0), (-0.0, 1.0), (1e-40, 1.0), (-1e-40, 1.0), (89.0, np.inf), (1e30, np.inf), (-88.0, 0.0),
            (-1e30, 0.0), (np.inf, np.nan), (-np.inf, np.nan), (np.nan, np.nan)],
    'expm1': [(0.0, 0.0), (-0.0, 0.0), (1e-40, 1e-40), (89.0, np.inf), (-1e30, -1.0), (np.inf, np.nan),
              (-np.inf, np.nan), (np.nan, np.nan)],
    'expm1_neg': [(0.0, 0.0), (-0.0, 0.0), (89.0, np.inf), (-1e30, -1.0), (-FLT_MAX, -1.0), (np.inf, np.inf),
                  (-np.inf, -1.0), (np.nan, np.nan)],
    'rcp': [(0.0, np.inf), (-0.0, -np.inf), (1e-40, np.inf), (-1e-40, -np.inf), (np.inf, 0.0), (-np.inf, -0.0),
            (3e38, 0.0), (np.nan, np.nan)],
    'log': [(1.0, 0.0), (0.0, -np.inf), (1e-40, -np.inf), (np.inf, np.inf), (-1.0, np.nan), (np.nan, np.nan)],
    'sqrt': [(0.0, 0.0), (1e-40, 0.0), (np.inf, np.inf), (-1.0, np.nan), (np.nan, np.nan)],
    'half_1p_tanh': [(0.0, 0.5), (50.0, 1.0), (-50.0, 0.0), (np.inf, np.nan), (-np.inf, np.nan), (np.nan, np.nan)],
}


def check_specials(got, cases):
    x = np.float32([c[0] for c in cases])
    want = np.float32([c[1] for c in cases])
    bad = ~((got == want) | (np.isnan(got) & np.isnan(want)))
    assert not bad.any(), ['%r -> %r (want %r)' % (float(a), float(b), float(c))
                           for a, b, c in zip(x[bad], got[bad], want[bad])]


def worst_by_region(got, x, ref, regions):
    """{region: worst ulp error}, plus the cases where fp32(ref) is not finite and normal: overflow must
    give +-inf, underflow an |error| <= FLT_MIN (the SFU flushes subnormal results to zero)."""
    err = ulp_error(got, ref)
    out = {}
    for label, mask, bar in regions:
        m = mask(x.astype(F64), ref) & np.isfinite(err)
        e = err[m] / bar(x[m].astype(F64)) if callable(bar) else err[m]
        out[label] = float(e.max()) if m.any() else 0.0
    return out


@gpu
@pytest.mark.parametrize('fn', sorted(PRIMITIVES))
def test_primitive_against_float64(ut, fn):
    """Worst error in ulps of the correctly rounded result per region of PRIMITIVES, measured on a B200
    (bar in brackets): exp 2.96 [3]; expm1 0.55 [2] on the polynomial side, 12.9 [13] beyond;
    expm1_neg 0.55 [2], 12.9 [13] for x <= -0.125, 9.92 [10] for 0.125 <= x <= 1, 0.85 of [8 + x] beyond;
    rcp 0.96 [1]; log 3.17 [3.5] outside [0.5, 2] and 0.80 of its absolute bound inside; sqrt 0.93 [1];
    half_1p_tanh 4.19 [4.5].  The packed flavour equals the scalar one bit for bit, the stated special
    values hold (SPECIALS), overflow gives +-inf and underflow stays within FLT_MIN."""
    make, regions = PRIMITIVES[fn]
    x = _f32(make())
    x = x[np.isfinite(x)]
    got = ut.unary(fn, x)
    ref = _ref64(fn, x)
    worst = worst_by_region(got, x, ref, regions)
    print('%-13s worst ulp error: %s' % (fn, ', '.join('%s %.2f [%g]' % (lab, worst[lab], 1 if callable(bar) else bar)
                                                       for lab, _, bar in regions)))
    # the packed flavour: bit for bit, with pairs that straddle the expm1 switch
    xp = np.concatenate([pairs_shuffled(x, 7), straddle([0.125, -0.125])])
    assert same_bits(ut.unary(fn, xp, packed=True), ut.unary(fn, xp)).all()
    sp = np.float32([c[0] for c in SPECIALS[fn]])
    check_specials(ut.unary(fn, sp), SPECIALS[fn])
    check_specials(ut.unary(fn, np.append(sp, sp[:1]) if sp.size % 2 else sp, packed=True)[:sp.size], SPECIALS[fn])
    # outside the finite normal results: overflow to inf, underflow within FLT_MIN
    r32 = np.abs(ref).astype(F32)
    with np.errstate(all='ignore'):
        over = np.isfinite(ref) & ~np.isfinite(r32)
        assert np.array_equal(got[over], np.sign(ref[over]).astype(F32) * F32(np.inf)), fn
        under = np.isfinite(ref) & (r32 < FLT_MIN)
        assert (np.abs(got[under].astype(F64) - ref[under]) <= FLT_MIN).all(), fn
    if fn == 'log':
        # through 0 near x = 1 the bar is absolute: lg2.approx.f32 (__log2f) is specified to 2^-22 absolute
        # error for x in [0.5, 2] (CUDA C++ Programming Guide, intrinsic functions), times ln 2, plus the
        # rounding of the product
        m = (x >= 0.5) & (x <= 2.0)
        abs_err = np.abs(got[m].astype(F64) - ref[m])
        bound = 2.0 ** -22 * np.log(2.0) + 0.5 * np.spacing(np.abs(ref[m]).astype(F32)).astype(F64)
        print('%-13s x in [0.5, 2]: worst |error| %.3g, worst |error| / bound %.2f' % (
            fn, abs_err.max(), (abs_err / bound).max()))
        assert (abs_err <= bound).all()
    for label, _, bar in regions:
        assert worst[label] <= (1.0 if callable(bar) else bar), (fn, label, worst[label])


EXP_AFFINE_CONSTANTS = [(1.0, 1.0), (1.0, 2.5), (1.0, 18.53), (1.0, 35.56), (1.0, 21.0), (40.0, 0.0),
                        (F32(2 * 0.095), 0.0), (F32(2 * 0.07), 0.0), (F32(2 * 0.012), 0.0), (F32(2 * 0.0065), 0.0),
                        (0.0005, 0.0), (0.0013, 0.0)]


@gpu
def test_exp_affine_against_float64(ut):
    """c e^x + add at the (c, add) of every call site, x in [-60, 60] and log-spaced over the range where
    e^x is a normal number: in ulps of the correctly rounded result (measured on a B200: 2.63 for every
    (c, add); bar 3.5).  Over- and underflow are those of e^x whatever c: +inf above ln(FLT_MAX) and add
    below ln(FLT_MIN), also where c e^x would still be a normal number (c < 1 above, c > 1 below; no call
    site comes near, their exponents are within +-60)."""
    x = _f32(np.concatenate([np.linspace(-60, 60, 1 << 17), log_sweep(100001, lo=1e-30, hi=87.3)]))
    beyond = _f32(np.concatenate([np.geomspace(88.73, 2.0 ** 24, 1001), -np.geomspace(87.35, 2.0 ** 24, 1001)]))
    worst = {}
    for c, add in EXP_AFFINE_CONSTANTS:
        c, add = F32(c), F32(add)
        got = ut.exp_affine(x, c, add)
        with np.errstate(all='ignore'):
            ref = F64(c) * np.exp(x.astype(F64)) + F64(add)
        err = ulp_error(got, ref)
        worst[(float(c), float(add))] = float(np.nanmax(err))
        xp = np.concatenate([pairs_shuffled(x, 3), beyond])
        assert same_bits(ut.exp_affine(xp, c, add, packed=True), ut.exp_affine(xp, c, add)).all()
        assert np.array_equal(ut.exp_affine(beyond, c, add), np.where(beyond > 0, F32(np.inf), add))
    print('exp_affine worst ulp error per (c, add):', ' '.join('%s=%.2f' % kv for kv in worst.items()))
    assert max(worst.values()) <= 3.5, worst


@gpu
def test_div_against_float64(ut):
    """m_div(a, b) = a * rcp(b) over quotients of log-uniform operands: measured on a B200 1.95 ulp (bar 2)."""
    rng = np.random.default_rng(9)
    n = 1 << 20
    a = (np.exp(rng.uniform(-40, 40, n)) * rng.choice([-1, 1], n)).astype(F32)
    b = (np.exp(rng.uniform(-40, 40, n)) * rng.choice([-1, 1], n)).astype(F32)
    got = ut.binary('div', a, b)
    ref = a.astype(F64) / b.astype(F64)
    worst = float(np.nanmax(ulp_error(got, ref)))
    print('div           worst ulp error: %.2f [2]' % worst)
    assert same_bits(ut.binary('div', a, b, packed=True), got).all()
    assert worst <= 2.0


# --------------------------------------------------------------------------------------------------
# (b) the packed-pair vocabulary
# --------------------------------------------------------------------------------------------------
PAIR_VALUES = np.concatenate([EDGES, ulps_around([0.125, -0.125, 0.03, -0.03], 2),
                              np.float32([3.0, -2.5, 1e-20, -7e-39, 1e-38, 6e37, -85.0, 25.0, 0.5, 2.0 ** -126 * 3]),
                              np.random.default_rng(2).normal(0, 10, 16).astype(F32)])


@gpu
def test_pair_vocabulary_equals_scalar_lane_for_lane(ut):
    """add2 / sub2 / mul2 / fma2, unary minus, vabs, sel(lt), sel(gt), vmin and vmax on f2 pairs against
    the scalar operation on each lane: bit for bit (signed zeros included: mul2 is fma(a, b, -0)), NaN
    against NaN, over every pair of PAIR_VALUES (+-0, subnormals, +-inf, NaN, FLT_MAX, the 0.125 and
    0.03 switches +-2 ulp) in two lane arrangements."""
    v = PAIR_VALUES
    a, b = (x.ravel() for x in np.meshgrid(v, v))
    if a.size % 2:
        a, b = np.append(a, a[0]), np.append(b, b[0])
    for seed in (0, 1):
        pa, pb = (np.random.default_rng(seed).permutation(a), np.random.default_rng(seed + 10).permutation(b))
        for fn in BINARY:
            assert same_bits(ut.binary(fn, pa, pb, packed=True), ut.binary(fn, pa, pb)).all(), fn
        for fn in ('neg', 'abs'):
            assert same_bits(ut.unary(fn, pa, packed=True), ut.unary(fn, pa)).all(), fn
    rng = np.random.default_rng(4)
    x, y, z = (rng.choice(v, 1 << 18) for _ in range(3))
    assert same_bits(ut.fma(x, y, z, packed=True), ut.fma(x, y, z)).all()
    # and the scalar operations are IEEE: rounded once, no flush to zero; min / max return the non-NaN
    # operand (the sign of a zero result of min(+0, -0) is compared as a value: fminf gives -0, np.fmin +0)
    with np.errstate(all='ignore'):
        assert same_bits(ut.binary('mul', a, b), a * b).all()
        assert same_bits(ut.binary('add', a, b), a + b).all()
        assert same_bits(ut.binary('sub', a, b), a - b).all()
        for fn, ref in (('min', np.fmin(a, b)), ('max', np.fmax(a, b))):
            got = ut.binary(fn, a, b)
            assert ((got == ref) | (np.isnan(got) & np.isnan(ref))).all(), fn


# --------------------------------------------------------------------------------------------------
# (c) the Courtemanche intermediates
# --------------------------------------------------------------------------------------------------
INTER = ('d_infinity', 'f_infinity', 'tau_w', 'tau_d', 'tau_f', 'w_infinity', 'm_inf', 'h_inf', 'j_inf',
         'tau_oa', 'tau_oi', 'tau_ua', 'tau_ui', 'tau_xr', 'tau_xs', 'tau_m', 'tau_h', 'tau_j',
         'oa_infinity', 'oi_infinity', 'ua_infinity', 'ui_infinity', 'xr_infinity', 'xs_infinity',
         'g_Kur', 'f_NaK', 'i_NaCaa', 'i_NaCab', 'i_K1a', 'i_Kra', 'us_infinity', 'tau_us')
TAU_COLS = [k for k, n in enumerate(INTER) if n.startswith('tau_')]


def court_reference_voltages(V):
    """float64 voltages at which court_inter is evaluated for the fp32 voltages V: V itself, except where
    a guard of the model decides differently in fp32 (as the kernels and the fp32 reference evaluate it)
    than in float64.  At the five singular voltages fp32(c) + fp32(-c) == 0 takes the guarded constant
    (tau_d, tau_w, alpha/beta of xr and xs), which float64 reaches only at c itself; at the alpha_m guard
    |V + 47.13| < 0.001 one fp32 voltage (-47.131) is inside in fp32 and outside in float64.  Those
    voltages move by < 2e-6 mV to the float64 value with the fp32 decision: the guarded constants are
    not the limits of the formulas (4.579 / 2 against 1 / (6.24 * 0.07) for tau_d: 5e-5 apart;
    alpha_m: 3.2 against 3.20016), so comparing across the decision would compare two models."""
    V64 = V.astype(F64)
    for c in SINGULAR_MV:
        V64[V == F32(c)] = c
    with np.errstate(all='ignore'):
        in32 = np.abs(V - F32(-47.13)) < F32(0.001)
    w = V64 + 47.13
    in64 = np.abs(w) < 0.001
    V64[in32 & ~in64] = -47.13 + np.sign(w[in32 & ~in64]) * 0.000999999
    V64[~in32 & in64] = -47.13 + np.sign(w[~in32 & in64]) * 0.001
    return V64


@pytest.fixture(scope='module')
def court_ref():
    V = court_voltages()
    with np.errstate(all='ignore'):
        q = onp.court_inter(court_reference_voltages(V), ultra=True)
        q32 = onp.court_us(V, {})            # the reference's own fp32 evaluation of the us gate
    return (V, np.stack([np.asarray(q[n], F64) for n in INTER], axis=1),
            np.stack([np.asarray(q32[n], F64) for n in INTER[30:]], axis=1))


@gpu
@pytest.mark.parametrize('us', [False, True], ids=['no_us', 'us'])
@pytest.mark.parametrize('rates', [False, True], ids=['tau', 'rates'])
def test_court_inter_against_float64(ut, court_ref, us, rates):
    """court_inter_dev<US, RATES, float> on ~2^20 voltages (court_voltages) against court_inter in float64:
    relative error <= 1e-5 per entry (absolute floor 1e-30: h_inf and j_inf are V * 1e-20-sized above
    -40 mV); with RATES the tau columns hold 1/tau and are compared with 1/tau64.  Finite wherever the
    reference is finite and normal.

    alpha_m = 0.32 w / (1 - e^y), y = -0.1 w, w = V + 47.13, is the reference's expression: the reference
    guards only |w| < 0.001, and just outside the guard 1 - e^y cancels, in the reference's fp32 (up to
    2^-24 / |y| relative) as in the kernels, whose e^y is m_exp's (< 3 ulp).  So m_inf and tau_m are held
    to 1e-5 + 3 2^-23 / |y|, that conditioning with m_exp's bound.  (Routing this e^y - 1 through the
    expm1 fix-up of the singularities brings m_inf to 2.4e-6 of float64, but also away from the fp32
    reference: the Courtemanche spiral's APD then leaves its 1 % bound in
    tests/test_spiral_statistics.py, so the kernels keep the reference's expression.)

    Measured on a B200, for every (US, RATES): worst 3.3e-6 (oi_infinity at 61.6 mV) outside m_inf and
    tau_m; those reach 5.7e-4 at w = -0.001, inside their bar.

    us_infinity and tau_us are the reference's fp32 expression 0.5 (1 -+ tanh z) with libm tanhf, on
    purpose (court_ultra.py:445-450): 1 - tanh z cancels for z >> 1 (V > -40 mV), so the reference's own
    fp32 result is 2e-2 off float64 at V = 80 mV.  Their bar is never tighter than 3x that distance of
    the fp32 reference (onp.court_us in fp32) from float64, the fixtures' `rounding` term."""
    V, want, us32 = court_ref
    got = ut.court_inter(V, us, rates).astype(F64)
    if not us:
        assert (got[:, 30] == 0).all() and (got[:, 31] == 1).all()
    want = want.copy()
    us32 = us32.copy()
    if rates:
        with np.errstate(divide='ignore'):
            want[:, TAU_COLS] = 1.0 / want[:, TAU_COLS]
            us32[:, 1] = 1.0 / us32[:, 1]
    cols = range(32 if us else 30)
    worst = {}
    for k in cols:
        w, g = want[:, k], got[:, k]
        normal = np.isfinite(w) & (np.abs(w) >= FLT_MIN)
        assert np.isfinite(g[normal]).all(), (INTER[k], V[normal & ~np.isfinite(g)][:5])
        scale = np.maximum(np.abs(w), 1e-30)
        err = np.abs(g - w) / scale
        if k in (INTER.index('m_inf'), INTER.index('tau_m')):
            with np.errstate(divide='ignore'):
                bar = 1e-5 + 3.0 * 2.0 ** -23 / np.abs(0.1 * (V.astype(F64) + 47.13))
        elif k < 30:
            bar = 1e-5
        else:
            bar = np.maximum(1e-5, 3.0 * np.abs(us32[:, k - 30] - w) / scale)
        i = int(np.argmax(err / bar))
        worst[INTER[k]] = (float(err[i]), float(V[i]))
        assert (err <= bar).all(), (INTER[k], float(err[i]), float(V[i]))
    name = max(INTER[:30], key=lambda n: worst[n][0])
    print('court_inter<us=%d, rates=%d>: worst relative error %.2e (%s at V = %r); per column: %s' % (
        us, rates, worst[name][0], name, worst[name][1], ' '.join('%s=%.1e' % (n, e) for n, (e, _) in worst.items())))


@gpu
def test_court_rates_agree_with_time_constants(ut, court_ref):
    """RATES = true against RATES = false column by column on the same voltages: 1/rate against tau, the
    other columns directly, in ulps of the RATES = false value.  Measured on a B200: worst 7.1 ulp
    (tau_oa / tau_ua), bar 8; the columns the rate form does not touch are identical."""
    V = court_ref[0]
    tau = ut.court_inter(V, True, False).astype(F64)
    rate = ut.court_inter(V, True, True).astype(F64)
    with np.errstate(divide='ignore'):
        rate[:, TAU_COLS] = 1.0 / rate[:, TAU_COLS]
    worst = {}
    for k, n in enumerate(INTER):
        err = ulp_error(rate[:, k], tau[:, k])
        tiny = ~np.isfinite(err)
        assert (np.abs(rate[tiny, k] - tau[tiny, k]) <= FLT_MIN).all(), n
        worst[n] = float(np.nanmax(err))
    print('1/rate against tau, worst ulps per column:', ' '.join('%s=%.1f' % kv for kv in worst.items()))
    assert max(worst.values()) <= 8.0, worst


def court_pairs():
    """The voltages in a shuffled order, plus pairs whose lanes straddle -40 mV, the alpha_m guard, every
    singular voltage and every |y| = 0.03 voltage, and pairs of one such voltage with a regular one."""
    V = court_voltages()
    special = np.float32([-40.0, F32(-47.13) - F32(0.001), F32(-47.13) + F32(0.001)])
    s = np.concatenate([special, COURT_SINGULAR, COURT_Y003])
    mixed = np.stack([ulps_around(s, 4), np.resize(np.float32([-80.0, 10.0, 33.3, -55.5]), 9 * s.size)], -1).ravel()
    return np.concatenate([pairs_shuffled(V, 11), straddle(s, 16), mixed])


@gpu
@pytest.mark.parametrize('us', [False, True], ids=['no_us', 'us'])
@pytest.mark.parametrize('rates', [False, True], ids=['tau', 'rates'])
def test_court_inter_pairs_equal_scalar(ut, us, rates):
    """court_inter_dev on f2 pairs equals the scalar flavour lane for lane, bit for bit, also where the
    two lanes take different sides of a switch or guard."""
    V = court_pairs()
    assert same_bits(ut.court_inter(V, us, rates, packed=True), ut.court_inter(V, us, rates)).all()


@gpu
@pytest.mark.parametrize('packed', [False, True], ids=['float', 'f2'])
def test_court_inter_lane_does_not_depend_on_its_warp(ut, packed):
    """The expm1 fix-up next to the removable singularities sits behind a warp vote (__any_sync).  The
    same voltages are evaluated grouped (the near-singular ones fill whole warps, the regular ones
    others) and interleaved (one near-singular voltage in every warp of regular ones): every lane's
    result is bit-identical between the two layouts."""
    lanes = 2 if packed else 1
    W = 32 * lanes
    near = np.concatenate([ulps_around(COURT_SINGULAR, 16), ulps_around(COURT_Y003, 16)])
    grid = np.linspace(-120.0, 80.0, 1 << 18).astype(F32)
    far = np.min(np.abs(grid[:, None].astype(F64) - np.concatenate([COURT_SINGULAR, COURT_Y003])[None, :]), 1) > 1.0
    regular = grid[far]
    m = -(-near.size // W) * W
    near = np.resize(near, m)
    assert regular.size >= m * (W - 1)
    grouped = np.concatenate([near, regular[:m * (W - 1)]])
    # interleaved warp k: near[k], then W - 1 regular voltages
    perm = np.concatenate([np.concatenate([[k], m + k * (W - 1) + np.arange(W - 1)]) for k in range(m)])
    for us, rates in ((True, True), (False, False)):
        a = ut.court_inter(grouped, us, rates, packed)
        b = ut.court_inter(grouped[perm], us, rates, packed)
        assert same_bits(b, a[perm]).all(), (us, rates)


# --------------------------------------------------------------------------------------------------
# (d) the Beeler-Reuter gates
# --------------------------------------------------------------------------------------------------
BR_SLOT = {'XI': 6, 'M': 1, 'H': 2, 'J': 3, 'D': 4, 'F': 5}       # BR_GATES -> index in the cell's s[7]
BR_DT, BR_DT_SLOW = 0.1, 0.4


def br_voltages():
    """[-90, 30] mV dense, and +-16 ulps around -23 and -47 mV (removable singularities) and around
    -47 -+ 1.25 mV (|0.1 (V + 47)| = 0.125, the expm1 switch of alpha_m)."""
    return np.concatenate([np.linspace(-90.0, 30.0, 1 << 16).astype(F32),
                           ulps_around([-23.0, -47.0, -48.25, -45.75], 16)])


def br_planted(V, seed=6):
    s = np.random.default_rng(seed).uniform(0.01, 0.99, (V.size, 7)).astype(F32)
    s[:, 0] = F32(2e-7)                     # C: not a gate, left alone
    return s


def br_oracle(V, s, wide, relax=None):
    """One Rush-Larsen update of the six gates with inf and tau from onp.br_inf_tau_exact, in float64
    (wide) or in the oracle's fp32; -> [n, 7] (column 0 = C unchanged).  relax, if given, receives
    8 ulp(fp32 inf) * |expm1(-dt / tau)| per gate."""
    out = np.empty(s.shape, F64 if wide else F32)
    out[:, 0] = s[:, 0]
    Vx = V.astype(F64) if wide else V
    with np.errstate(all='ignore'):
        for g, name in enumerate(onp.BR_GATES):
            inf, tau = onp.br_inf_tau_exact(Vx, g)
            k = BR_SLOT[name]
            gk = s[:, k].astype(F64) if wide else s[:, k]
            dt = BR_DT if name in ('M', 'H') else BR_DT_SLOW
            out[:, k] = onp.rush_larsen(gk, inf, tau, dt)
            if relax is not None:
                relax[:, k] = np.nan_to_num(8.0 * np.spacing(np.abs(inf).astype(F32)) * np.abs(np.expm1(F32(-dt) / tau)))
    return out


@gpu
def test_br_exact_gates_one_update_against_float64(ut):
    """br_gates_exact<SLOW=true> (the trimmed exact gates: folded exponentials, rush_larsen_frac), one update
    at fixed V from planted gates, scalar and packed, against Rush-Larsen in float64 with inf and tau of
    onp.br_inf_tau_exact in float64.  Bar per cell: 1e-5 of the increment (floor 1e-6) plus one ulp, never
    tighter than 3x how far the fp32 oracle moves when V moves by one ulp, nor than 3x the fp32 oracle's
    own distance from float64 (the fixtures' `rounding` term), plus 8 ulps of g_inf times the fraction
    |expm1(-dt/tau)| by which the gate relaxes towards it: g_inf comes out of four or five few-ulp SFU
    operations, and a cell planted next to its equilibrium has an increment too small to carry that
    error.  Measured on a B200: see the printout (worst |error| / bar per gate)."""
    V = br_voltages()
    s = br_planted(V)
    got = ut.br_gates_exact(V, s, F32(-BR_DT), F32(-BR_DT_SLOW))
    assert np.array_equal(got[:, 0], s[:, 0])
    relax = np.zeros(s.shape)
    want = br_oracle(V, s, wide=True, relax=relax)
    base = br_oracle(V, s, wide=False).astype(F64)
    drift = np.zeros(s.shape)
    for d in (np.inf, -np.inf):
        drift = np.fmax(drift, np.abs(br_oracle(np.nextafter(V, F32(d)), s, wide=False).astype(F64) - base))
    worst = {}
    for name, k in BR_SLOT.items():
        inc = np.abs(want[:, k] - s[:, k])
        bar = 1e-5 * np.maximum(inc, 1e-6) + np.spacing(np.abs(want[:, k]).astype(F32)).astype(F64) + relax[:, k]
        bar = np.fmax(bar, 3.0 * np.fmax(drift[:, k], np.abs(base[:, k] - want[:, k])))
        ratio = np.abs(got[:, k] - want[:, k]) / bar
        i = int(np.argmax(ratio))
        worst[name] = (float(ratio[i]), float(V[i]))
    print('br_gates_exact one update: worst |error| / bar per gate:',
          ' '.join('%s=%.2f (V=%r)' % (n, r, v) for n, (r, v) in worst.items()))
    assert max(r for r, _ in worst.values()) <= 1.0, worst
    Vp = np.concatenate([pairs_shuffled(V, 13), straddle([-23.0, -47.0, -48.25, -45.75], 16)])
    sp = br_planted(Vp, 8)
    assert same_bits(ut.br_gates_exact(Vp, sp, F32(-BR_DT), F32(-BR_DT_SLOW), packed=True),
                     ut.br_gates_exact(Vp, sp, F32(-BR_DT), F32(-BR_DT_SLOW))).all()


@gpu
def test_br_inf_rate_exact_against_float64(ut):
    """br_inf_rate_exact (the readable statement of the exact gates, used by the accurate-math build)
    against inf = a / (a + b) and rate = a + b in float64: relative error <= 1e-5 (floor 1e-30, NaN where
    the reference is NaN: alpha_m's 0/0 at V = -47.0f).  Measured on a B200: worst 1.2e-6 (H_inf, J_inf)."""
    V = br_voltages()
    got = ut.br_inf_rate_exact(V)
    worst = {}
    with np.errstate(all='ignore'):
        for g, name in enumerate(onp.BR_GATES):
            inf, tau = onp.br_inf_tau_exact(V.astype(F64), g)
            for j, want in ((0, inf), (1, 1.0 / tau)):
                worst['%s_%s' % (name, ('inf', 'rate')[j])] = onp.rel_err(got[:, 2 * g + j], want, 1e-30)
    print('br_inf_rate_exact worst relative error:', ' '.join('%s=%.1e' % kv for kv in worst.items()))
    assert max(worst.values()) <= 1e-5, worst


@gpu
def test_br_poly8_horner_is_at_least_as_accurate_as_the_reference_sum(ut):
    """br_poly8 with the coefficients the library passes (c_i = ldexp(fp32(d_i), i - 1), fib_capi.cu) at the
    kernel's x = (V + 30) * fp32(1/60), against sum fp32(d_i) S_i(x) in float64 at the same x.  Per gate
    function the worst absolute error over [-90, 30] mV is no larger than that of the reference's fp32
    left-to-right sum in the S basis (onp.br_cheby_eval).  Measured on a B200: Horner's worst error is
    0.38 - 0.64 of the reference sum's, per gate function (M_tau 0.64)."""
    V = np.linspace(-90.0, 30.0, 1 << 16).astype(F32)
    x = (V + F32(30.0)) * F32(1.0 / 60.0)
    d = onp.br_cheby_coeffs()
    Ts = [F32(1.0), x]
    for _ in range(7):
        Ts.append(2 * x * Ts[-1])
    names = ['%s_%s' % (g, q) for g in onp.BR_GATES for q in ('inf', 'tau')]
    ratios = {}
    for r in range(12):
        d32 = d[r].astype(F32)
        c = np.float32([d32[i] if i < 2 else np.ldexp(d32[i], i - 1) for i in range(9)])
        exact = np.zeros(x.shape)
        for ci in c[::-1].astype(F64):
            exact = exact * x.astype(F64) + ci
        got = ut.br_poly8(c, x)
        e_dev = np.abs(got - exact).max()
        e_ref = np.abs(onp.br_cheby_eval(Ts, d[r]).astype(F64) - exact).max()
        ratios[names[r]] = (e_dev, e_ref)
        xp = pairs_shuffled(x, r)
        assert same_bits(ut.br_poly8(c, xp, packed=True), ut.br_poly8(c, xp)).all()
    print('br_poly8 worst |error| (Horner / reference sum):',
          ' '.join('%s=%.2g/%.2g' % (n, a, b) for n, (a, b) in ratios.items()))
    assert all(a <= b for a, b in ratios.values()), ratios
