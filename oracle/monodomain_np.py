"""
TEST INFRASTRUCTURE (see oracle/README.md) -- THE ORACLE.  Never imported by
fib_tf_b200/; only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline leg
may use it, and only as the checker / timed baseline.

monodomain_np: a hand restatement, in NumPy fp32, of the reference's hot path
(no-flux boundary + 9-point Laplacian + phase-field term + pointwise ionic update)
for the three ionic models and their schedules.  Each function cites the reference
`file:line` (relative to /root/reference) it restates.  The arithmetic keeps the
reference's operand order and its Python-level constant folding so that the
result is BIT-IDENTICAL to the unmodified reference executed through
oracle/tfshim.py; tests/test_oracle_golden.py pins that against tests/golden/*.npz.

Parity pin: golden fixtures generated from the reference's own code (see
oracle/make_golden.py).  The reference itself ships no golden vectors.
"""
import numpy as np
from numpy.polynomial.chebyshev import Chebyshev

F32 = np.float32


# --------------------------------------------------------------------------
# stencil helpers (ionic.py)
# --------------------------------------------------------------------------
def enforce_boundary(X):
    """ionic.py:107-113 -- border ring := SYMMETRIC pad of the interior."""
    return np.pad(X[1:-1, 1:-1], 1, mode='symmetric')


def phase_term(Xp, phase):
    """ionic.py:70-81 -- (dX.dphi)/(4 phi) with central differences, phi REFLECT-padded."""
    P = np.pad(phase, 1, mode='reflect')
    return ((Xp[2:, 1:-1] - Xp[:-2, 1:-1]) * (P[2:, 1:-1] - P[:-2, 1:-1]) +
            (Xp[1:-1, 2:] - Xp[1:-1, :-2]) * (P[1:-1, 2:] - P[1:-1, :-2])
            ) / (F32(4) * P[1:-1, 1:-1])


def laplace(X0, phase=None):
    """ionic.py:44-60 -- REFLECT pad, then N+S+W+E + 0.5*(NW+SW+NE+SE) - 6*C (+ phase term)."""
    Xp = np.pad(X0, 1, mode='reflect')
    lap = (Xp[:-2, 1:-1] + Xp[2:, 1:-1] + Xp[1:-1, :-2] + Xp[1:-1, 2:] +
           F32(0.5) * (Xp[:-2, :-2] + Xp[2:, :-2] + Xp[:-2, 2:] + Xp[2:, 2:]) -
           F32(6) * Xp[1:-1, 1:-1])
    if phase is not None:
        lap = lap + phase_term(Xp, phase)
    return lap


def clip_by_value(x, lo, hi):
    """tf.clip_by_value = maximum(minimum(x, hi), lo) with the NaN behaviour of the reference's GPU
    target (Eigen's CUDA mini/maxi = fminf/fmaxf: the non-NaN operand wins), see
    fib_tf_b200/csrc/fib_common.cuh.  np.fmin/np.fmax have exactly those semantics."""
    return np.fmax(np.fmin(x, F32(hi)), F32(lo))


def rush_larsen(g, g_inf, tau, dt, clip=True):
    """ionic.py:115-123 -- clip(g + (g - g_inf) * expm1(-dt / tau), 1e-5, 0.99999).
    clip=False: no clip, the rule of courtemanche.h (FIB_F_NO_CLIP)."""
    if isinstance(tau, np.ndarray):
        e = np.expm1(F32(-dt) / tau)
    else:                                   # Python-scalar tau: folded in Python, then fp32
        e = np.expm1(F32(-dt / tau))
    g1 = g + (g - g_inf) * e
    return clip_by_value(g1, 0.00001, 0.99999) if clip else g1


def hole_phase(phase, height, width, x, y, radius, neg=False):
    """ionic.py:83-105 -- multiply a tanh hole into the phase field; floor 1e-5."""
    if phase is None:
        phase = np.ones([height, width], dtype=np.float32)
    xx, yy = np.meshgrid(np.arange(width), np.arange(height))
    dist = np.hypot(xx - x, yy - y)
    if neg:
        phase = phase * np.array(0.5 * (np.tanh(0.1 * (radius - dist)) + 1.0), dtype=np.float32)
    else:
        phase = phase * np.array(0.5 * (np.tanh(dist - radius) + 1.0), dtype=np.float32)
    return np.maximum(phase, 1e-5).astype(np.float32)


def pace_region(loc, height, width):
    """ionic.py:144-162 -- (r0, r1, c0, c1) half-open rectangle of a named stimulus site."""
    H, W = height, width
    table = {
        'left': (0, H, 0, 5), 'right': (0, H, W - 5, W),
        'top': (0, 5, 0, W), 'bottom': (H - 5, H, 0, W),
        'luq': (1, H // 2, 1, W // 2), 'llq': (H // 2, H - 1, 1, W // 2),
        'ruq': (1, H // 2, W // 2, W - 1), 'rlq': (H // 2, H - 1, W // 2, W - 1),
    }
    return table.get(loc)       # None: unknown site -> V := max(V, min_v) everywhere


def apply_pace(X, loc, v, min_v):
    """ionic.py:144-163 -- X := max(X, s), s = min_v outside the region and v inside."""
    H, W = X.shape
    s = np.full([H, W], min_v, dtype=np.float32)
    reg = pace_region(loc, H, W)
    if reg is not None:
        r0, r1, c0, c1 = reg
        s[max(r0, 0):r1, max(c0, 0):c1] = v
    return np.fmax(X, s)       # tf.maximum on the GPU target: the non-NaN operand wins


# --------------------------------------------------------------------------
# Fenton 4v (fenton.py)
# --------------------------------------------------------------------------
def fenton_rates(U, V, W, S):
    """fenton.py:46-92 -- dU, dV, dW, dS of the Cherry-Ehrlich-Nattel-Fenton 4v model."""
    tau_vp, tau_vn, tau_wp, tau_wn1, tau_wn2 = 3.33, 19.2, 160.0, 75.0, 75.0
    tau_d, tau_si, tau_a = 0.065, 31.8364, 0.009
    tau_so = tau_si
    u_c, u_w, u_0, u_m, u_csi, u_so = 0.23, 0.146, 0.0, 1.0, 0.8, 0.3
    r_sp, r_sn, k_ = 0.02, 1.2, 3.0
    a_so, b_so, c_so = 0.115, 0.84, 0.02

    def step_up(x):      # H, fenton.py:73-75
        return (F32(1) + np.sign(x)) * F32(0.5)

    def step_dn(x):      # G, fenton.py:77-79
        return (F32(1) - np.sign(x)) * F32(0.5)

    I_fi = -V * step_up(U - u_c) * (U - u_c) * (u_m - U) / tau_d
    I_si = -W * S / tau_si
    I_so = (0.5 * (a_so - tau_a) * (F32(1) + np.tanh((U - b_so) / c_so)) +
            (U - u_0) * step_dn(U - u_so) / tau_so + step_up(U - u_so) * tau_a)
    dU = -(I_fi + I_si + I_so)
    dV = np.where(U > u_c, -V / tau_vp, (F32(1) - V) / tau_vn)
    dW = np.where(U > u_c, -W / tau_wp,
                  np.where(U > u_w, (F32(1) - W) / tau_wn2, (F32(1) - W) / tau_wn1))
    r_s = (r_sp - r_sn) * step_up(U - u_c) + r_sn
    dS = r_s * (F32(0.5) * (F32(1) + np.tanh((U - u_csi) * k_)) - S)
    return dU, dV, dW, dS


def fenton_step(st, dt, diff, phase=None):
    """fenton.py:95-108 -- one explicit Euler step.  Reaction sees the RAW U; the Euler
    base and the Laplacian see the boundary-enforced U0."""
    U, V, W, S = st['U'], st['V'], st['W'], st['S']
    U0 = enforce_boundary(U)
    dU, dV, dW, dS = fenton_rates(U, V, W, S)
    return {
        'U': U0 + dt * dU + diff * dt * laplace(U0, phase),
        'V': V + dt * dV, 'W': W + dt * dW, 'S': S + dt * dS,
    }


def fenton_init(height, width, s1=True):
    """fenton.py:116-123."""
    st = {'U': np.zeros([height, width], np.float32), 'V': np.ones([height, width], np.float32),
          'W': np.ones([height, width], np.float32), 'S': np.zeros([height, width], np.float32)}
    if s1:
        st['U'][:, 1] = 1.0
    return st


# --------------------------------------------------------------------------
# Beeler-Reuter (br.py)
# --------------------------------------------------------------------------
BR_AB = np.array(                       # br.py:49-62 (d and f rates doubled, br.py:46-48)
    [[0.0005, 0.083, 50., 0.0, 0.0, 0.057, 1.0],        # alpha x1
     [0.0013, -0.06, 20., 0.0, 0.0, -0.04, 1.0],        # beta  x1
     [0.0000, 0.0, 47., -1.0, 47., -0.1, -1.0],         # alpha m
     [40., -0.056, 72., 0.0, 0.0, 0.0, 0.0],            # beta  m
     [0.126, -.25, 77., 0.0, 0.0, 0.0, 0.0],            # alpha h
     [1.7, 0.0, 22.5, 0.0, 0.0, -0.082, 1.0],           # beta  h
     [0.055, -.25, 78.0, 0.0, 0.0, -0.2, 1.0],          # alpha j
     [0.3, 0.0, 32., 0.0, 0.0, -0.1, 1.0],              # beta  j
     [2 * 0.095, -0.01, -5., 0.0, 0.0, -0.072, 1.0],    # alpha d
     [2 * 0.07, -0.017, 44., 0.0, 0.0, 0.05, 1.0],      # beta  d
     [2 * 0.012, -0.008, 28., 0.0, 0.0, 0.15, 1.0],     # alpha f
     [2 * 0.0065, -0.02, 30., 0.0, 0.0, -0.2, 1.0]],    # beta  f
    dtype=np.float32)
BR_MIN_V, BR_MAX_V = -90.0, 30.0
# gate order used everywhere below: xi, m, h, j, d, f  (br.py:285-286 column order)
BR_GATES = ('XI', 'M', 'H', 'J', 'D', 'F')


def br_rate(v, c):
    """br.py:255-264 -- (c0 e^{c1(v+c2)} + c3 (v+c4)) / (e^{c5(v+c2)} + c6)."""
    if c[3] == 0:
        return (c[0] * np.exp(c[1] * (v + c[2]))) / (np.exp(c[5] * (v + c[2])) + c[6])
    return ((c[0] * np.exp(c[1] * (v + c[2])) + c[3] * (v + c[4])) /
            (np.exp(c[5] * (v + c[2])) + c[6]))


def br_inf_tau_exact(v, gate):
    """br.py:266-273 -- inf = a/(a+b), tau = 1/(a+b); gate index in BR_GATES order."""
    a = br_rate(v, BR_AB[2 * gate])
    b = br_rate(v, BR_AB[2 * gate + 1])
    return a / (a + b), F32(1.0) / (a + b)


def br_cheby_coeffs(deg=8):
    """br.py:275-287 + 303-326 -- host-side (fp64) degree-8 Chebyshev least-squares fit of
    inf and tau of the six gates on V in [-90, 30] (1001 samples), re-expressed in the
    scaled-monomial basis S_i = 2^{i-1} x^i.  Returns d[12][deg+1] float64:
    rows 2g = inf of gate g, 2g+1 = tau of gate g (BR_GATES order)."""
    v = np.linspace(BR_MIN_V, BR_MAX_V, 1001)
    x = np.outer(v, np.ones(BR_AB.shape[0]))
    y = ((BR_AB[:, 0] * np.exp(BR_AB[:, 1] * (x + BR_AB[:, 2])) + BR_AB[:, 3] * (x + BR_AB[:, 4])) /
         (np.exp(BR_AB[:, 5] * (x + BR_AB[:, 2])) + BR_AB[:, 6]))
    alpha, beta = y[..., ::2], y[..., 1::2]
    # T_i in powers of x (integer), then divide column j by the leading coefficient of T_j
    a = np.zeros([deg + 1, deg + 1], dtype=int)
    a[0, 0] = 1
    a[1, 1] = 1
    for i in range(2, deg + 1):
        a[i, 1:] += 2 * a[i - 1, :-1]
        a[i, :] -= a[i - 2, :]
    a //= np.diag(a)
    out = np.zeros([12, deg + 1])
    for g in range(6):
        for k, yy in enumerate((alpha[:, g] / (alpha[:, g] + beta[:, g]),
                                1.0 / (alpha[:, g] + beta[:, g]))):
            c = Chebyshev.fit(v, yy, deg).coef
            out[2 * g + k] = np.matmul(np.transpose(a), c)
    return out


def br_cheby_eval(Ts, d):
    """br.py:327-331 -- r = d0 + sum_i d_i * S_i, left to right, coefficients cast to fp32."""
    r = F32(d[0]) + F32(d[1]) * Ts[1]
    for i in range(2, len(Ts)):
        r = r + F32(d[i]) * Ts[i]
    return r


def br_gate_update(V0, st, dt, n, cheby, coeffs):
    """br.py:175-205 (exact) / 207-252 (Chebyshev): m, h advance by dt every step; xi, j, d, f
    advance by dt*n when n > 0 and are frozen when n == 0."""
    if cheby:
        x = (V0 - 0.5 * (BR_MAX_V + BR_MIN_V)) / (0.5 * (BR_MAX_V - BR_MIN_V))
        Ts = [1.0, x]
        for _ in range(7):                      # br.py:289-301, deg fixed at 8 (br.py:219)
            Ts.append(2 * x * Ts[-1])

        def inf_tau(g):
            return br_cheby_eval(Ts, coeffs[2 * g]), br_cheby_eval(Ts, coeffs[2 * g + 1])
    else:
        def inf_tau(g):
            return br_inf_tau_exact(V0, g)
    new = {}
    for g, name in enumerate(BR_GATES):
        fast = name in ('M', 'H')
        if fast or n > 0:
            inf, tau = inf_tau(g)
            new[name] = rush_larsen(st[name], inf, tau, dt if fast else dt * n)
        else:
            new[name] = st[name]
    return new


def br_step(st, dt, diff, n=1, cheby=False, coeffs=None, phase=None):
    """br.py:125-173 -- one step; currents use V0 = enforce_boundary(V) and the OLD gates."""
    V, C = st['V'], st['C']
    M, Hg, J, D, Fg, XI = st['M'], st['H'], st['J'], st['D'], st['F'], st['XI']
    V0 = enforce_boundary(V)
    new = br_gate_update(V0, st, dt, n, cheby, coeffs)
    C_K1 = C_x1 = C_Na = C_s = 1.0
    g_s, g_Na, g_NaC, ENa, C_m = 0.09, 4.0, 0.005, 50.0 + 0.0, 1.0
    iK1 = 0.35 * (4 * (np.exp(0.04 * (V0 + 85)) - 1) /
                  (np.exp(0.08 * (V0 + 53)) + np.exp(0.04 * (V0 + 53))) +
                  0.2 * ((V0 + 23.0) / (1.0 - np.exp(-0.04 * (V0 + 23)))))
    ix1 = XI * 0.8 * (np.exp(0.04 * (V0 + 77)) - 1) / np.exp(0.04 * (V0 + 35))
    iNa = C_Na * (g_Na * M * M * M * Hg * J + g_NaC) * (V0 - ENa)
    ECa = 0.0 - 82.3 - 13.0278 * np.log(C)
    iCa = C_s * g_s * D * Fg * (V0 - ECa)
    I_sum = iK1 + ix1 + iNa + iCa
    V1 = V0 + diff * dt * laplace(V0, phase) - dt * I_sum / C_m
    new['V'] = clip_by_value(V1, -85.0, 25.0)
    dC = -1.0e-7 * iCa + 0.07 * (1.0e-7 - C)
    new['C'] = C + dt * dC
    return new


def br_init(height, width, s1=True):
    """br.py:71-82."""
    vals = {'V': -84.624, 'C': 1e-4, 'M': 0.01, 'H': 0.988, 'J': 0.975, 'D': 0.003,
            'F': 0.994, 'XI': 0.0001}
    st = {k: np.full([height, width], v, dtype=np.float32) for k, v in vals.items()}
    if s1:
        st['V'][:, 1] = 10.0
    return st


# --------------------------------------------------------------------------
# Courtemanche (court.py, court_ultra.py)
# --------------------------------------------------------------------------
COURT_INIT = (                         # court.py:57-78 (dict insertion order)
    ('V', -81.18), ('_Na_i_', 1.117e+01), ('_m_', 2.98e-3), ('_h_', 9.649e-1),
    ('_j_', 9.775e-1), ('_K_i_', 1.39e+02), ('_oa_', 3.043e-2), ('_oi_', 9.992e-1),
    ('_ua_', 4.966e-3), ('_ui_', 9.986e-1), ('_xr_', 3.296e-5), ('_xs_', 1.869e-2),
    ('_Ca_i_', 1.013e-4), ('_d_', 1.367e-4), ('_f_', 9.996e-1), ('_f_Ca_', 7.755e-1),
    ('_Ca_rel_', 1.488), ('_u_', 0.0), ('_v_', 1.0), ('_w_', 0.9992), ('_Ca_up_', 1.488))
COURT_FAST = ('V', '_Na_i_', '_m_', '_h_')      # court.py:42


def court_init(height, width, s1=True, ultra_slow=False):
    """court.py:57-82; court_ultra.py:81-82 adds '_us_' = 0.72."""
    st = {k: np.full([height, width], v, dtype=np.float32) for k, v in COURT_INIT}
    if ultra_slow:
        st['_us_'] = np.full([height, width], 0.72, dtype=np.float32)
    if s1:
        st['V'][:, :25] = 20.0
    return st


def court_inter(V, ultra=False):
    """court.py:273-429 (V-only intermediates); court_ultra.py:445-450 adds the us gate."""
    R, T, F, Cm, Na_o = 8.3143, 310, 96.4867, 100, 140
    g_K1, K_Q10, g_Kr, Ca_o = 0.09, 3, 0.029411765, 1.8
    I_NaCa_max, K_mNa, K_mCa, K_sat, gamma_, sigma = 1600, 87.5, 1.38, 0.1, 0.35, 1.0
    exp, rcp, absf, where = np.exp, np.reciprocal, np.abs, np.where
    q = {}
    eps = V * 1e-20

    q['d_infinity'] = rcp(1.0 + exp((V + 10.0) / -8.0))
    q['tau_d'] = where(
        absf(V + 10.0001) < 1.0e-10,
        4.579 / (1.0 + exp((V + 10.0) / -6.24)),
        (1.0 - exp((V + 10.0001) / -6.24)) /
        (0.0350000 * (V + 10.0001) * (1.0 + exp((V + 10.0001) / -6.24))))
    q['f_infinity'] = exp(-(V + 28.0) / 6.9) / (1.0 + exp(-(V + 28.0) / 6.9))
    q['tau_f'] = 9.0 * rcp(0.0197000 * exp(-np.square(F32(0.0337)) * np.square(V + 10.0)) + 0.02)
    q['tau_w'] = where(
        absf(V - 7.9) < 1.0e-10,
        eps + ((6.0 * 0.2) / 1.3),
        (6.0 * (1.0 - exp(-(V - 7.9) / 5.0))) /
        ((1.0 + 0.3 * exp(-(V - 7.9) / 5.0)) * 1.0 * (V - 7.9)))
    q['w_infinity'] = 1.0 - rcp(1.0 + exp(-(V - 40.0) / 17.0))

    alpha_m = where(absf(V - -47.13) < 0.001, eps + 3.2,
                    (0.32 * (V + 47.13)) / (1.0 - exp(-0.1 * (V + 47.13))))
    beta_m = 0.08 * exp(-V / 11.0)
    q['m_inf'] = alpha_m / (alpha_m + beta_m)
    q['tau_m'] = rcp(alpha_m + beta_m)

    lo = V < -40.0
    alpha_h = where(lo, 0.135 * exp((V + 80.0) / -6.8), eps)
    beta_h = where(lo, 3.56 * exp(0.079 * V) + 310000. * exp(0.35 * V),
                   rcp(0.13 * (1.0 + exp((V + 10.66) / -11.1))))
    q['h_inf'] = alpha_h / (alpha_h + beta_h)
    q['tau_h'] = rcp(alpha_h + beta_h)

    alpha_j = where(
        lo,
        ((-127140. * exp(0.2444 * V) - 3.474e-05 * exp(-0.04391 * V)) * (V + 37.78)) /
        (1.0 + exp(0.311 * (V + 79.23))),
        eps)
    beta_j = where(lo,
                   (0.1212 * exp(-0.01052 * V)) / (1.0 + exp(-0.1378 * (V + 40.14))),
                   (0.3 * exp(-2.535e-07 * V)) / (1.0 + exp(-0.1 * (V + 32.0))))
    q['j_inf'] = alpha_j / (alpha_j + beta_j)
    q['tau_j'] = rcp(alpha_j + beta_j)

    Vs = V - -10.0
    alpha_oa = 0.65 * rcp(exp(Vs / -8.5) + exp((Vs - 40.0) / -59.0))
    beta_oa = 0.65 * rcp(2.5 + exp((Vs + 72.0) / 17.0))
    q['tau_oa'] = rcp(alpha_oa + beta_oa) / K_Q10
    q['oa_infinity'] = rcp(1.0 + exp((Vs + 10.47) / -17.54))

    alpha_oi = rcp(18.53 + 1.0 * exp((Vs + 103.7) / 10.95))
    beta_oi = rcp(35.56 + 1.0 * exp((Vs - 8.74) / -7.44))
    q['tau_oi'] = rcp(alpha_oi + beta_oi) / K_Q10
    q['oi_infinity'] = rcp(1.0 + exp((Vs + 33.1) / 5.3))

    alpha_ua = 0.65 * rcp(exp(Vs / -8.5) + exp((Vs - 40.0) / -59.0))
    beta_ua = 0.65 * rcp(2.5 + exp((Vs + 72.0) / 17.0))
    q['tau_ua'] = rcp(alpha_ua + beta_ua) / K_Q10
    q['ua_infinity'] = rcp(1.0 + exp((Vs + 20.3) / -9.6))

    alpha_ui = rcp(21.0 + 1.0 * exp((Vs - 195.000) / -28.0))
    beta_ui = rcp(exp((Vs - 168.0) / -16.0))
    q['tau_ui'] = rcp(alpha_ui + beta_ui) / K_Q10
    q['ui_infinity'] = rcp(1.0 + exp((Vs - 109.45) / 27.48))

    alpha_xr = where(absf(V + 14.1) < 1.0e-10, eps + 0.0015,
                     (0.0003 * (V + 14.1)) / (1.0 - exp((V + 14.1) / -5.0)))
    beta_xr = where(absf(V - 3.3328) < 1.0e-10, eps + 0.000378361,
                    (7.3898e-05 * (V - 3.3328)) / (exp((V - 3.3328) / 5.1237) - 1.0))
    q['tau_xr'] = rcp(alpha_xr + beta_xr)
    q['xr_infinity'] = rcp(1.0 + exp((V + 14.1) / -6.5))

    alpha_xs = where(absf(V - 19.9) < 1.0e-10, eps + 0.00068,
                     (4.0e-05 * (V - 19.9)) / (1.0 - exp((V - 19.9) / -17.0)))
    beta_xs = where(absf(V - 19.9) < 1.0e-10, eps + 0.000315,
                    (3.5e-05 * (V - 19.9)) / (exp((V - 19.9) / 9.0) - 1.0))
    q['tau_xs'] = 0.5 * rcp(alpha_xs + beta_xs)
    q['xs_infinity'] = np.sqrt(rcp(1.0 + exp((V - 19.9) / -12.7)))

    q['g_Kur'] = 0.005 + 0.05 / (1.0 + exp((V - 15.0) / -13.0))
    q['f_NaK'] = rcp(1.0 + 0.1245 * exp((-0.1 * F * V) / (R * T)) +
                     0.0365 * sigma * exp((-F * V) / (R * T)))
    i_NaCad = ((K_mNa * K_mNa * K_mNa + Na_o * Na_o * Na_o) * (K_mCa + Ca_o) *
               (1.0 + K_sat * exp(((gamma_ - 1.0) * V * F) / (R * T))))
    q['i_NaCaa'] = (Cm * I_NaCa_max * (exp((gamma_ * F * V) / (R * T)) * Ca_o)) / i_NaCad
    q['i_NaCab'] = (Cm * I_NaCa_max *
                    (exp(((gamma_ - 1.0) * F * V) / (R * T)) * (Na_o * Na_o * Na_o))) / i_NaCad
    q['i_K1a'] = (Cm * g_K1) / (1.0 + exp(0.07 * (V + 80.0)))
    q['i_Kra'] = (Cm * g_Kr) / (1.0 + exp((V + 15.0) / 22.4))

    if ultra:
        court_us(V, q)
    return q


def court_us(V, q):
    """court_ultra.py:445-450 -- us_infinity and tau_us into the dict q."""
    V_us, K_us = -83.0, 23.0
    alpha_us = 3e-5 * (0.5 * (1 - np.tanh((V - V_us) / K_us)))
    beta_us = 1e-5 * (0.5 * (1 + np.tanh((V - (V_us + 30)) / K_us)))
    q['us_infinity'] = alpha_us / (alpha_us + beta_us)
    q['tau_us'] = np.reciprocal(alpha_us + beta_us)
    return q


# courtemanche.h:105-134 -- the 30 columns of the lookup table, in the header's order (the kernels'
# CourtQ enum and fib_tf_b200._capi.INTER_NAMES[:30])
COURT_LUT_COLUMNS = (
    'd_infinity', 'f_infinity', 'tau_w', 'tau_d', 'tau_f', 'w_infinity', 'm_inf', 'h_inf', 'j_inf',
    'tau_oa', 'tau_oi', 'tau_ua', 'tau_ui', 'tau_xr', 'tau_xs', 'tau_m', 'tau_h', 'tau_j',
    'oa_infinity', 'oi_infinity', 'ua_infinity', 'ui_infinity', 'xr_infinity', 'xs_infinity',
    'g_Kur', 'f_NaK', 'i_NaCaa', 'i_NaCab', 'i_K1a', 'i_Kra')
COURT_LUT_ROWS = 150                   # V = -100 ... 49 mV, 1 mV apart (courtemanche.h:473-479)


def court_lut_table():
    """float32 [150, 30]: row k = court_inter(k - 100) in COURT_LUT_COLUMNS order."""
    q = court_inter(np.arange(COURT_LUT_ROWS, dtype=np.float32) - F32(100))
    return np.stack([np.asarray(q[n], np.float32) for n in COURT_LUT_COLUMNS], axis=1)


def court_lut_row(V):
    """courtemanche.h:354-356 -- row clamp(int(fp32(V) + fp32(100)), 0, 149): the sum is rounded to
    fp32 before it is truncated towards zero (so V = -1e-6 reads row 100).  NaN reads row 0 (the
    device's float-to-int conversion)."""
    s = np.asarray(V, np.float32) + F32(100)
    with np.errstate(invalid='ignore'):
        r = np.clip(np.trunc(np.nan_to_num(s, nan=0.0)), 0, COURT_LUT_ROWS - 1)
    return r.astype(np.intp)


def court_lookup(V, table):
    """The court_inter dict of the 30 tabulated columns, read from `table` [150, 30] at the row of
    the truncating lookup (court_lut_row).  Every array has V's shape."""
    t = np.asarray(table, np.float32)
    if t.shape != (COURT_LUT_ROWS, len(COURT_LUT_COLUMNS)):
        raise ValueError('court_lookup: table shape %r' % (t.shape,))
    rows = t[court_lut_row(V)]
    return {n: rows[..., k] for k, n in enumerate(COURT_LUT_COLUMNS)}


def court_solve(S, dt, diff, phase=None, multirate=True, chronic=True, ultra_slow=False, table=None,
                clip=True):
    """court.py:124-271 -- the full next-state dict S1 from the current state S.
    multirate=True (court.py:118-122): fast states (COURT_FAST) use dt, all others 10*dt.
    multirate=False (court_ultra.py:127-128): every state uses dt.
    table: the LUT flavour -- the 30 tabulated intermediates come from court_lookup(V, table);
    us_infinity / tau_us are still computed directly (the table has no such columns).
    clip=False: the gates are not clipped to [1e-5, 0.99999] (FIB_F_NO_CLIP).
    The caller decides which entries of S1 are assigned (court.py:94-103)."""
    def step_of(name):
        return dt if (not multirate or name in COURT_FAST) else dt * 10

    V = enforce_boundary(S['V'])
    R, T, F, Cm = 8.3143, 310, 96.4867, 100
    g_Na, Na_o, K_o, g_to, g_Ks, g_Ca_L = 7.8, 140, 5.4, 0.1652, 0.12941176, 0.12375
    Km_Na_i, Km_K_o, i_NaK_max, i_CaP_max = 10, 1.5, 0.59933874, 0.275
    g_B_Na, g_B_Ca, g_B_K, Ca_o = 0.0006744375, 0.001131, 0, 1.8
    K_rel, tau_tr, I_up_max, K_up, Ca_up_max = 30, 180, 0.005, 0.00092, 15
    CMDN_max, TRPN_max, CSQN_max = 0.05, 0.07, 10
    Km_CMDN, Km_TRPN, Km_CSQN = 0.00238, 0.0005, 0.8
    V_cell = 20100
    V_i = V_cell * 0.68
    tau_f_Ca, tau_u = 2.0, 8.0
    V_rel = 0.0048 * V_cell
    V_up = 0.0552 * V_cell
    chron = 1.0 if chronic else 0.0
    rcp, exp, log, power, square = np.reciprocal, np.exp, np.log, np.power, np.square

    if table is None:
        q = court_inter(V, ultra=ultra_slow)
    else:                                               # model_court.cuh:386-396
        q = court_lookup(V, table)
        if ultra_slow:
            court_us(V, q)
    N = {}
    # court.py:175-186 -- note _w_ is stepped with the step of '_d_' (court.py:177)
    for g, inf, tau, clock in (
            ('_d_', 'd_infinity', 'tau_d', '_d_'), ('_f_', 'f_infinity', 'tau_f', '_f_'),
            ('_w_', 'w_infinity', 'tau_w', '_d_'), ('_m_', 'm_inf', 'tau_m', '_m_'),
            ('_h_', 'h_inf', 'tau_h', '_h_'), ('_j_', 'j_inf', 'tau_j', '_j_'),
            ('_oa_', 'oa_infinity', 'tau_oa', '_oa_'), ('_oi_', 'oi_infinity', 'tau_oi', '_oi_'),
            ('_ua_', 'ua_infinity', 'tau_ua', '_ua_'), ('_ui_', 'ui_infinity', 'tau_ui', '_ui_'),
            ('_xr_', 'xr_infinity', 'tau_xr', '_xr_'), ('_xs_', 'xs_infinity', 'tau_xs', '_xs_')):
        N[g] = rush_larsen(S[g], q[inf], q[tau], step_of(clock), clip=clip)
    f_Ca_inf = rcp(1.0 + S['_Ca_i_'] / 0.00035)
    N['_f_Ca_'] = rush_larsen(S['_f_Ca_'], f_Ca_inf, tau_f_Ca, step_of('_f_Ca_'), clip=clip)
    if ultra_slow:                                      # court_ultra.py:198-199
        N['_us_'] = rush_larsen(S['_us_'], q['us_infinity'], q['tau_us'], step_of('_us_'), clip=clip)

    E_K = ((R * T) / F) * log(K_o / S['_K_i_'])
    i_K1 = q['i_K1a'] * (V - E_K)
    i_to = (1.0 - 0.5 * chron) * Cm * g_to * power(S['_oa_'], F32(3)) * S['_oi_'] * (V - E_K)
    i_Kur = (1.0 - 0.5 * chron) * Cm * q['g_Kur'] * power(S['_ua_'], F32(3)) * S['_ui_'] * (V - E_K)
    i_Kr = q['i_Kra'] * S['_xr_'] * (V - E_K)
    i_Ks = Cm * g_Ks * square(S['_xs_']) * (V - E_K)
    i_NaK = (((Cm * i_NaK_max * q['f_NaK']) /
              (1.0 + np.sqrt(power(Km_Na_i / S['_Na_i_'], F32(3.0))))) * (K_o / (K_o + Km_K_o)))
    i_B_K = Cm * g_B_K * (V - E_K)
    N['_K_i_'] = S['_K_i_'] + ((2.0 * i_NaK - (i_K1 + i_to + i_Kur + i_Kr + i_Ks + i_B_K)) /
                               (V_i * F)) * step_of('_K_i_')

    E_Na = ((R * T) / F) * log(Na_o / S['_Na_i_'])
    i_Na = Cm * g_Na * power(S['_m_'], F32(3)) * S['_h_'] * S['_j_'] * (V - E_Na)
    if ultra_slow:                                      # court_ultra.py:221-222
        i_Na = i_Na * S['_us_']
    i_NaCa = q['i_NaCaa'] * power(S['_Na_i_'], F32(3)) - q['i_NaCab'] * S['_Ca_i_']
    i_B_Na = Cm * g_B_Na * (V - E_Na)
    N['_Na_i_'] = S['_Na_i_'] + ((-3.0 * i_NaK - (3.0 * i_NaCa + i_B_Na + i_Na)) /
                                 (V_i * F)) * step_of('_Na_i_')

    i_st = 0.0
    i_Ca_L = (1.0 - 0.7 * chron) * Cm * g_Ca_L * S['_d_'] * S['_f_'] * S['_f_Ca_'] * (V - 65.0)
    i_CaP = (Cm * i_CaP_max * S['_Ca_i_']) / (0.0005 + S['_Ca_i_'])
    E_Ca = ((R * T) / (2.0 * F)) * log(Ca_o / S['_Ca_i_'])
    i_B_Ca = Cm * g_B_Ca * (V - E_Ca)
    DV = V + (-(i_Na + i_K1 + i_to + i_Kur + i_Kr + i_Ks + i_B_Na + i_B_Ca + i_NaK + i_CaP +
                i_NaCa + i_Ca_L + i_st) / Cm) * step_of('V')
    N['V'] = DV + diff * step_of('V') * laplace(V, phase)

    i_rel = K_rel * square(S['_u_']) * S['_v_'] * S['_w_'] * (S['_Ca_rel_'] - S['_Ca_i_'])
    i_tr = (S['_Ca_up_'] - S['_Ca_rel_']) / tau_tr
    N['_Ca_rel_'] = S['_Ca_rel_'] + ((i_tr - i_rel) * rcp(
        1.0 + (CSQN_max * Km_CSQN) / square(S['_Ca_rel_'] + Km_CSQN))) * step_of('_Ca_rel_')

    Fn = 1000.0 * (1.0e-15 * V_rel * i_rel - (1.0e-15 / (2.0 * F)) * (0.5 * i_Ca_L - 0.2 * i_NaCa))
    with np.errstate(over='ignore'):
        u_inf = rcp(1.0 + exp(-(Fn - 3.4175e-13) / 1.367e-15))
        N['_u_'] = rush_larsen(S['_u_'], u_inf, tau_u, step_of('_u_'), clip=clip)
        tau_v = 1.91 + 2.09 * u_inf
        v_inf = 1.0 - rcp(1.0 + exp(-(Fn - 6.835e-14) / 1.367e-15))
    N['_v_'] = rush_larsen(S['_v_'], v_inf, tau_v, step_of('_v_'), clip=clip)

    i_up = I_up_max / (1.0 + K_up / S['_Ca_i_'])
    i_up_leak = (I_up_max * S['_Ca_up_']) / Ca_up_max
    N['_Ca_up_'] = S['_Ca_up_'] + (i_up - (i_up_leak + (i_tr * V_rel) / V_up)) * step_of('_Ca_up_')

    B1 = ((2.0 * i_NaCa - (i_CaP + i_Ca_L + i_B_Ca)) / (2.0 * V_i * F) +
          (V_up * (i_up_leak - i_up) + i_rel * V_rel) / V_i)
    B2 = (1.0 + (TRPN_max * Km_TRPN) / square(S['_Ca_i_'] + Km_TRPN) +
          (CMDN_max * Km_CMDN) / square(S['_Ca_i_'] + Km_CMDN))
    N['_Ca_i_'] = S['_Ca_i_'] + (B1 / B2) * step_of('_Ca_i_')
    return N


# --------------------------------------------------------------------------
# the parity metric
# --------------------------------------------------------------------------
def var_floor(kind, name):
    """Absolute floor of the relative-error denominator for one state variable.

    Gates, concentrations and the 4v variables evolve multiplicatively (g += (g - g_inf) * e,
    U ~ 0 at rest), so their fp32 error is relative to their own size: floor = 0.1 % of the
    dynamic range.  The transmembrane voltage of BR / Courtemanche is an ACCUMULATING sum that
    sits at |V| ~ 85 mV most of the time, so every step deposits an absolute rounding error of
    ~ulp(85 mV) = 7.6e-6 mV whatever V's instantaneous value; where V crosses 0 mV a relative
    error against |V| would demand sub-ulp agreement.  Its floor is the voltage range itself."""
    if kind == 'fenton4v':
        return 1e-3
    if kind == 'br':
        return {'V': 120.0, 'C': 1e-3 * 1e-5}.get(name, 1e-3)
    return {'V': 150.0, '_Na_i_': 1e-3 * 11.17, '_K_i_': 1e-3 * 139.0, '_Ca_i_': 1e-3 * 1e-3,
            '_Ca_rel_': 1e-3 * 1.488, '_Ca_up_': 1e-3 * 1.488}.get(name, 1e-3)


def rel_err(got, ref, floor):
    """max |got - ref| / max(|ref|, floor): per-cell relative error with an absolute floor
    (var_floor); the metric of SURVEY.md Appendix B.2.

    Non-finite cells are NOT ignored: the NaN pattern and the infinities of `got` must equal the
    reference's, otherwise the error is +inf (every assertion on it fails)."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    if got.shape != ref.shape:
        raise ValueError('rel_err: shapes %r and %r differ' % (got.shape, ref.shape))
    if got.size == 0:
        return 0.0
    bad_g, bad_r = ~np.isfinite(got), ~np.isfinite(ref)
    if bad_g.any() or bad_r.any():
        same = np.array_equal(np.isnan(got), np.isnan(ref)) and np.array_equal(got[bad_r & ~np.isnan(ref)],
                                                                               ref[bad_r & ~np.isnan(ref)]) \
            and np.array_equal(bad_g, bad_r)
        if not same:
            return float('inf')
        got, ref = got[~bad_r], ref[~bad_r]
        if got.size == 0:
            return 0.0
    return float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), floor)))


PARITY_RTOL = 1e-5      # north_star: 1e-5 relative per step over the first 100 steps
NOISE_FACTOR = 3.0      # waived variables only: never tighter than 3x the reference's own fp32 uncertainty

# The bar is a FLAT 1e-5 for every state variable of every model flavour, except the variables
# named here.  For these the reference's own fp32 result is not defined to 1e-5: the fixtures record,
# per plane, `noise` = how far the UNMODIFIED reference moves when only its fp32 math library is
# swapped for another correctly-rounding one (oracle/tfshim.ALT_LIBM) and `rounding` = its distance
# from the same graph evaluated in float64 (oracle/tfshim.WIDE).  RULE: a variable is waived iff that
# own uncertainty reaches WAIVE_FROM = 0.7e-5 in some fixture of the flavour (the lists below are
# exactly that set; tests/test_oracle_golden.py re-derives them from the fixtures).  A waived variable
# is held to min(cap, max(1e-5, 3 * max(noise, rounding))).  profiles/r2_parity_report.txt lists the
# measured error of every variable of every fixture against the flat bar.
WAIVE_FROM = 0.7e-5
WAIVERS = {
    # degree-8 polynomial gates (br.py:207-252): the S-basis sum d_i 2^(i-1) x^i cancels ~4 digits
    # (|d_i S_i| ~ 1e2 for a result ~1) and tau_h < 0 at rest makes the Rush-Larsen factor blow up
    # into the clip: the reference's own libm swap moves M, H, D by 2-4e-5, its float64 evaluation
    # by 1.2e-4.  The same set applies to config['cheby_strict'] (the reference's operation order):
    # measured there 1.0e-5 ... 4.5e-5 on the fixtures' flavour, i.e. the libm-swap level -- closer
    # than Horner (up to 9.2e-5) but not 1e-5, which no second fp32 implementation can reach.
    'br/cheby': {'vars': ('D', 'H', 'J', 'M', 'XI'), 'cap': 4e-4},
    # exact gates with the multi-rate schedule: D advances with 5 dt in one Rush-Larsen step; the
    # libm swap alone moves the reference by 1.4e-5
    'br/skip': {'vars': ('D',), 'cap': 5e-5},
    # Courtemanche: u and v relax towards 1/(1 + exp(-(Fn - 3.4175e-13)/1.367e-15)) (court.py:241-247),
    # a sigmoid whose argument is a difference of ~1e-13 quantities scaled by 7e14: one ulp of Fn is
    # ~1e-2 in the exponent (own uncertainty 3e-5 ... 1.9e-4); they gate the release current that
    # feeds Ca_rel and Ca_i (8e-6 / 1.1e-5); j advances with 10 dt in the multi-rate split (9.3e-6).
    'court': {'vars': ('_Ca_i_', '_Ca_rel_', '_j_', '_u_', '_v_'), 'cap': 6e-4},
    # all states every step: u as above; w's tau has the removable singularity at 7.9 mV (1.3e-5)
    'court_ultra': {'vars': ('_u_', '_w_'), 'cap': 6e-4},
}


def flavour_of(kind, cfg):
    """Key into WAIVERS for a model kind + config."""
    if kind == 'br':
        if cfg.get('cheby'):
            return 'br/cheby'
        return 'br/skip' if cfg.get('skip') else 'br/exact'
    return kind


def is_waived(kind, cfg, var):
    w = WAIVERS.get(flavour_of(kind, cfg))
    return bool(w) and var in w['vars']


def tolerance(kind, cfg, var, noise=0.0, rounding=0.0):
    """The parity bar (rel_err metric) of one state variable: 1e-5 flat, or -- for the variables
    named in WAIVERS -- min(cap, max(1e-5, 3 * the reference's own uncertainty))."""
    w = WAIVERS.get(flavour_of(kind, cfg))
    if not w or var not in w['vars']:
        return PARITY_RTOL
    return min(w['cap'], max(PARITY_RTOL, NOISE_FACTOR * max(noise, rounding)))


def parity_tolerance(meta, key):
    """Bar for snapshot plane `key` = 's{i}__{var}' of a golden fixture (see tolerance())."""
    var = key.split('__', 1)[1]
    return tolerance(meta['model'], meta['config'], var, meta.get('noise', {}).get(key, 0.0),
                     meta.get('rounding', {}).get(key, 0.0))


def ulp_jitter(state, rng):
    """Moves every cell of every plane by -1, 0 or +1 ulp at random (in place).  Applied after every
    iteration of a second oracle run it models "another fp32 implementation": one ulp of difference
    per variable per iteration.  How far that run drifts from the unperturbed oracle is the model's
    own sensitivity in the scenario at hand -- no implementation can be asked to agree with the oracle
    more closely (live-oracle tests: bar = max(tolerance(), 3 * this drift))."""
    for k, a in state.items():
        d = rng.integers(-1, 2, size=a.shape)
        up = np.nextafter(a, np.float32(np.inf))
        dn = np.nextafter(a, np.float32(-np.inf))
        state[k] = np.where(d > 0, up, np.where(d < 0, dn, a)).astype(np.float32)


def model_uncertainty(metas, kind, cfg, var):
    """Worst (noise, rounding) of `var` over the fixtures of the same flavour: the reference's own
    uncertainty to use where no fixture exists for the exact run (live-oracle tests)."""
    fl = flavour_of(kind, cfg)
    n = r = 0.0
    for meta in metas:
        if flavour_of(meta['model'], meta['config']) != fl:
            continue
        for key, v in meta.get('noise', {}).items():
            if key.split('__', 1)[1] == var:
                n = max(n, v)
        for key, v in meta.get('rounding', {}).items():
            if key.split('__', 1)[1] == var:
                r = max(r, v)
    return n, r


# --------------------------------------------------------------------------
# a small driver with the reference's iteration structure
# --------------------------------------------------------------------------
class OracleModel:
    """Mirrors the reference's define()/add_pace_op()/fire_op()/run()-iteration structure
    (ionic.py:125-245) on top of the step functions above.

    kind: 'fenton4v' | 'br' | 'court' | 'court_ultra'.  One iterate() == one run()
    iteration == dt_per_step time steps (10 / 5 / 1 / 1: fenton.py:135-138, br.py:96-107,
    court.py:92).

    Courtemanche: config['lut'] selects the table flavour (court_lookup), with `table` [150, 30]
    if given and court_lut_table() otherwise; config['chronic'] (default True) the chronic-AF
    remodelling constants."""

    POT = {'fenton4v': 'U', 'br': 'V', 'court': 'V', 'court_ultra': 'V'}
    RANGE = {'fenton4v': (0.0, 1.0), 'br': (-90.0, 30.0), 'court': (-100.0, 50.0),
             'court_ultra': (-100.0, 50.0)}

    def __init__(self, kind, config, table=None):
        self.kind = kind
        self.cfg = dict(config)
        self.height, self.width = config['height'], config['width']
        self.dt, self.diff = config['dt'], config['diff']
        self.phase = None
        self.min_v, self.max_v = self.RANGE[kind]
        self.paces = {}
        self.state = None
        self.coeffs = None
        self.chronic = bool(self.cfg.get('chronic', True))
        self.table = None
        if kind in ('court', 'court_ultra') and self.cfg.get('lut'):
            self.table = np.array(table if table is not None else court_lut_table(), dtype=np.float32)

    def add_hole(self, x, y, radius, neg=False):
        self.phase = hole_phase(self.phase, self.height, self.width, x, y, radius, neg)

    def define(self, s1=True, state=None):
        H, W = self.height, self.width
        if self.kind == 'fenton4v':
            self.state, self.dt_per_step = fenton_init(H, W, s1), 10
        elif self.kind == 'br':
            self.state, self.dt_per_step = br_init(H, W, s1), 5
            if self.cfg.get('cheby'):
                self.coeffs = br_cheby_coeffs()
        else:
            us = self.kind == 'court_ultra' and bool(self.cfg.get('ultra_slow'))
            self.state = ({k: np.array(v, dtype=np.float32) for k, v in state.items()}
                          if state is not None else court_init(H, W, s1, us))
            self.dt_per_step = 1

    def add_pace(self, name, loc, v):
        self.paces[name] = (loc, v)

    def fire(self, name):
        if name == 'slow':
            return self.fire_slow()
        loc, v = self.paces[name]
        k = self.POT[self.kind]
        self.state[k] = apply_pace(self.state[k], loc, v, self.min_v)

    def fire_slow(self):
        """court.py:103 -- assign the 17 slow states from a solve of the CURRENT state."""
        if self.kind != 'court':
            return                              # court_ultra.py:108: 'slow' is an empty group
        new = court_solve(self.state, self.dt, self.diff, self.phase, multirate=True,
                          chronic=self.chronic, table=self.table)
        for k in new:
            if k not in COURT_FAST:
                self.state[k] = new[k]

    def iterate(self):
        c = self.cfg
        if self.kind == 'fenton4v':
            for _ in range(10):
                self.state = fenton_step(self.state, self.dt, self.diff, self.phase)
        elif self.kind == 'br':
            sched = (5, 0, 0, 0, 0) if c.get('skip') else (1, 1, 1, 1, 1)
            for n in sched:
                self.state = br_step(self.state, self.dt, self.diff, n, bool(c.get('cheby')),
                                     self.coeffs, self.phase)
        elif self.kind == 'court':
            new = court_solve(self.state, self.dt, self.diff, self.phase, multirate=True,
                              chronic=self.chronic, table=self.table)
            for k in COURT_FAST:
                self.state[k] = new[k]
        else:
            self.state = court_solve(self.state, self.dt, self.diff, self.phase, multirate=False,
                                     chronic=self.chronic, ultra_slow=bool(c.get('ultra_slow')),
                                     table=self.table)

    def pot(self):
        return self.state[self.POT[self.kind]]

    def image(self):
        """fenton.py:152 / br.py:337-343 / court.py:574-580."""
        if self.kind == 'fenton4v':
            return self.pot().copy()
        return (self.pot() - self.min_v) / (self.max_v - self.min_v)


def run_fixture(meta, on_snapshot=None, model_factory=None):
    """Replay a tests/golden fixture's schedule (see oracle/make_golden.py) on an
    OracleModel-like object.  on_snapshot(i, model) is called for every i in meta['snaps'];
    returns (model, probe_trace)."""
    make = model_factory or OracleModel
    m = make(meta['model'], meta['config'])
    for h in meta['holes']:
        m.add_hole(*h)
    m.define(meta.get('s1', True))
    for (_w, name, loc, v) in meta['paces']:
        m.add_pace(name, loc, v)
    trace = []
    for i in range(meta['samples']):
        m.iterate()
        if meta['slow_every'] and i % meta['slow_every'] == 0:
            m.fire('slow')
        for (when, name, _l, _v) in meta['paces']:
            if i == when:
                m.fire(name)
        if on_snapshot is not None and i in meta['snaps']:
            on_snapshot(i, m)
        if meta['probe']:
            trace.append(m.pot()[meta['probe'][0], meta['probe'][1]])
    return m, np.asarray(trace, dtype=np.float32)
