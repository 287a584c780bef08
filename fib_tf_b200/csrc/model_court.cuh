// model_court.cuh -- Courtemanche-Ramirez-Nattel 1998 atrial model ("chronic AF" variant),
// pointwise part.  Restates court.py:124-271 (solve), :273-429 (calc_inter), :115-122 (euler, dt
// selection), court_ultra.py:81-82,127-128,198-199,221-222,445-450 (all-states-every-step variant
// and the ultra-slow Na inactivation gate) and courtemanche.h:354-357 (truncating LUT lookup).
#pragma once
#include "fib_kernels.cuh"

namespace fib {

constexpr int kLutRows = 150;   // ionic.h:47  TABLE_ROWS
constexpr int kLutCols = 30;    // ionic.h:48  TABLE_COLS
constexpr int kInterCols = 32;  // 30 LUT columns + us_infinity, tau_us
constexpr int kLutTStride = 160;  // row stride of the device-side TRANSPOSED table [30][160]

// column order of courtemanche.h:105-134
enum CourtQ {
  Q_d_inf = 0, Q_f_inf, Q_tau_w, Q_tau_d, Q_tau_f, Q_w_inf, Q_m_inf, Q_h_inf, Q_j_inf, Q_tau_oa,
  Q_tau_oi, Q_tau_ua, Q_tau_ui, Q_tau_xr, Q_tau_xs, Q_tau_m, Q_tau_h, Q_tau_j, Q_oa_inf, Q_oi_inf,
  Q_ua_inf, Q_ui_inf, Q_xr_inf, Q_xs_inf, Q_g_Kur, Q_f_NaK, Q_i_NaCaa, Q_i_NaCab, Q_i_K1a, Q_i_Kra,
  Q_us_inf, Q_tau_us
};

// state planes after V (index in StepArgs::s); same order as the reference's dict (court.py:57-78)
enum CourtS {
  S_Na_i = 0, S_m, S_h, S_j, S_K_i, S_oa, S_oi, S_ua, S_ui, S_xr, S_xs, S_Ca_i, S_d, S_f, S_f_Ca,
  S_Ca_rel, S_u, S_v, S_w, S_Ca_up, S_us, S_COUNT
};

namespace cc {   // constants, folded in double exactly where the reference folds them in Python
constexpr double R = 8.3143, T_K = 310, F = 96.4867, Cm = 100, Na_o = 140, K_o = 5.4, Ca_o = 1.8;
constexpr double g_K1 = 0.09, K_Q10 = 3, g_Kr = 0.029411765, I_NaCa_max = 1600, K_mNa = 87.5;
constexpr double K_mCa = 1.38, K_sat = 0.1, gamma_ = 0.35, sigma = 1.0;
constexpr double g_Na = 7.8, g_to = 0.1652, g_Ks = 0.12941176, g_Ca_L = 0.12375, Km_Na_i = 10;
constexpr double Km_K_o = 1.5, i_NaK_max = 0.59933874, i_CaP_max = 0.275, g_B_Na = 0.0006744375;
constexpr double g_B_Ca = 0.001131, K_rel = 30, tau_tr = 180, I_up_max = 0.005, K_up = 0.00092;
constexpr double Ca_up_max = 15, CMDN_max = 0.05, TRPN_max = 0.07, CSQN_max = 10;
constexpr double Km_CMDN = 0.00238, Km_TRPN = 0.0005, Km_CSQN = 0.8, V_cell = 20100;
constexpr double V_i = V_cell * 0.68, V_rel = 0.0048 * V_cell, V_up = 0.0552 * V_cell;
}  // namespace cc

#define FIB_RCPF(c) ((float)(1.0 / (double)(float)(c)))   /* x / c  ->  x * rcp(fp32(c)) */

// f applied to every lane (libm calls in the rare / optional branches have no packed form)
template <class F> __device__ __forceinline__ float map_lanes(float x, F f) { return f(x); }
template <class F> __device__ __forceinline__ f2 map_lanes(f2 x, F f) { return f2(f(x.x), f(x.y)); }

// calc_inter (court.py:273-429): the V-only intermediates, generic over T = float / f2 (fib_math.cuh).
// eps = V*1e-20 is the reference's broadcast trick (court.py:299); it is kept where it is observable
// (alpha_h, alpha_j).
//
// RATES = false is the reference's table: the Q_tau_* columns hold time constants (the lookup
// table, fib_court_inter).  RATES = true is what the direct (no-table) kernels use: the Q_tau_*
// slots hold 1/tau instead, because the only consumer is expm1(-dt/tau) and every tau here is
// itself 1/(alpha + beta): forming tau and dividing by it again costs two SFU reciprocals per gate
// for nothing.  Where alpha and beta are both fractions the sum goes over the common denominator
// (one reciprocal).  Same formulas in real arithmetic, ~22 of ~130 SFU operations per cell fewer;
// the all-state kernel is SFU-bound (profiles/r1_ncu_summary.txt: xu pipe 75 %).
template <bool WANT_US, bool RATES = false, class T = float>
__device__ __forceinline__ void court_inter_dev(T V, T (&q)[kInterCols]) {
  using namespace cc;
  const T eps = V * 1e-20f;

  // The six removable singularities (tau_d at -10.0001 mV, tau_w at 7.9, alpha/beta of xr at -14.1
  // and 3.3328, of xs at 19.9) are x/(e^y - 1) shapes that the reference guards only at x == 0
  // exactly (court.py:316-327,398-413).  One ulp away y is ~5e-8 and e^y - 1 from the SFU
  // exponential can be exactly 0 with the wrong sign, i.e. a rate of -inf and a gate thrown onto
  // its clip bound -- correctly rounded expf never does that at these magnitudes.  So e^y - 1 comes
  // from the expm1 polynomial when |y| < 0.03 (beyond, e^y - 1 is within 4e-6).  The fix-up sits
  // behind a warp vote because it is rare; each lane's result depends on its own y only.
  const T wd = V + 10.0001f, ww = V - 7.9f, wr = V + 14.1f, zr = V - 3.3328f, ws = V - 19.9f;
  const T y[6] = {wd * -FIB_RCPF(6.24), ww * -0.2f, wr * -0.2f, zr * FIB_RCPF(5.1237),
                  ws * -FIB_RCPF(17.0), ws * FIB_RCPF(9.0)};
  T ey[6], em1[6];
  T ymin = T(1.0f);
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    ey[k] = m_exp(y[k]);
    em1[k] = ey[k] - 1.0f;
    ymin = vmin(ymin, vabs(y[k]));
  }
  if (__any_sync(__activemask(), any_lane(lt(ymin, T(0.03f))))) {
#pragma unroll
    for (int k = 0; k < 6; ++k) em1[k] = sel(lt(vabs(y[k]), T(0.03f)), m_expm1(y[k]), em1[k]);
  }

  q[Q_d_inf] = m_rcp(m_exp_affine((V + 10.0f) * -0.125f, 1.f, 1.0f));
  {
    const T e = ey[0], one_m_e = -em1[0];
    T t = RATES ? m_div((wd * 0.0350000f) * (1.0f + e), one_m_e) : m_div(one_m_e, (wd * 0.0350000f) * (1.0f + e));
    if (any_lane(lt(vabs(wd), T(1.0e-10f)))) {
      const T sp = map_lanes(V, [](float v) {
        return RATES ? (1.0f + expf((v + 10.0f) * -FIB_RCPF(6.24))) / 4.579f
                     : 4.579f / (1.0f + expf((v + 10.0f) * -FIB_RCPF(6.24)));
      });
      t = sel(lt(vabs(wd), T(1.0e-10f)), sp, t);
    }
    q[Q_tau_d] = t;
  }
  {
    const T e = m_exp((V + 28.0f) * -FIB_RCPF(6.9));
    q[Q_f_inf] = m_div(e, 1.0f + e);
  }
  {
    const T a = (V + 10.0f);
    const T x = vfma(T(0.0197000f), m_exp((a * a) * -(0.0337f * 0.0337f)), T(0.02f));
    q[Q_tau_f] = RATES ? x * FIB_RCPF(9.0) : m_rcp(x) * 9.0f;
  }
  {
    const T e = ey[1], one_m_e = -em1[1];
    const T num = vfma(T(0.3f), e, T(1.0f)) * ww;
    T t = RATES ? m_div(num, one_m_e * 6.0f) : m_div(one_m_e * 6.0f, num);
    t = sel(lt(vabs(ww), T(1.0e-10f)), T(RATES ? (float)(1.3 / (6.0 * 0.2)) : (float)((6.0 * 0.2) / 1.3)), t);
    q[Q_tau_w] = t;
  }
  q[Q_w_inf] = 1.0f - m_rcp(m_exp_affine((V - 40.0f) * -FIB_RCPF(17.0), 1.f, 1.0f));
  {
    const T w = V + 47.13f;
    const T alpha_m = sel(lt(vabs(V - -47.13f), T(0.001f)), T(3.2f), m_div(w * 0.32f, 1.0f - m_exp(w * -0.1f)));
    const T beta_m = m_exp(V * -FIB_RCPF(11.0)) * 0.08f;
    const T r = m_rcp(alpha_m + beta_m);
    q[Q_m_inf] = alpha_m * r;
    q[Q_tau_m] = RATES ? alpha_m + beta_m : r;
  }
  // alpha/beta of h and j switch formula at -40 mV (court.py:331-360).  Each exponential slot is
  // evaluated ONCE with the argument of the lane's own branch selected first (same value as
  // evaluating that branch alone, no divergence): 8 exponentials, the cost of the V < -40 side.
  const auto lo = lt(V, T(-40.0f));
  {
    const T alpha_h = sel(lo, m_exp((V + 80.0f) * -FIB_RCPF(6.8)) * 0.135f, eps);
    const T e1 = m_exp(sel(lo, V * 0.079f, (V + 10.66f) * -FIB_RCPF(11.1)));
    const T beta_h = sel(lo, vfma(T(310000.f), m_exp(V * 0.35f), e1 * 3.56f), m_rcp((1.0f + e1) * 0.13f));
    const T r = m_rcp(alpha_h + beta_h);
    q[Q_h_inf] = alpha_h * r;
    q[Q_tau_h] = RATES ? alpha_h + beta_h : r;
  }
  {
    // alpha_j = aN/aD, beta_j = bN/bD
    const T aN = sel(lo, vfma(T(-127140.f), m_exp(V * 0.2444f), m_exp(V * -0.04391f) * -3.474e-05f) * (V + 37.78f),
                     eps);
    const T aD = sel(lo, m_exp_affine((V + 79.23f) * 0.311f, 1.f, 1.0f), T(1.0f));
    const T bN = m_exp(sel(lo, V * -0.01052f, V * -2.535e-07f)) * sel(lo, T(0.1212f), T(0.3f));
    const T bD = m_exp_affine(sel(lo, (V + 40.14f) * -0.1378f, (V + 32.0f) * -0.1f), 1.f, 1.0f);
    if (RATES) {        // over the common denominator: one reciprocal each for inf and rate
      const T x = aN * bD;
      const T t = vfma(bN, aD, x);
      q[Q_j_inf] = x * m_rcp(t);
      q[Q_tau_j] = t * m_rcp(aD * bD);
    } else {
      const T alpha_j = m_div(aN, aD);       // (aD == 1 on the V >= -40 side: alpha_j = eps)
      const T beta_j = m_div(bN, bD);
      const T r = m_rcp(alpha_j + beta_j);
      q[Q_j_inf] = alpha_j * r;
      q[Q_tau_j] = r;
    }
  }
  const T Vs = V - -10.0f;
  {
    // alpha/beta of oa and ua are the same expressions (court.py:363-364, 375-376)
    const T x = m_exp(Vs * -FIB_RCPF(8.5)) + m_exp((Vs - 40.0f) * -FIB_RCPF(59.0));
    const T y2 = m_exp_affine((Vs + 72.0f) * FIB_RCPF(17.0), 1.f, 2.5f);
    T t;
    if (RATES) {      // K_Q10 (0.65/x + 0.65/y) = 1.95 (x + y)/(x y)
      t = ((x + y2) * (float)(3.0 * 0.65)) * m_rcp(x * y2);
    } else {
      const T alpha = m_rcp(x) * 0.65f;
      const T beta = m_rcp(y2) * 0.65f;
      t = m_rcp(alpha + beta) * FIB_RCPF(3.0);
    }
    q[Q_tau_oa] = t;
    q[Q_tau_ua] = t;
  }
  q[Q_oa_inf] = m_rcp(m_exp_affine((Vs + 10.47f) * -FIB_RCPF(17.54), 1.f, 1.0f));
  {
    const T x = m_exp_affine((Vs + 103.7f) * FIB_RCPF(10.95), 1.f, 18.53f);
    const T y2 = m_exp_affine((Vs - 8.74f) * -FIB_RCPF(7.44), 1.f, 35.56f);
    if (RATES) q[Q_tau_oi] = ((x + y2) * 3.0f) * m_rcp(x * y2);
    else q[Q_tau_oi] = m_rcp(m_rcp(x) + m_rcp(y2)) * FIB_RCPF(3.0);
  }
  q[Q_oi_inf] = m_rcp(m_exp_affine((Vs + 33.1f) * FIB_RCPF(5.3), 1.f, 1.0f));
  q[Q_ua_inf] = m_rcp(m_exp_affine((Vs + 20.3f) * -FIB_RCPF(9.6), 1.f, 1.0f));
  {
    const T alpha = m_rcp(m_exp_affine((Vs - 195.000f) * -FIB_RCPF(28.0), 1.f, 21.0f));
    const T beta = m_exp((Vs - 168.0f) * 0.0625f);          // 1 / e^{-z} = e^{z}
    q[Q_tau_ui] = RATES ? (alpha + beta) * 3.0f : m_rcp(alpha + beta) * FIB_RCPF(3.0);
  }
  q[Q_ui_inf] = m_rcp(m_exp_affine((Vs - 109.45f) * FIB_RCPF(27.48), 1.f, 1.0f));
  {
    const auto sw = lt(vabs(wr), T(1.0e-10f)), sz = lt(vabs(zr), T(1.0e-10f));
    const T aN = sel(sw, T(0.0015f), wr * 0.0003f), aD = sel(sw, T(1.0f), -em1[2]);    // 1 - e^{-0.2 w}
    const T bN = sel(sz, T(0.000378361f), zr * 7.3898e-05f);
    const T bD = sel(sz, T(1.0f), em1[3]);                                       // e^{z/5.1237} - 1
    if (RATES) q[Q_tau_xr] = vfma(aN, bD, bN * aD) * m_rcp(aD * bD);
    else q[Q_tau_xr] = m_rcp(m_div(aN, aD) + m_div(bN, bD));
    q[Q_xr_inf] = m_rcp(m_exp_affine(wr * -FIB_RCPF(6.5), 1.f, 1.0f));
  }
  {
    const auto z0 = lt(vabs(ws), T(1.0e-10f));
    const T aN = sel(z0, T(0.00068f), ws * 4.0e-05f), aD = sel(z0, T(1.0f), -em1[4]);   // 1 - e^{-w/17}
    const T bN = sel(z0, T(0.000315f), ws * 3.5e-05f), bD = sel(z0, T(1.0f), em1[5]);    // e^{w/9} - 1
    if (RATES) q[Q_tau_xs] = (vfma(aN, bD, bN * aD) * 2.0f) * m_rcp(aD * bD);
    else q[Q_tau_xs] = m_rcp(m_div(aN, aD) + m_div(bN, bD)) * 0.5f;
    q[Q_xs_inf] = m_sqrt(m_rcp(m_exp_affine(ws * -FIB_RCPF(12.7), 1.f, 1.0f)));
  }
  q[Q_g_Kur] = vfma(T(0.05f), m_rcp(m_exp_affine((V - 15.0f) * -FIB_RCPF(13.0), 1.f, 1.0f)), T(0.005f));
  {
    constexpr float rRT = FIB_RCPF(R * T_K);
    q[Q_f_NaK] = m_rcp(vfma(T((float)(0.0365 * sigma)), m_exp((V * (float)(-F)) * rRT),
                            vfma(T(0.1245f), m_exp((V * (float)(-0.1 * F)) * rRT), T(1.0f))));
    const T eg1 = m_exp(((V * (float)(gamma_ - 1.0)) * (float)F) * rRT);
    const T rd = m_rcp(vfma(T((float)K_sat), eg1, T(1.0f)) *
                       (float)((K_mNa * K_mNa * K_mNa + Na_o * Na_o * Na_o) * (K_mCa + Ca_o)));
    q[Q_i_NaCaa] = ((m_exp((V * (float)(gamma_ * F)) * rRT) * (float)Ca_o) * (float)(Cm * I_NaCa_max)) * rd;
    // e^{(gamma-1) F V / RT} is eg1 again (court.py:421 vs :417 differ only in operand order)
    q[Q_i_NaCab] = ((eg1 * (float)(Na_o * Na_o * Na_o)) * (float)(Cm * I_NaCa_max)) * rd;
  }
  q[Q_i_K1a] = m_rcp(m_exp_affine((V + 80.0f) * 0.07f, 1.f, 1.0f)) * (float)(Cm * g_K1);
  q[Q_i_Kra] = m_rcp(m_exp_affine((V + 15.0f) * FIB_RCPF(22.4), 1.f, 1.0f)) * (float)(Cm * g_Kr);
  if (WANT_US) {   // court_ultra.py:445-450
    const T a_us = map_lanes(V, [](float v) { return 3e-5f * (0.5f * (1.f - tanhf((v - -83.0f) * FIB_RCPF(23.0)))); });
    const T b_us = map_lanes(V, [](float v) {
      return 1e-5f * (0.5f * (1.f + tanhf((v - (float)(-83.0 + 30)) * FIB_RCPF(23.0))));
    });
    const T r = m_rcp(a_us + b_us);
    q[Q_us_inf] = a_us * r;
    q[Q_tau_us] = RATES ? a_us + b_us : r;
  } else {
    q[Q_us_inf] = T(0.f);
    q[Q_tau_us] = T(1.f);
  }
}

enum CourtMode {
  COURT_FAST = 0,   // court.py:94-102  _ode_op: assign V, _Na_i_, _m_, _h_ (step dt)
  COURT_SLOW = 1,   // court.py:103     'slow':  assign the other 17 (step 10*dt), no stencil
  COURT_ALL = 2     // court_ultra.py:107-111: assign everything, step dt
};

template <int MODE, bool LUT, bool US>
struct Courtemanche {
  static constexpr int NS = S_COUNT;      // 21 slots; S_us only used when US
  // cells per thread / resident CTAs per SM / packed pairs per kernel flavour, measured on B200 (4096^2,
  // Gcell-steps/s; profiles/r2_tuning_log.md):
  //   fast op   2 scalar cells @8 CTAs 78.3 (packed pair @6/8/10: 73.5 / 75.2 / 55.7: HBM-bound, packing only
  //             costs registers)
  //   all-state 1 cell @8 CTAs 28.0 -> packed pair @4 CTAs 32.7 -> @5 CTAs 34.8 (89 % of the 168-B roofline)
  //   LUT       packed pair @4/5/6 CTAs 32.2 / 33.1 / 31.1; 2 scalar cells @4 CTAs 34.1 -> @5 CTAs 36.6 (94 %):
  //             the table flavour is load-bound (60 table reads per pair), the pair registers do not pay
  static constexpr int VEC = 2;
  static constexpr int VEC_SMALL = 1;   // cells per thread on small grids (kSmallGridCells)
  static constexpr int BY = 4;
  static constexpr int MAX_R = LUT ? 2 : 1;
  static constexpr int AUTO_R = LUT ? 2 : 1;   // marching depth picked by launch_step (measured best)
  static constexpr int MIN_BLOCKS = MODE == COURT_FAST ? 8 : 5;
  // the one-cell-per-thread flavour of the direct all-state kernel (small grids) keeps 8 CTAs per SM
  static __host__ __device__ constexpr int min_blocks(int vec, bool /*phase*/) {
    return (MODE == COURT_ALL && !LUT && vec == 1) ? 8 : MIN_BLOCKS;
  }
  static constexpr bool PACKED = MODE != COURT_FAST && !LUT;
  static constexpr bool PREFETCH = false;
  static constexpr bool NEED_RAW = false; // V = enforce_boundary(V0) everywhere (court.py:126-127)
  static constexpr bool NEED_LAP = MODE != COURT_SLOW;
  static constexpr bool STORE_X = MODE != COURT_SLOW;
  static __host__ __device__ constexpr bool is_fast(int k) { return k == S_Na_i || k == S_m || k == S_h; }
  static __host__ __device__ constexpr bool stores(int k) {
    return (k == S_us) ? (US && MODE != COURT_FAST)
                       : (MODE == COURT_ALL ? true : (MODE == COURT_FAST ? is_fast(k) : !is_fast(k)));
  }
  static const char* name() {
    static const char* n[3][2][2] = {
        {{"Courtemanche<fast>", "Courtemanche<fast,us>"}, {"Courtemanche<fast,lut>", "Courtemanche<fast,lut,us>"}},
        {{"Courtemanche<slow>", "Courtemanche<slow,us>"}, {"Courtemanche<slow,lut>", "Courtemanche<slow,lut,us>"}},
        {{"Courtemanche<all>", "Courtemanche<all,us>"}, {"Courtemanche<all,lut>", "Courtemanche<all,lut,us>"}}};
    return n[MODE][LUT ? 1 : 0][US ? 1 : 0];
  }
  struct Params {
    float dt_fast, neg_dt_fast;   // V, _Na_i_, _m_, _h_        (court.py:118-120)
    float dt_slow, neg_dt_slow;   // everything else: 10*dt for court.py, dt for court_ultra.py
    float ddt;                    // fp32(diff * dt_fast)        (court.py:229)
    float e_fCa;                  // expm1(fp32(-dt_x / 2.0)), Python-scalar tau (court.py:189)
    float e_u;                    // expm1(fp32(-dt_x / 8.0))                    (court.py:243)
    float clip_lo, clip_hi;       // gate clip: (1e-5, 0.99999) (ionic.py:122-123) or (-inf, +inf)
    float k_to, k_Kur, k_CaL;     // (1-0.5c)*Cm*g_to, (1-0.5c)*Cm, (1-0.7c)*Cm*g_Ca_L folded in double
                                  // on the host like the reference's Python (court.py:193-194,218)
  };

  // rush_larsen_b with t = tau (table flavours) or t = 1/tau (direct flavours)
  template <class T>
  static __device__ __forceinline__ T gate(T g, T g_inf, T t, float neg_dt, const Params& p) {
    const T e = m_expm1_neg(LUT ? m_div(T(neg_dt), t) : t * neg_dt);
    return rush_larsen_eb(g, g_inf, e, p.clip_lo, p.clip_hi);
  }

  // courtemanche.h:354-356: row of the truncating lookup
  static __device__ __forceinline__ int lut_row(float V) {
    int i = static_cast<int>(V + 100.f);
    return i < 0 ? 0 : (i >= kLutRows ? kLutRows - 1 : i);
  }
  // Where the table lives: the transposed copy [30][160] (19 KB) in global memory, read through L1
  // with ld.global.nc -- it stays L1-resident (every CTA of every wave reads the same 19 KB) and costs
  // no shared memory, so five CTAs per SM keep all of L1 (measured against a shared-memory copy on
  // B200, profiles/r2_tuning_log.md).
  static __device__ __forceinline__ void lut_fetch(const float* lut, float V, float (&q)[kInterCols]) {
    const float* col = lut + lut_row(V);
#pragma unroll
    for (int k = 0; k < kLutCols; ++k) q[k] = __ldg(col + k * kLutTStride);
  }
  static __device__ __forceinline__ void lut_fetch(const float* lut, f2 V, f2 (&q)[kInterCols]) {
    const float* c0 = lut + lut_row(V.x);
    const float* c1 = lut + lut_row(V.y);
#pragma unroll
    for (int k = 0; k < kLutCols; ++k) q[k] = f2(__ldg(c0 + k * kLutTStride), __ldg(c1 + k * kLutTStride));
  }

  // A: StepArgs<Courtemanche> or StepArgsZ<Courtemanche> (fib_kernels.cuh)
  template <class A, class T>
  static __device__ __forceinline__ void cell(const A& a, T /*raw*/, T V, T lap,
                                              T (&s)[NS], T& Vnew) {
    using namespace cc;
    const Params& p = a.p;
    T q[kInterCols];
    if (LUT) {
      // The table is kept TRANSPOSED on the device ([column][voltage], 19 KB, L1-resident): the
      // lanes of a warp sit within a few mV of each other, so each of the 30 column reads touches
      // one or two 128-B lines instead of one line per distinct voltage row.
      lut_fetch(a.lut, V, q);
      if (US) {
        T qq[kInterCols];
        court_inter_dev<true, false>(V, qq);                // not tabulated in the reference
        q[Q_us_inf] = qq[Q_us_inf];
        q[Q_tau_us] = qq[Q_tau_us];
      }
    } else {
      court_inter_dev<US, true>(V, q);                // Q_tau_* hold 1/tau
    }
    const float ndf = p.neg_dt_fast, nds = p.neg_dt_slow, dtf = p.dt_fast, dts = p.dt_slow;
    const T Na_i = s[S_Na_i], K_i = s[S_K_i], Ca_i = s[S_Ca_i], Ca_rel = s[S_Ca_rel], Ca_up = s[S_Ca_up];
    const T m = s[S_m], h = s[S_h], j = s[S_j], oa = s[S_oa], oi = s[S_oi], ua = s[S_ua],
            ui = s[S_ui], xr = s[S_xr], xs = s[S_xs], d = s[S_d], f = s[S_f], f_Ca = s[S_f_Ca],
            u = s[S_u], v = s[S_v], w = s[S_w];

    // gates (court.py:175-189); _w_ is clocked with the step of '_d_' (court.py:177) = slow.
    // `gate` takes tau from the table and 1/tau from the direct evaluation (court_inter_dev).
    s[S_d] = gate(d, q[Q_d_inf], q[Q_tau_d], nds, p);
    s[S_f] = gate(f, q[Q_f_inf], q[Q_tau_f], nds, p);
    s[S_w] = gate(w, q[Q_w_inf], q[Q_tau_w], nds, p);
    s[S_m] = gate(m, q[Q_m_inf], q[Q_tau_m], ndf, p);
    s[S_h] = gate(h, q[Q_h_inf], q[Q_tau_h], ndf, p);
    s[S_j] = gate(j, q[Q_j_inf], q[Q_tau_j], nds, p);
    s[S_oa] = gate(oa, q[Q_oa_inf], q[Q_tau_oa], nds, p);
    s[S_oi] = gate(oi, q[Q_oi_inf], q[Q_tau_oi], nds, p);
    s[S_ua] = gate(ua, q[Q_ua_inf], q[Q_tau_ua], nds, p);
    s[S_ui] = gate(ui, q[Q_ui_inf], q[Q_tau_ui], nds, p);
    s[S_xr] = gate(xr, q[Q_xr_inf], q[Q_tau_xr], nds, p);
    s[S_xs] = gate(xs, q[Q_xs_inf], q[Q_tau_xs], nds, p);
    const T f_Ca_inf = m_rcp(vfma(Ca_i, T(FIB_RCPF(0.00035)), T(1.0f)));
    s[S_f_Ca] = rush_larsen_eb(f_Ca, f_Ca_inf, T(p.e_fCa), p.clip_lo, p.clip_hi);
    T us = T(1.f);
    if (US) {
      us = s[S_us];
      s[S_us] = gate(us, q[Q_us_inf], q[Q_tau_us], nds, p);   // court_ultra.py:198-199
    }

    // currents (court.py:191-221)
    constexpr float RTF = (float)((R * T_K) / F);
    const T E_K = m_log(m_div((float)K_o, K_i)) * RTF;
    const T dVK = V - E_K;
    const T i_K1 = q[Q_i_K1a] * dVK;
    const T i_to = (oa * oa * oa) * p.k_to * oi * dVK;
    const T i_Kur = q[Q_g_Kur] * p.k_Kur * (ua * ua * ua) * ui * dVK;
    const T i_Kr = q[Q_i_Kra] * xr * dVK;
    const T i_Ks = (xs * xs) * (float)(Cm * g_Ks) * dVK;
    const T r_na = m_div((float)Km_Na_i, Na_i);
    const T i_NaK = m_div(q[Q_f_NaK] * (float)(Cm * i_NaK_max), 1.0f + m_sqrt(r_na * r_na * r_na)) *
                    (float)(K_o / (K_o + Km_K_o));
    // i_B_K = Cm * g_B_K * (V - E_K) with g_B_K = 0 (court.py:198): contributes +0
    const T i_Ksum = i_K1 + i_to + i_Kur + i_Kr + i_Ks;
    s[S_K_i] = vfma(vfma(T(2.0f), i_NaK, -i_Ksum) * FIB_RCPF(V_i * F), T(dts), K_i);

    const T E_Na = m_log(m_div((float)Na_o, Na_i)) * RTF;
    const T dVNa = V - E_Na;
    T i_Na = (m * m * m) * (float)(Cm * g_Na) * h * j * dVNa;
    if (US) i_Na = i_Na * us;                                      // court_ultra.py:221-222
    const T i_NaCa = vfma(q[Q_i_NaCaa], Na_i * Na_i * Na_i, -(q[Q_i_NaCab] * Ca_i));
    const T i_B_Na = dVNa * (float)(Cm * g_B_Na);
    s[S_Na_i] = vfma(vfma(T(-3.0f), i_NaK, -(vfma(T(3.0f), i_NaCa, i_B_Na) + i_Na)) * FIB_RCPF(V_i * F), T(dtf),
                     Na_i);

    const T i_Ca_L = d * p.k_CaL * f * f_Ca * (V - 65.0f);
    const T i_CaP = m_div(Ca_i * (float)(Cm * i_CaP_max), 0.0005f + Ca_i);
    const T E_Ca = m_log(m_div((float)Ca_o, Ca_i)) * (float)((R * T_K) / (2.0 * F));
    const T i_B_Ca = (V - E_Ca) * (float)(Cm * g_B_Ca);
    const T I_tot = i_Na + i_K1 + i_to + i_Kur + i_Kr + i_Ks + i_B_Na + i_B_Ca + i_NaK + i_CaP + i_NaCa + i_Ca_L;
    // reference rounding sequence, no FMA contraction (V crosses 0 mV with ~80 mV operands)
    const T DV = add_rn(V, mul_rn(div_rn(-I_tot, T((float)Cm)), T(dtf)));       // court.py:223-227
    Vnew = add_rn(DV, mul_rn(T(ddt_of(a)), lap));                                    // court.py:229

    // Ca handling (court.py:232-265)
    const T i_rel = (u * u) * (float)K_rel * v * w * (Ca_rel - Ca_i);
    const T i_tr = (Ca_up - Ca_rel) * FIB_RCPF(tau_tr);
    {
      const T z = Ca_rel + (float)Km_CSQN;
      s[S_Ca_rel] = vfma((i_tr - i_rel) * m_rcp(1.0f + m_div((float)(CSQN_max * Km_CSQN), z * z)), T(dts), Ca_rel);
    }
    const T Fn = vfma(T((float)(1.0e-15 * V_rel)), i_rel,
                      -(vfma(T(0.5f), i_Ca_L, -(i_NaCa * 0.2f)) * (float)(1.0e-15 / (2.0 * F)))) * 1000.0f;
    const T u_inf = m_rcp(m_exp_affine((Fn - 3.4175e-13f) * -FIB_RCPF(1.367e-15), 1.f, 1.0f));
    s[S_u] = rush_larsen_eb(u, u_inf, T(p.e_u), p.clip_lo, p.clip_hi);
    const T tau_v = vfma(T(2.09f), u_inf, T(1.91f));
    const T v_inf = 1.0f - m_rcp(m_exp_affine((Fn - 6.835e-14f) * -FIB_RCPF(1.367e-15), 1.f, 1.0f));
    s[S_v] = rush_larsen_b(v, v_inf, tau_v, nds, p.clip_lo, p.clip_hi);
    const T i_up = m_rcp(1.0f + m_div((float)K_up, Ca_i)) * (float)I_up_max;
    const T i_up_leak = (Ca_up * (float)I_up_max) * FIB_RCPF(Ca_up_max);
    s[S_Ca_up] = vfma(i_up - vfma(i_tr * (float)V_rel, T(FIB_RCPF(V_up)), i_up_leak), T(dts), Ca_up);
    const T B1 = vfma(vfma(T(2.0f), i_NaCa, -(i_CaP + i_Ca_L + i_B_Ca)), T(FIB_RCPF(2.0 * V_i * F)),
                      vfma(T((float)V_up), i_up_leak - i_up, i_rel * (float)V_rel) * FIB_RCPF(V_i));
    const T zt = Ca_i + (float)Km_TRPN, zc = Ca_i + (float)Km_CMDN;
    const T B2 = 1.0f + m_div((float)(TRPN_max * Km_TRPN), zt * zt) + m_div((float)(CMDN_max * Km_CMDN), zc * zc);
    s[S_Ca_i] = vfma(m_div(B1, B2), T(dts), Ca_i);
  }
};

}  // namespace fib
