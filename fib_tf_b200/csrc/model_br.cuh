// model_br.cuh -- modified 8-variable Beeler-Reuter model, pointwise part.
// Restates br.py:125-173 (solve), :175-205 (exact gates), :207-252 (Chebyshev gates),
// :255-273 (alpha/beta), :289-331 (scaled-monomial expansion), coefficients br.py:49-62.
//
// Instruction budget (this kernel is issue-bound, not HBM-bound): see fib_math.cuh.  The cell is
// written once, generic over T = float (one cell per thread, small grids) and T = f2 (two cells per
// thread, every multiply-add a packed FFMA2 / FMUL2 / FADD2).  Beyond the few-ulp transcendental
// layer two algebraic identities are used, both exact in real arithmetic:
//   * the six current exponentials of br.py:150-157 are all e^{0.04 V0} times a constant;
//   * r = d0 + sum d_i S_i with S_i = 2^{i-1} x^i is the ordinary polynomial sum c_i x^i,
//     c_i = d_i 2^{i-1} (exact scaling), evaluated by Horner's scheme with FMAs (8 per gate
//     function).  This is MORE accurate than the reference's left-to-right
//     fp32 sum in the ill-conditioned S basis; the two differ by the reference's own rounding
//     error (recorded in the fixtures as meta['rounding']).  config['cheby_strict'] selects the
//     reference's own operation order instead (CHEBY == 2 below).
#pragma once
#include "fib_kernels.cuh"

namespace fib {

// (c0 e^{c1(v+c2)} + c3 (v+c4)) / (e^{c5(v+c2)} + c6)  -- br.py:255-264.  Called with literal
// coefficients only, so every `== 0` test below folds at compile time (exp(0) == 1 exactly).
// Scalar: the readable statement of the exact gates, checked against float64 by the math-layer tests.
__device__ __forceinline__ float br_rate(float v, float c0, float c1, float c2, float c3, float c4,
                                         float c5, float c6) {
  const float e_num = (c1 == 0.f) ? 1.f : m_exp(c1 * (v + c2));
  float num = (c0 == 0.f) ? 0.f : c0 * e_num;
  if (c3 != 0.f) num = (c0 == 0.f) ? c3 * (v + c4) : num + c3 * (v + c4);
  if (c5 == 0.f) return num * (1.0f / (1.0f + c6));
  // e^z - 1 (alpha_m, removable singularity at -47 mV) goes through expm1
  if (c6 == -1.f) return m_div(num, m_expm1(c5 * (v + c2)));
  return m_div(num, m_exp(c5 * (v + c2)) + c6);
}

// gate order: 0 xi, 1 m, 2 h, 3 j, 4 d, 5 f  (br.py:285-286); d/f rates doubled (br.py:46-48).
// Returns inf = a/(a+b) and rate = a+b = 1/tau (br.py:266-273).
template <int G>
__device__ __forceinline__ void br_inf_rate_exact(float v, float& inf, float& rate) {
  float a, b;
  if (G == 0) { a = br_rate(v, 0.0005f, 0.083f, 50.f, 0.f, 0.f, 0.057f, 1.f);
                b = br_rate(v, 0.0013f, -0.06f, 20.f, 0.f, 0.f, -0.04f, 1.f); }
  if (G == 1) { a = br_rate(v, 0.f, 0.f, 47.f, -1.f, 47.f, -0.1f, -1.f);
                b = br_rate(v, 40.f, -0.056f, 72.f, 0.f, 0.f, 0.f, 0.f); }
  if (G == 2) { a = br_rate(v, 0.126f, -.25f, 77.f, 0.f, 0.f, 0.f, 0.f);
                b = br_rate(v, 1.7f, 0.f, 22.5f, 0.f, 0.f, -0.082f, 1.f); }
  if (G == 3) { a = br_rate(v, 0.055f, -.25f, 78.f, 0.f, 0.f, -0.2f, 1.f);
                b = br_rate(v, 0.3f, 0.f, 32.f, 0.f, 0.f, -0.1f, 1.f); }
  if (G == 4) { a = br_rate(v, (float)(2 * 0.095), -0.01f, -5.f, 0.f, 0.f, -0.072f, 1.f);
                b = br_rate(v, (float)(2 * 0.07), -0.017f, 44.f, 0.f, 0.f, 0.05f, 1.f); }
  if (G == 5) { a = br_rate(v, (float)(2 * 0.012), -0.008f, 28.f, 0.f, 0.f, 0.15f, 1.f);
                b = br_rate(v, (float)(2 * 0.0065), -0.02f, 30.f, 0.f, 0.f, -0.2f, 1.f); }
  rate = a + b;
  inf = m_div(a, rate);
}

// rush_larsen with tau given as its reciprocal: expm1(-dt/tau) = expm1(-dt * rate)
template <class T> __device__ __forceinline__ T rush_larsen_rate(T g, T g_inf, T rate, float neg_dt) {
  return rush_larsen_e(g, g_inf, m_expm1_neg(T(neg_dt) * rate));
}

// a = n1/d1, b = n2/d2 (all four positive): rate = a + b = (n1 d2 + n2 d1)/(d1 d2) and
// inf = a/rate = n1 d2/(n1 d2 + n2 d1) -- two SFU reciprocals instead of three, no cancellation.
template <class T>
__device__ __forceinline__ T rush_larsen_frac(T g, T n1, T d1, T n2, T d2, float neg_dt) {
  const T n1d2 = n1 * d2;
  const T N = vfma(n2, d1, n1d2);
  const T rate = N * m_rcp(d1 * d2);
  return rush_larsen_rate(g, n1d2 * m_rcp(N), rate, neg_dt);
}

// The exact gates of br.py:175-205 / 255-273 for one cell (or a pair), same formulas as
// br_inf_rate_exact (which stays as the readable statement), with the SFU work trimmed -- the
// exact-gate kernel is MUFU-bound (~47 SFU ops per cell): exponentials that differ only by a
// constant factor are computed once
//   e^{-0.25(v+78)} = e^{-0.25(v+77)} e^{-0.25}          (alpha_j <- alpha_h)
//   e^{-0.2(v+30)}  = e^{-0.2(v+78)} e^{9.6}              (beta_f  <- alpha_j)
//   e^{-0.1(v+32)}  = e^{-0.1(v+47)} e^{1.5}              (beta_j  <- alpha_m)
//   e^{-0.04(v+20)} = e^{-0.8} / e^{0.04 v}                (beta_xi <- the currents' k)
// and the two-fraction gates use rush_larsen_frac.  m and h keep the reference's operation
// structure, so V0 == -47.0f still yields the reference's 0/0 -> clip upper bound (fib_common.cuh).
template <bool SLOW, class T>
__device__ __forceinline__ void br_gates_exact(T v, T rk, T (&s)[7], float neg_dt, float neg_dt_slow) {
  // m: a = -(v+47)/expm1(-0.1(v+47)), b = 40 e^{-0.056(v+72)}
  const T v47 = v + T(47.f);
  const T zm = T(-0.1f) * v47;
  const T E10 = m_exp(zm);
  {
    const T den = sel(lt(vabs(zm), T(0.125f)), expm1_poly(zm), E10 - T(1.0f));   // m_expm1 with its exponential kept
    const T a = m_div(-v47, den);
    const T b = m_exp_affine(T(-0.056f) * (v + T(72.f)), 40.f, 0.f);
    const T rate = a + b;
    s[1] = rush_larsen_rate(s[1], m_div(a, rate), rate, neg_dt);
  }
  // h: a = 0.126 e^{-0.25(v+77)}, b = 1.7/(e^{-0.082(v+22.5)} + 1)
  const T E25 = m_exp(T(-.25f) * (v + T(77.f)));
  {
    const T a = T(0.126f) * E25;
    const T b = m_div(1.7f, m_exp_affine(T(-0.082f) * (v + T(22.5f)), 1.f, 1.f));
    const T rate = a + b;
    s[2] = rush_larsen_rate(s[2], m_div(a, rate), rate, neg_dt);
  }
  if (SLOW) {
    // j: a = 0.055 e^{-0.25(v+78)}/(e^{-0.2(v+78)} + 1), b = 0.3/(e^{-0.1(v+32)} + 1)
    const T E20 = m_exp(T(-0.2f) * (v + T(78.f)));
    s[3] = rush_larsen_frac(s[3], E25 * T(0.055f * 0.7788007830714049f), E20 + T(1.f), T(0.3f),
                            vfma(E10, T(4.4816890703380645f), T(1.f)), neg_dt_slow);
    // d (rates doubled, br.py:46-48): a = 0.19 e^{-0.01(v-5)}/(e^{-0.072(v-5)} + 1),
    //                                 b = 0.14 e^{-0.017(v+44)}/(e^{0.05(v+44)} + 1)
    const T v5 = v - T(5.f), v44 = v + T(44.f), v28 = v + T(28.f), v50 = v + T(50.f);
    s[4] = rush_larsen_frac(s[4], m_exp_affine(T(-0.01f) * v5, (float)(2 * 0.095), 0.f),
                            m_exp_affine(T(-0.072f) * v5, 1.f, 1.f),
                            m_exp_affine(T(-0.017f) * v44, (float)(2 * 0.07), 0.f),
                            m_exp_affine(T(0.05f) * v44, 1.f, 1.f), neg_dt_slow);
    // f (doubled): a = 0.024 e^{-0.008(v+28)}/(e^{0.15(v+28)} + 1),
    //              b = 0.013 e^{-0.02(v+30)}/(e^{-0.2(v+30)} + 1)
    s[5] = rush_larsen_frac(s[5], m_exp_affine(T(-0.008f) * v28, (float)(2 * 0.012), 0.f),
                            m_exp_affine(T(0.15f) * v28, 1.f, 1.f),
                            m_exp_affine(T(-0.02f) * (v + T(30.f)), (float)(2 * 0.0065), 0.f),
                            vfma(E20, T(14764.781565577266f), T(1.f)), neg_dt_slow);
    // xi: a = 0.0005 e^{0.083(v+50)}/(e^{0.057(v+50)} + 1), b = 0.0013 e^{-0.06(v+20)}/(e^{-0.04(v+20)} + 1)
    s[6] = rush_larsen_frac(s[6], m_exp_affine(T(0.083f) * v50, 0.0005f, 0.f),
                            m_exp_affine(T(0.057f) * v50, 1.f, 1.f),
                            m_exp_affine(T(-0.06f) * (v + T(20.f)), 0.0013f, 0.f),
                            vfma(rk, T(0.44932896411722156f), T(1.f)), neg_dt_slow);
  }
}
// rush_larsen with the argument-compensated expm1 (same result class, three instructions longer)
template <class T> __device__ __forceinline__ T rush_larsen_comp(T g, T g_inf, T tau, float neg_dt) {
  const T e = m_expm1(m_div(T(neg_dt), tau));
  return clip_tf(vfma(g - g_inf, e, g), 0.00001f, 0.99999f);
}
// Horner evaluation of c0 + c1 x + ... + c8 x^8.  Every FMA takes its coefficient straight from the
// kernel parameter bank (scalar: a constant-bank operand; packed: a uniform register broadcast to
// both lanes), so no per-thread register holds a coefficient; Estrin's scheme was measured slower
// because its two-constant FMAs saturate the ADU pipe with constant loads.  The 12 gate functions
// are independent chains, which is all the ILP the scheduler needs.
template <class T> __device__ __forceinline__ T br_poly8(const float* __restrict__ c, T x) {
  T r = T(c[8]);
#pragma unroll
  for (int i = 7; i >= 0; --i) r = vfma(r, x, T(c[i]));
  return r;
}

// strict-order evaluation of the reference's polynomial gates (br.py:215, 289-301, 327-331): x by an
// fp32 DIVISION, S_i = (2x) S_{i-1}, r = d_0 + d_1 S_1 + ... left to right with one rounding per
// multiply and per add (no FMA), then ionic.py:115-123 with IEEE division, libm expm1f and unfused
// multiply / add (rush_larsen_strict).  d = the fp32-rounded table coefficients, unscaled.  This is
// the reference's own operation sequence; the only thing left to differ is the last bit of expm1f
// (CUDA libm vs glibc).
template <class T> __device__ __forceinline__ T br_strict_eval(const float* __restrict__ d, const T (&S)[9]) {
  T r = add_rn(T(d[0]), mul_rn(T(d[1]), S[1]));
#pragma unroll
  for (int i = 2; i <= 8; ++i) r = add_rn(r, mul_rn(T(d[i]), S[i]));
  return r;
}

// CHEBY: 0 = exact gates (br.py:175-205), 1 = polynomial gates by Horner's scheme (default for
// config 'cheby'), 2 = polynomial gates in the reference's strict operation order (config
// 'cheby_strict', FIB_F_CHEBY_STRICT)
template <int CHEBY, bool SLOW>
struct BeelerReuter {
  static constexpr int NS = 7;            // C, M, H, J, D, F, XI  (V is the diffusing variable)
  // cells per thread and resident CTAs per SM, chosen by measurement on B200: the kernels are
  // issue/latency bound, so occupancy beats per-thread vector width.  The step that also advances
  // the four slow gates holds more live values than the fast-only step of the skip schedule; the
  // exact slow step's packed pairs want registers (4 / 5 / 6 / 7 CTAs -> 77.9 / 79.3 / 77.1 / 60.8).
  static constexpr int VEC = 2;
  static constexpr int VEC_SMALL = 1;   // cells per thread on small grids (kSmallGridCells)
  static constexpr bool PACKED = true;  // two cells per thread as one f2 pair
  static constexpr int BY = 4;
  static constexpr int MAX_R = 4;
  static constexpr int AUTO_R = 2;   // marching depth picked by launch_step (measured best)
  static constexpr int MIN_BLOCKS = SLOW ? (CHEBY == 1 ? 7 : 5) : 8;
  // the one-cell-per-thread flavour of small grids keeps 6 (512^2 + hole: 45.7 vs 44.2 at 7)
  static __host__ __device__ constexpr int min_blocks(int vec, bool /*phase*/) {
    return (SLOW && CHEBY == 1 && vec == 1) ? 6 : MIN_BLOCKS;
  }
  static constexpr bool PREFETCH = true;
  static constexpr bool NEED_RAW = false; // everything sees V0 = enforce_boundary(V) (br.py:128)
  static constexpr bool NEED_LAP = true;
  static constexpr bool STORE_X = true;
  // slow gates J, D, F, XI are frozen when n == 0 (br.py:199-203): not even written back
  static __host__ __device__ constexpr bool stores(int k) { return k <= 2 || SLOW; }
  static const char* name() {
    return CHEBY == 2 ? (SLOW ? "BeelerReuter<strict,slow>" : "BeelerReuter<strict,fast>")
         : CHEBY == 1 ? (SLOW ? "BeelerReuter<cheby,slow>" : "BeelerReuter<cheby,fast>")
                      : (SLOW ? "BeelerReuter<exact,slow>" : "BeelerReuter<exact,fast>");
  }
  struct Params {
    float dt;            // fp32(dt)
    float neg_dt;        // fp32(-dt)                  m, h
    float neg_dt_slow;   // fp32(-(dt*n))              xi, j, d, f when n > 0 (br.py:197-200)
    float ddt;           // fp32(diff*dt)
    float poly[12][9];   // FIB_TABLE_BR_CHEBY re-expressed as monomial coefficients c_i = d_i 2^(i-1)
                         // (CHEBY == 2: the table's own d_i, fp32)
  };

  // A: anything with a member `p` of type Params (StepArgs<BeelerReuter>, or a reference wrapper)
  template <class A, class T, class L>
  static __device__ __forceinline__ void cell(const A& a, T /*raw*/, T V0, const L& lap, T (&s)[NS], T& Vnew) {
    const Params& p = a.p;
    const T C = s[0], M = s[1], H = s[2], J = s[3], D = s[4], F = s[5], XI = s[6];
    // every current exponential is k = e^{0.04 V0} times a constant; the exact gates reuse 1/k.
    // (The polynomial flavour computes k AFTER its gates: hoisting it costs that kernel 10 %.)
    T k, rk;

    if (CHEBY == 2) {
      const T x = div_rn(sub_rn(V0, T(-30.0f)), T(60.0f));          // br.py:215
      const T tx = mul_rn(T(2.0f), x);                              // br.py:299: T = 2*x*Ts[-1]
      T S[9];
      S[0] = T(1.0f);
      S[1] = x;
#pragma unroll
      for (int i = 2; i <= 8; ++i) S[i] = mul_rn(tx, S[i - 1]);
#define FIB_BR_GATE(g, idx, ndt)                                                            \
  s[idx] = rush_larsen_strict(s[idx], br_strict_eval(p.poly[2 * (g)], S),                  \
                              br_strict_eval(p.poly[2 * (g) + 1], S), ndt)
      FIB_BR_GATE(1, 1, p.neg_dt);                                 // m
      FIB_BR_GATE(2, 2, p.neg_dt);                                 // h
      if (SLOW) {
        FIB_BR_GATE(0, 6, p.neg_dt_slow);                          // xi
        FIB_BR_GATE(3, 3, p.neg_dt_slow);                          // j
        FIB_BR_GATE(4, 4, p.neg_dt_slow);                          // d
        FIB_BR_GATE(5, 5, p.neg_dt_slow);                          // f
      }
#undef FIB_BR_GATE
      k = m_exp(T(0.04f) * V0);
      rk = m_rcp(k);
    } else if (CHEBY == 1) {
      // x = (V0 - 0.5(max+min)) / (0.5(max-min)) = (V0 + 30)/60   (br.py:215)
      const T x = (V0 + T(30.0f)) * T(1.0f / 60.0f);
#define FIB_BR_GATE(RL, g, idx, ndt) \
  s[idx] = RL(s[idx], br_poly8(p.poly[2 * (g)], x), br_poly8(p.poly[2 * (g) + 1], x), ndt)
      if (SLOW) {
        FIB_BR_GATE(rush_larsen, 1, 1, p.neg_dt);                 // m
        FIB_BR_GATE(rush_larsen, 2, 2, p.neg_dt);                 // h
      } else {   // the HBM-bound two-gate step schedules better around the longer expm1 (114 -> 118)
        FIB_BR_GATE(rush_larsen_comp, 1, 1, p.neg_dt);            // m
        FIB_BR_GATE(rush_larsen_comp, 2, 2, p.neg_dt);            // h
      }
      if (SLOW) {
        FIB_BR_GATE(rush_larsen, 0, 6, p.neg_dt_slow);         // xi
        FIB_BR_GATE(rush_larsen, 3, 3, p.neg_dt_slow);         // j
        FIB_BR_GATE(rush_larsen, 4, 4, p.neg_dt_slow);         // d
        FIB_BR_GATE(rush_larsen, 5, 5, p.neg_dt_slow);         // f
      }
#undef FIB_BR_GATE
      k = m_exp(T(0.04f) * V0);
      rk = m_rcp(k);
    } else {
      k = m_exp(T(0.04f) * V0);
      rk = m_rcp(k);
      br_gates_exact<SLOW>(V0, rk, s, p.neg_dt, p.neg_dt_slow);
    }

    // currents from V0 and the OLD gates (br.py:150-165); k = e^{0.04 V0}
    constexpr float E85 = 29.96410004739701f;    // e^{0.04*85}
    constexpr float E53 = 8.331137487687693f;     // e^{0.04*53}
    constexpr float E77 = 21.75840239619708f;    // e^{0.04*77}
    constexpr float E35 = 4.055199966844675f;    // e^{0.04*35}
    const T k53 = k * T(E53);
    const T d23 = V0 + T(23.0f);
    // (V0+23) / (1 - e^{-0.04 (V0+23)}): removable singularity at -23 mV.  Away from it
    // 1 - e^{-0.92}/k is accurate and free (k is already known); within +-3 mV the expm1
    // polynomial takes over (|z| < 0.125 <=> within 3.1 mV of the singularity).
    constexpr float E23N = 0.3985190410845142f;   // e^{-0.04*23}
    const T z = T(-0.04f) * d23;
    const T one_m_e = sel(lt(vabs(z), T(0.125f)), -expm1_poly(z), vfma(T(-E23N), rk, T(1.0f)));
    const T sing = m_div(d23, one_m_e);
    const T iK1 = T(0.35f) * vfma(T(0.2f), sing,
                                  m_div(T(4.f) * vfma(k, T(E85), T(-1.f)), vfma(k53, k53, k53)));
    // measured: reusing 1/k is +3 % for the six-gate polynomial step, -1.5 % for its two-gate one
    const T ix1 = (SLOW || CHEBY != 1)
                      ? XI * T(0.8f) * (vfma(k, T(E77), T(-1.f)) * (rk * T(1.0f / E35)))
                      : XI * T(0.8f) * m_div(vfma(k, T(E77), T(-1.f)), k * T(E35));
    const T gNa = vfma(T(4.0f) * M * M * M * H, J, T(0.005f));       // g_Na M^3 H J + g_NaC
    const T ECa = vfma(T(-13.0278f), m_log(C), T(-82.3f));
    const T iCa = T(0.09f) * D * F * (V0 - ECa);
    const T I_sum = vfma(gNa, V0 - T(50.0f), (iK1 + ix1) + iCa);
    // (V0 + ddt*lap) - dt*I_sum/C_m with the reference's rounding sequence (br.py:167-168): the
    // result crosses 0 mV while the operands are ~80 mV, so no FMA contraction here
    const T dC = vfma(T(-1.0e-7f), iCa, T(0.07f) * (T(1.0e-7f) - C));
    s[0] = vfma(T(p.dt), dC, C);
    const T reaction = mul_rn(T(p.dt), I_sum);
    Vnew = clip_tf(sub_rn(add_rn(V0, mul_rn(T(ddt_of(a)), lap_value<T>(lap))), reaction), -85.0f, 25.0f);
  }
};

}  // namespace fib
