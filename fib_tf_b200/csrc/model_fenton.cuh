// model_fenton.cuh -- Cherry-Ehrlich-Nattel-Fenton 4-variable model, pointwise part.
// Restates fenton.py:46-92 (differentiate) and fenton.py:103-106 (explicit Euler).
#pragma once
#include "fib_kernels.cuh"

namespace fib {

struct Fenton4v {
  static constexpr int NS = 3;            // V, W, S  (U is the diffusing variable)
  static constexpr int VEC = 4;
  static constexpr int VEC_SMALL = 4;   // cells per thread on small grids (kSmallGridCells)
  static constexpr int BY = 4;
  static constexpr int MAX_R = 4;
  static constexpr int AUTO_R = 4;   // marching depth picked by launch_step (measured best)
  static constexpr int MIN_BLOCKS = 8;
  // the phase-field flavour holds the phi window as well: at 8 CTAs per SM (64 registers) it spilled 33
  // values per thread (round-1 ncu); 6 CTAs (80 registers) keeps everything in registers
  static __host__ __device__ constexpr int min_blocks(int /*cells per thread*/, bool phase) {
    return phase ? 6 : MIN_BLOCKS;
  }
  static constexpr bool PACKED = true;   // the four cells of a thread as two f2 pairs
  static constexpr bool PREFETCH = true;
  static constexpr bool NEED_RAW = true;  // reaction sees the raw U (fenton.py:101), SURVEY fact 3
  static constexpr bool NEED_LAP = true;
  static constexpr bool STORE_X = true;
  static __host__ __device__ constexpr bool stores(int) { return true; }
  static const char* name() { return "Fenton4v"; }
  struct Params {
    float dt;    // fp32(dt)
    float ddt;   // fp32(diff * dt), folded in double like the reference (fenton.py:103)
  };

  // Divisions by literals are multiplications by the correctly rounded reciprocal (<= 1 ulp from
  // the reference's fp32 division; budgeted in SURVEY.md Appendix B.2).
  // Generic over T = float (one cell) and T = f2 (two cells as one packed pair: FFMA2 / FMUL2 / FADD2,
  // fib_math.cuh); every operation is spelled with its own rounding (mul_rn / add_rn / vfma), so a lane of
  // the pair computes exactly what the scalar cell computes and every kernel that calls this function --
  // one step per launch, two steps per launch, the persistent kernel -- agrees bit for bit.
  // A: anything with a member `p` of type Params (StepArgs<Fenton4v>, or a reference wrapper)
  // L: T, or a callable returning T (lap_value, fib_math.cuh)
  template <class A, class T, class L>
  static __device__ __forceinline__ void cell(const A& a, T U, T U0, const L& lap, T (&s)[NS], T& Unew) {
    constexpr float tau_vp = 3.33f, tau_vn = 19.2f, tau_wp = 160.0f, tau_wn = 75.0f;
    constexpr float tau_d = 0.065f, tau_si = 31.8364f, tau_so = 31.8364f, tau_a = 0.009f;
    constexpr float u_c = 0.23f, u_m = 1.0f, u_csi = 0.8f, u_so = 0.3f;
    constexpr float r_sn = 1.2f, k_ = 3.0f, b_so = 0.84f, c_so = 0.02f;
    constexpr float c_so_half = (float)(0.5 * (0.115 - 0.009));   // 0.5*(a_so - tau_a), fenton.py:83
    constexpr float r_diff = (float)(0.02 - 1.2);                 // (r_sp - r_sn),      fenton.py:89
    const T dt = T(a.p.dt);
    const T V = s[0], W = s[1], S = s[2];

    // H(x) = (1+sign x)/2, G(x) = (1-sign x)/2 (fenton.py:73-79): 0.5 at x == 0
    const auto above_c = gt(U, T(u_c));
    const T Hc = sel(above_c, T(1.f), sel(lt(U, T(u_c)), T(0.f), T(0.5f)));
    const T Hso = sel(gt(U, T(u_so)), T(1.f), sel(lt(U, T(u_so)), T(0.f), T(0.5f)));
    const T Gso = sub_rn(T(1.f), Hso);

    const T X_fi = mul_rn(mul_rn(mul_rn(-V, Hc), sub_rn(U, T(u_c))), sub_rn(T(u_m), U));
    const T I_si = mul_rn(mul_rn(-W, S), T(1.0f / tau_si));
    // 0.5 (a_so - tau_a) (1 + tanh z) = (a_so - tau_a) * [0.5 (1 + tanh z)]
    const T T_so = m_half_1p_tanh(mul_rn(sub_rn(U, T(b_so)), T(1.0f / c_so)));
    const T I_so = vfma(T(2.0f * c_so_half), T_so,
                        vfma(mul_rn(U, Gso), T(1.0f / tau_so), mul_rn(Hso, T(tau_a))));
    // dU = -(I_fi + I_si + I_so), I_fi = X_fi / tau_d
    const T dU = -add_rn(vfma(X_fi, T(1.0f / tau_d), I_si), I_so);
    const T dV = sel(above_c, mul_rn(-V, T(1.0f / tau_vp)), mul_rn(sub_rn(T(1.f), V), T(1.0f / tau_vn)));
    // tau_wn1 == tau_wn2 == 75 (fenton.py:53-54): the inner tf.where is an identity
    const T dW = sel(above_c, mul_rn(-W, T(1.0f / tau_wp)), mul_rn(sub_rn(T(1.f), W), T(1.0f / tau_wn)));
    const T r_s = vfma(T(r_diff), Hc, T(r_sn));
    const T dS = mul_rn(r_s, sub_rn(m_half_1p_tanh(mul_rn(sub_rn(U, T(u_csi)), T(k_))), S));

    // (U0 + dt*dU) + ddt*lap with the reference's rounding sequence (fenton.py:103): near U ~ 0 an
    // FMA's missing rounding would show up as a 1-ulp(|U0|) absolute difference
    s[0] = vfma(dt, dV, V);
    s[1] = vfma(dt, dW, W);
    s[2] = vfma(dt, dS, S);
    const T reaction = add_rn(U0, mul_rn(dt, dU));
    Unew = add_rn(reaction, mul_rn(T(ddt_of(a)), lap_value<T>(lap)));
  }

  // four cells of a thread as two packed pairs
  template <class A>
  static __device__ __forceinline__ void cell4(const A& a, const float (&raw)[4], const float* x0,
                                               const float (&lap)[4], float (&sv)[3][4], float (&unew)[4]) {
#pragma unroll
    for (int l = 0; l < 4; l += 2) {
      f2 sp[3] = {f2(sv[0][l], sv[0][l + 1]), f2(sv[1][l], sv[1][l + 1]), f2(sv[2][l], sv[2][l + 1])};
      f2 un;
      cell(a, f2(raw[l], raw[l + 1]), f2(x0[l], x0[l + 1]), f2(lap[l], lap[l + 1]), sp, un);
      unew[l] = un.x;
      unew[l + 1] = un.y;
#pragma unroll
      for (int k = 0; k < 3; ++k) { sv[k][l] = sp[k].x; sv[k][l + 1] = sp[k].y; }
    }
  }
};

}  // namespace fib
