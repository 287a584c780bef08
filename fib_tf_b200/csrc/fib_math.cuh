// fib_math.cuh -- the arithmetic layer of the ionic kernels: packed fp32 pairs + few-ulp transcendentals.
//
// BR and Courtemanche are instruction-issue bound, not HBM bound (SURVEY.md section 7): with
// CUDA's IEEE division (~10 instr + slow path) and libm-grade expf/expm1f/logf/tanhf (12-35
// instr) the BR cell costs ~700 instructions.  Two things bring that down:
//
//  1. Few-ulp transcendentals built on the SFU approximations (MUFU.EX2 / LG2 / RCP), 1 - 4.5 ulp
//     each (expm1 away from 0: < 13 ulp; the numbers below were measured on a B200 by
//     tests/test_gpu_math_layer.py against float64) -- the same error class as swapping one fp32
//     libm for another, which is what the parity bars are calibrated against
//     (oracle/tfshim.ALT_LIBM, tests/test_gpu_parity.py).
//
//  2. Packed fp32 (sm_100: fma/mul/add.rn.f32x2 -> SASS FFMA2 / FMUL2 / FADD2): a thread that owns
//     two cells carries every quantity as an `f2` pair and issues ONE instruction for both cells'
//     multiply-adds -- half the issue slots for the FMA chains that dominate these kernels
//     (Horner gates, exp argument compensation, expm1 polynomials, current sums).  Each lane rounds
//     exactly like the scalar instruction (IEEE rn, no flush), so a packed kernel computes per cell
//     what the scalar flavour of the same source computes.  SFU ops, min/max, compares and selects
//     have no packed form and are issued per lane.
//
// All model code is written ONCE, generic over T = float (one cell per thread) or T = f2 (two):
// the functions below are overloaded for both, `f2` converts implicitly from a float (broadcast), and
// multiply-adds are spelled vfma() explicitly.  Nothing else is ever fused: the library is built with
// -fmad=false (scalar code) and the packed multiply is written so that ptxas cannot contract it (mul2
// below), so the scalar and the packed flavour of a model round identically, cell by cell.
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

namespace fib {

// ---------------------------------------------------------------------------------------------
// f2: two fp32 lanes in an aligned register pair
// ---------------------------------------------------------------------------------------------
struct f2 {
  float x, y;
  __device__ __forceinline__ f2() {}
  __device__ __forceinline__ f2(float a) : x(a), y(a) {}              // broadcast
  __device__ __forceinline__ f2(float a, float b) : x(a), y(b) {}
};
struct b2 { bool x, y; };      // per-lane predicate

#define FIB_F2_OP3(NAME, PTX)                                                                           \
  __device__ __forceinline__ f2 NAME(f2 a, f2 b, f2 c) {                                                \
    f2 d;                                                                                               \
    asm("{.reg .b64 ra, rb, rc, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; mov.b64 rc, {%6,%7}; "    \
        PTX " rd, ra, rb, rc; mov.b64 {%0,%1}, rd;}"                                                    \
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));           \
    return d;                                                                                           \
  }
#define FIB_F2_OP2(NAME, PTX)                                                                           \
  __device__ __forceinline__ f2 NAME(f2 a, f2 b) {                                                      \
    f2 d;                                                                                               \
    asm("{.reg .b64 ra, rb, rd; mov.b64 ra, {%2,%3}; mov.b64 rb, {%4,%5}; "                             \
        PTX " rd, ra, rb; mov.b64 {%0,%1}, rd;}"                                                        \
        : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));                               \
    return d;                                                                                           \
  }
FIB_F2_OP3(fma2, "fma.rn.f32x2")
FIB_F2_OP2(add2, "add.rn.f32x2")
FIB_F2_OP2(sub2, "sub.rn.f32x2")
#undef FIB_F2_OP3
#undef FIB_F2_OP2

// Packed multiply.  ptxas CONTRACTS mul.rn.f32x2 + add.rn.f32x2 into one FFMA2 whatever -fmad says,
// although the scalar mul.rn / add.rn are never fused (checked in SASS; it even sees through
// fma(a,b,-0) and fma(p,1,b) with literal constants), which would make a packed lane round differently
// from the scalar cell.  So a * b is issued as fma(a, b, NZERO) with NZERO = -0.0f read from constant
// memory at run time: exactly fl(a * b), signed zeros included (+0 + -0 = +0, -0 + -0 = -0; tested lane
// for lane against the scalar multiply), one FFMA2 instead of one FMUL2 -- and with no packed multiply
// left in the code there is nothing to contract.
static __constant__ float kFibNegZero = -0.0f;
__device__ __forceinline__ f2 mul2(f2 a, f2 b) {
  const float nz = kFibNegZero;
  return fma2(a, b, f2(nz));
}

__device__ __forceinline__ f2 operator+(f2 a, f2 b) { return add2(a, b); }
__device__ __forceinline__ f2 operator-(f2 a, f2 b) { return sub2(a, b); }
__device__ __forceinline__ f2 operator*(f2 a, f2 b) { return mul2(a, b); }
__device__ __forceinline__ f2 operator-(f2 a) { return f2(-a.x, -a.y); }   // folds into operand modifiers

// ---- the generic vocabulary: the same names for float and f2 -----------------------------------
// multiply-add (one rounding)
__device__ __forceinline__ float vfma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ f2 vfma(f2 a, f2 b, f2 c) { return fma2(a, b, c); }
// single operations with their own rounding, never contracted (the reference's operation order)
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ f2 add_rn(f2 a, f2 b) { return add2(a, b); }
__device__ __forceinline__ f2 sub_rn(f2 a, f2 b) { return sub2(a, b); }
__device__ __forceinline__ f2 mul_rn(f2 a, f2 b) { return mul2(a, b); }
__device__ __forceinline__ f2 div_rn(f2 a, f2 b) { return f2(__fdiv_rn(a.x, b.x), __fdiv_rn(a.y, b.y)); }
// per-lane predicates and selects
__device__ __forceinline__ bool lt(float a, float b) { return a < b; }
__device__ __forceinline__ bool gt(float a, float b) { return a > b; }
__device__ __forceinline__ b2 lt(f2 a, f2 b) { return b2{a.x < b.x, a.y < b.y}; }
__device__ __forceinline__ b2 gt(f2 a, f2 b) { return b2{a.x > b.x, a.y > b.y}; }
__device__ __forceinline__ float sel(bool m, float a, float b) { return m ? a : b; }
__device__ __forceinline__ f2 sel(b2 m, f2 a, f2 b) { return f2(m.x ? a.x : b.x, m.y ? a.y : b.y); }
__device__ __forceinline__ bool any_lane(bool m) { return m; }
__device__ __forceinline__ bool any_lane(b2 m) { return m.x || m.y; }
__device__ __forceinline__ float vabs(float a) { return fabsf(a); }
__device__ __forceinline__ f2 vabs(f2 a) { return f2(fabsf(a.x), fabsf(a.y)); }
__device__ __forceinline__ float vmin(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ float vmax(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ f2 vmin(f2 a, f2 b) { return f2(fminf(a.x, b.x), fminf(a.y, b.y)); }
__device__ __forceinline__ f2 vmax(f2 a, f2 b) { return f2(fmaxf(a.x, b.x), fmaxf(a.y, b.y)); }
// lanes
__device__ __forceinline__ float lane(float a, int) { return a; }
__device__ __forceinline__ float lane(f2 a, int i) { return i == 0 ? a.x : a.y; }
template <class T> struct Lanes;
template <> struct Lanes<float> { static constexpr int N = 1; };
template <> struct Lanes<f2> { static constexpr int N = 2; };
template <class T> __device__ __forceinline__ T from_lanes(const float* v);
template <> __device__ __forceinline__ float from_lanes<float>(const float* v) { return v[0]; }
template <> __device__ __forceinline__ f2 from_lanes<f2>(const float* v) { return f2(v[0], v[1]); }
__device__ __forceinline__ void to_lanes(float a, float* v) { v[0] = a; }
__device__ __forceinline__ void to_lanes(f2 a, float* v) { v[0] = a.x; v[1] = a.y; }

// ---------------------------------------------------------------------------------------------
// SFU approximations
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float sfu_rcp(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sfu_ex2(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sfu_lg2(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float sfu_sqrt(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ f2 sfu_rcp(f2 a) { return f2(sfu_rcp(a.x), sfu_rcp(a.y)); }
__device__ __forceinline__ f2 sfu_ex2(f2 a) { return f2(sfu_ex2(a.x), sfu_ex2(a.y)); }
__device__ __forceinline__ f2 sfu_lg2(f2 a) { return f2(sfu_lg2(a.x), sfu_lg2(a.y)); }
__device__ __forceinline__ f2 sfu_sqrt(f2 a) { return f2(sfu_sqrt(a.x), sfu_sqrt(a.y)); }

// < 1 ulp (measured 0.96) / < 2 ulp (1.95); subnormal inputs and results flush to zero
template <class T> __device__ __forceinline__ T m_rcp(T x) { return sfu_rcp(x); }
template <class T, class U> __device__ __forceinline__ T m_div(U a, T b) { return T(a) * sfu_rcp(b); }

// e^x = 2^t * 2^r, t = fl(x*log2e), r = the rounding error of that product + x*lo(log2e),
// 2^r ~ 1 + r ln2.  < 3 ulp (measured 2.96) for |x| <= 2^24; +inf on overflow; 0 below
// ln(FLT_MIN) = -87.34 (the SFU flushes the subnormal results that expf returns down to -103.9).
// Beyond |x| ~ 2.3e7, |r| exceeds 1/ln2 and 1 + r ln2 can be negative: x that large gives -inf or NaN
// (negative x: +-0), and x = +-inf gives NaN (r = inf - inf).  No call site comes near: the models'
// exponents are within +-60 for V in [-120, 80] mV, and those of the Ca-release sigmoids (u_inf, v_inf)
// are large only when negative, where 2^t = 0 whatever the factor.
template <class T> __device__ __forceinline__ T m_exp(T x) {
  const float L2E_HI = 1.44269502162933349609375f, L2E_LO = 1.92596299112661746e-8f;
  const T t = x * T(L2E_HI);
  T r = vfma(x, T(L2E_HI), -t);
  r = vfma(x, T(L2E_LO), r);
  return sfu_ex2(t) * vfma(r, T(0.693147182464599609375f), T(1.0f));
}

// c e^x + add with the scale folded into the compensation factor and the add into an FMA: one or
// two instructions fewer than c * m_exp(x) + add (c and add are compile-time literals at the call
// sites; add == 0 folds to a multiply).
template <class T> __device__ __forceinline__ T m_exp_affine(T x, float c, float add) {
  const float L2E_HI = 1.44269502162933349609375f, L2E_LO = 1.92596299112661746e-8f;
  const T t = x * T(L2E_HI);
  T r = vfma(x, T(L2E_HI), -t);
  r = vfma(x, T(L2E_LO), r);
  const T f = vfma(r, T(c * 0.693147182464599609375f), T(c));
  return add == 0.f ? sfu_ex2(t) * f : vfma(sfu_ex2(t), f, T(add));
}

// x + x^2 (1/2 + x/3! + ... + x^4/6!): expm1 for |x| < 0.125 (truncation x^6/7! < 1e-9 relative)
template <class T> __device__ __forceinline__ T expm1_poly(T x) {
  T p = T(1.38888888888889e-3f);                  // 1/6!
  p = vfma(p, x, T(8.33333333333333e-3f));        // 1/5!
  p = vfma(p, x, T(4.16666666666667e-2f));        // 1/4!
  p = vfma(p, x, T(1.66666666666667e-1f));        // 1/3!
  p = vfma(p, x, T(0.5f));
  return vfma(p * x, x, x);
}

// expm1: the polynomial for |x| < 0.125, exp(x)-1 beyond.  The polynomial side is the one that
// matters for accuracy: |x| = dt/tau is small exactly for the slow gates, whose per-step error would
// otherwise accumulate over hundreds of steps; for |x| >= 0.125 a gate relaxes within ~10 steps and
// exp(x)-1 (|result| >= 0.117, so < 13 ulp; measured 12.9) is plenty.  The polynomial side is < 1 ulp
// (0.55).  Built on m_exp: NaN for x = +-inf.  Both sides are computed and selected: no
// divergence.
template <class T> __device__ __forceinline__ T m_expm1(T x) {
  const T p = expm1_poly(x);
  const T e = m_exp(x) - T(1.0f);
  return sel(lt(vabs(x), T(0.125f)), p, e);
}

// expm1 for the Rush-Larsen factor, x = -dt/tau <= 0.  On the far side the exponential needs no
// argument compensation: the uncompensated 2^(x log2e) is off by e^x (2 ulp + |x| 2^-24), i.e. an
// ABSOLUTE error <= 1.6e-7 (|x| e^x <= 1/e), against a result of magnitude >= 0.117 -- the same
// < 13 ulp as m_expm1 (measured 12.9), three instructions cheaper per gate.  Negative tau (the BR
// polynomial tau_h below -83.85 mV) feeds it x > 0, where the uncompensated product costs up to
// x 2^-24 relative: measured < 10 ulp for 0 < x <= 1 and < 8 + x ulp beyond.  Valid for every x:
// +inf -> +inf, -inf -> -1.
template <class T> __device__ __forceinline__ T m_expm1_neg(T x) {
  const T p = expm1_poly(x);
  const T e = sfu_ex2(x * T(1.44269502162933349609375f)) - T(1.0f);
  return sel(lt(vabs(x), T(0.125f)), p, e);
}

// log: lg2.approx has an absolute error bound (2^-22 for x in [0.5, 2]), so through 0 near x = 1 the
// error is absolute (measured <= 1.6e-7); < 3.5 ulp elsewhere (3.17).  sqrt: < 1 ulp (0.93).
template <class T> __device__ __forceinline__ T m_log(T x) { return sfu_lg2(x) * T(0.693147182464599609375f); }
template <class T> __device__ __forceinline__ T m_sqrt(T x) { return sfu_sqrt(x); }
// 1 + e^{-2z} as ONE explicit FMA: left to the compiler, ptxas decides per kernel whether the
// multiply and the add fuse, and two kernels that must agree bit for bit (the one- and the
// two-steps-per-launch 4v kernels) would differ in the last place.  < 4.5 ulp (4.19) for |z| <= 2^23.
template <class T> __device__ __forceinline__ T m_half_1p_tanh(T z) {
  return sfu_rcp(m_exp_affine(T(-2.0f) * z, 1.0f, 1.0f));
}

// The Laplacian enters a cell function only in its last expression.  A cell function takes it either
// as a value or as a callable evaluated at that point: the persistent kernel passes a callable that
// first waits for the neighbour tiles' rows, so everything of the cell that does not depend on them
// is already computed when they arrive (fib_persist.cuh).
template <class T, class L>
__device__ __forceinline__ T lap_value(const L& lap) {
  if constexpr (std::is_convertible<L, T>::value) return lap;
  else return lap();
}

}  // namespace fib
