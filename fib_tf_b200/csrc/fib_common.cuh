// fib_common.cuh -- geometry, vector access and small math helpers shared by every kernel.
// sm_100a only.  No CPU fallback exists anywhere in this library.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "fib_math.cuh"

namespace fib {

// Geometry of one shard.  Planes are SoA fp32, row pitch `pitch` floats (multiple of 32 -> every
// row starts 128-B aligned, so float4 accesses are always legal and padded columns are in-bounds).
// The diffusing variable and the phase field carry one halo row above and below the shard:
//   diffusing/phase plane:  element (global row g, col c) = p[(g - row0 + 1) * pitch + c]
//   every other plane:      element (global row g, col c) = p[(g - row0) * pitch + c]
struct Geom {
  int H, W;         // global grid (config 'height', 'width')
  int row0, rows;   // this shard owns global rows [row0, row0+rows)
  int pitch;        // floats per row
};

// The planes are read through the non-coherent path (ld.global.nc, __ldg).  An in-place plane is
// read exactly once, by the thread that later overwrites the same address, and L1 is invalidated at
// every kernel boundary, so no stale line can be observed AS LONG AS consecutive step kernels do not
// overlap (no programmatic dependent launch).  It lets the scheduler interleave the state loads with
// the phase-field / lookup-table reads: 4v + phase field 157 -> 169, Courtemanche LUT 28.5 -> 32.3
// Gcell-steps/s; no effect on the other flavours.
template <int VEC> struct VecIO;
template <> struct VecIO<1> {
  static __device__ __forceinline__ void ld(const float* p, float* v) { v[0] = __ldg(p); }
  static __device__ __forceinline__ void st(float* p, const float* v) { *p = v[0]; }
};
template <> struct VecIO<2> {
  static __device__ __forceinline__ void ld(const float* p, float* v) {
    float2 t = __ldg(reinterpret_cast<const float2*>(p)); v[0] = t.x; v[1] = t.y;
  }
  static __device__ __forceinline__ void st(float* p, const float* v) {
    *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
  }
};
template <> struct VecIO<4> {
  static __device__ __forceinline__ void ld(const float* p, float* v) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p)); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void st(float* p, const float* v) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};

// tf.clip_by_value(x, lo, hi) = maximum(minimum(x, hi), lo) (ionic.py:122-123, br.py:167-168) with the
// NaN behaviour of the reference's TARGET, TensorFlow on the GPU: Eigen's CUDA mini/maxi are
// fminf/fmaxf (and XLA:GPU lowered min/max to minnum/maxnum), which return the non-NaN operand.
// This matters: the BR currents are 0/0 when V hits -23.0f (or -47.0f) exactly (br.py:150-151,
// 52), which happens to a few cells of a 512^2 grid in every repolarisation wave; on the GPU the
// clip turns that NaN into the upper bound for one step and the run goes on (docs/br.png), whereas
// NaN-propagating min/max (NumPy, TF on the CPU) would poison the whole grid within 50 ms.
// (All of these are generic over T = float or f2, see fib_math.cuh.)
template <class T> __device__ __forceinline__ T clip_tf(T x, float lo, float hi) {
  return vmax(vmin(x, T(hi)), T(lo));
}

// IonicModel.rush_larsen (ionic.py:115-123): clip(g + (g - g_inf) * expm1(-dt / tau), 1e-5, 0.99999).
// neg_dt = fp32(-dt) (or fp32(-(dt*n)) folded in double on the host, br.py:197-200).
template <class T> __device__ __forceinline__ T rush_larsen(T g, T g_inf, T tau, float neg_dt) {
  const T e = m_expm1_neg(m_div(T(neg_dt), tau));
  return clip_tf(vfma(g - g_inf, e, g), 0.00001f, 0.99999f);
}
// Rush-Larsen with caller-supplied clip bounds: (1e-5, 0.99999) for the Python models, (-inf, +inf)
// for the native courtemanche.h rule, which does not clip (courtemanche.h:287-292)
template <class T> __device__ __forceinline__ T rush_larsen_eb(T g, T g_inf, T e, float lo, float hi) {
  const T r = vfma(g - g_inf, e, g);
  return lo == -INFINITY ? r : clip_tf(r, lo, hi);      // uniform select; no clip in native mode
}
template <class T> __device__ __forceinline__ T rush_larsen_b(T g, T g_inf, T tau, float neg_dt, float lo,
                                                              float hi) {
  return rush_larsen_eb(g, g_inf, m_expm1_neg(m_div(T(neg_dt), tau)), lo, hi);
}
// same with e = expm1(-dt/tau) precomputed (Python-scalar tau: court.py:189,243)
template <class T> __device__ __forceinline__ T rush_larsen_e(T g, T g_inf, T e) {
  return clip_tf(vfma(g - g_inf, e, g), 0.00001f, 0.99999f);
}
// the reference's operation sequence, unfused, IEEE division, libm expm1f (strict-order flavour)
__device__ __forceinline__ float rush_larsen_strict(float g, float g_inf, float tau, float neg_dt) {
  const float e = expm1f(__fdiv_rn(neg_dt, tau));
  return clip_tf(__fadd_rn(g, __fmul_rn(__fsub_rn(g, g_inf), e)), 0.00001f, 0.99999f);
}
__device__ __forceinline__ f2 rush_larsen_strict(f2 g, f2 g_inf, f2 tau, float neg_dt) {
  return f2(rush_larsen_strict(g.x, g_inf.x, tau.x, neg_dt), rush_larsen_strict(g.y, g_inf.y, tau.y, neg_dt));
}

}  // namespace fib
