// fib_stencil.cuh -- no-flux boundary + 9-point Laplacian + phase-field term, fused.
//
// Reference semantics (two-stage boundary, SURVEY.md facts 1-2):
//   X0 = enforce_boundary(X)  : border ring := SYMMETRIC pad of X[1:-1,1:-1]      (ionic.py:107-113)
//   Xp = REFLECT-pad(X0, 1)   : one more ring                                       (ionic.py:49-50)
//   lap = N+S+W+E + 0.5*(NW+SW+NE+SE) - 6*C  on Xp                                   (ionic.py:51-53)
// Both stages collapse to one index map on the RAW plane:
//   Xp[r][c] = X[clamp(r,1,H-2)][clamp(c,1,W-2)]   for r in [-1,H], c in [-1,W]
// so no padded copy is ever materialised; the kernel reads X through clamped indices.
// The phase field is only REFLECT-padded (ionic.py:75-76): index -1 -> 1, H -> H-2.
#pragma once
#include "fib_common.cuh"

namespace fib {

__device__ __forceinline__ int clampi(int v, int lo, int hi) { return min(max(v, lo), hi); }
__device__ __forceinline__ int reflecti(int v, int n) { return v < 0 ? -v : (v >= n ? 2 * n - 2 - v : v); }

// Column indices of the VEC+2 window entries of a thread owning columns [c, c+VEC): row-invariant,
// computed once per thread.  `interior` threads (the overwhelming majority) read one aligned vector
// plus the two neighbours; edge threads gather through the clamped / reflected indices.
template <int VEC>
struct ColWindow {
  int c;                 // first owned column
  bool interior_x;       // c-1 >= 1 && c+VEC <= W-2  (no clamping needed for the diffusing variable)
  bool interior_p;       // c-1 >= 0 && c+VEC <= W-1  (no reflection needed for the phase field)
  __device__ __forceinline__ ColWindow(int c_, int W)
      : c(c_), interior_x(c_ >= 2 && c_ + VEC <= W - 2), interior_p(c_ >= 1 && c_ + VEC <= W - 1) {}
};

// e[j] = Xp[row][c-1+j], j = 0..VEC+1; `row` = element index of the row start (32-bit: the host
// guarantees (rows+2)*pitch < 2^31), already row-clamped by the caller.
template <int VEC>
__device__ __forceinline__ void load_enforced_row(const float* __restrict__ x, int row,
                                                  const ColWindow<VEC>& cw, int W,
                                                  float (&e)[VEC + 2]) {
  if (cw.interior_x) {
    const float* p = x + (row + cw.c);
    VecIO<VEC>::ld(p, &e[1]);
    e[0] = __ldg(p - 1);
    e[VEC + 1] = __ldg(p + VEC);
  } else {
#pragma unroll
    for (int j = 0; j < VEC + 2; ++j) e[j] = __ldg(x + (row + clampi(cw.c - 1 + j, 1, W - 2)));
  }
}

// p[j] = phi_pad[row][c-1+j] with REFLECT columns.
template <int VEC>
__device__ __forceinline__ void load_reflect_row(const float* __restrict__ ph, int row,
                                                 const ColWindow<VEC>& cw, int W,
                                                 float (&p)[VEC + 2]) {
  if (cw.interior_p) {
    const float* q = ph + (row + cw.c);
    VecIO<VEC>::ld(q, &p[1]);
    p[0] = q[-1];
    p[VEC + 1] = q[VEC];
  } else {
#pragma unroll
    for (int j = 0; j < VEC + 2; ++j) p[j] = ph[row + clampi(reflecti(cw.c - 1 + j, W), 0, W - 1)];
  }
}

// ionic.py:51-53, same association order as the reference, no FMA contraction: given identical
// inputs this is bit-identical to the NumPy oracle.
// lap9_combine: its last three operations, edges + 0.5 corners - 6 C, on the two sums.  T = float, or
// f2 for two neighbouring cells (FADD2 / FFMA2; each lane rounds like the scalar form, fib_math.cuh).
template <class T>
__device__ __forceinline__ T lap9_combine(T edges, T corners, T C) {
  return sub_rn(add_rn(edges, mul_rn(T(0.5f), corners)), mul_rn(T(6.0f), C));
}
__device__ __forceinline__ float lap9(float N, float S, float Wv, float E, float NW, float SW,
                                      float NE, float SE, float C) {
  float edges = __fadd_rn(__fadd_rn(__fadd_rn(N, S), Wv), E);
  float corners = __fadd_rn(__fadd_rn(__fadd_rn(NW, SW), NE), SE);
  return lap9_combine(edges, corners, C);
}

// ionic.py:78-80: ((X_S-X_N)(phi_S-phi_N) + (X_E-X_W)(phi_E-phi_W)) / (4 phi_C)
__device__ __forceinline__ float phase_term(float xN, float xS, float xW, float xE, float pN,
                                            float pS, float pW, float pE, float pC) {
  float a = __fmul_rn(__fsub_rn(xS, xN), __fsub_rn(pS, pN));
  float b = __fmul_rn(__fsub_rn(xE, xW), __fsub_rn(pE, pW));
  return m_div(__fadd_rn(a, b), __fmul_rn(4.0f, pC));   // 2-ulp SFU division
}

}  // namespace fib
