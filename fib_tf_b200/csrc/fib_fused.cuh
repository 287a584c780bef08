// fib_fused.cuh -- Fenton 4v, TWO explicit time steps per launch (temporal blocking, k = 2).
//
// Why: the one-step kernel runs at the HBM roofline (32 B per cell-step) with half of the issue
// slots idle (profiles/r1_ncu_summary.txt).  Two steps per pass read and write every plane once
// per TWO steps: 16 B per cell-step plus the halo re-reads.
//
// How: a warp owns 32 x 4 = 128 consecutive columns for the FIRST step and the inner 120 of them
// (lanes 1..30) for the SECOND one, and marches down its rows.  Per iteration j it
//   1. advances row j by one step from global memory (same loads and the same Fenton4v::cell as
//      step_kernel) and keeps the results in registers: U1 (4 cells) and V1, W1, S1;
//   2. completes the U1 window of row j with the two neighbour cells by warp shuffles;
//   3. advances row j-1 by the second step from the register windows of rows j-2, j-1, j and
//      stores U2, V2, W2, S2.
// The first step is recomputed in the overlap (8 of 128 columns per warp, 2 extra rows per row
// block), never exchanged, so every cell goes through exactly the arithmetic of two one-step
// launches and the result is BIT-IDENTICAL to them (tests/test_gpu_parity.py).  Because a cell
// of the overlap is read by two warps, no plane can be updated in place: all four planes are
// ping-ponged, and all four carry kFuseHalo = 2 halo rows (fib_capi.cu) -- a shard exchanges two
// rows of each plane per launch instead of one row of U per step.
//
// Boundary (fib_stencil.cuh): step 2 sees U1 through the same index map as step 1 sees U,
//   Xp[r][c] = U1[clamp(r,1,H-2)][clamp(c,1,W-2)]; the column clamp is applied when the window is
// formed, the row clamp when the three window rows are picked.
// The phase field is read like in step_kernel (on demand, where fib_set_phase flagged the block),
// from a copy of phi in the same two-halo-row layout.  Restriction: W % 4 == 0 (fib_create).
#pragma once
#include "model_fenton.cuh"

namespace fib {

constexpr int kFuseHalo = 2;     // halo rows of every plane in the fused layout
constexpr int kFuseCols = 120;   // output columns per warp: lanes 1..30 x 4 cells
constexpr int kFuseBY = 4;       // warps (row blocks) per CTA
// resident CTAs per SM without the phase field: 96 registers.  4 (128 registers) and 6 (80, spills) are
// slower at 32768^2 and 8192^2 (profiles/r3_fused_march.md)
constexpr int kFuseMinB = 5;
// prefetch distance in rows: a trip is short enough now that one row ahead leaves part of the load
// latency uncovered with 20 warps per SM (32768^2: 334 at 1 row, 347 at 2, 274 without the prefetch)
constexpr int kFusePFD = 2;

struct Fused2Args {
  const float* in[4];   // U, V, W, S at time t   (halo layout, kFuseHalo rows above and below)
  float* out[4];        // the same at time t + 2 dt
  const float* phase;   // phi in the SAME halo layout (kFuseHalo rows), or nullptr
  const unsigned char* pmask;   // [rows + 2][pmask_pitch], local rows -1 .. rows: 1 where the phase term
  int pmask_pitch;              //   of a 32-column block can be non-zero (fib_set_phase)
  int lr0, nrows;       // local OUTPUT row range of this launch
  int R;                // output rows per warp
  int nz;               // replicas, blockIdx.z (fib_kernels.cuh StepArgs)
  const float* zddt;    // per-replica p.ddt, or nullptr
  Fenton4v::Params p;
};

__device__ __forceinline__ float pick4(const float (&v)[4], int i) {
  return i == 0 ? v[0] : (i == 1 ? v[1] : (i == 2 ? v[2] : v[3]));
}

// The march of one warp over its output rows [g0, g1).  IX: every lane's columns are at least two
// away from the grid's side borders, so no lane needs the column clamp (known per CTA column).
//
// A marching trip j (step 1 on row j, step 2 on row j - 1) comes in two bodies.  The EDGE body
// handles everything: rows outside the grid, the row clamps of rows 0, 1, H-2, H-1, the first
// trips of the march (no step 2 yet) and the last one.  The interior body, for
// j in [max(g0 + 1, 3), min(g1 - kFusePFD, H - 3)], needs none of that: all its rows are rows of
// the grid without a clamp, and all its addresses are one row offset plus multiples of the pitch.
// Interior trips of IX warps are unrolled by three, with the three-row windows passed by reference
// in rotated order, so the rows' roles never move between registers; the remainder of the trip
// count modulo 3 runs through the EDGE body before them.  Both bodies make the same loads, the same
// cell4 calls with the same operands and hence the same results.
template <bool PHASE, bool IX, bool Z>
struct Fused2March {
  const Geom& g;
  const Fused2Args& a;
  StepArgsOf<Fenton4v, Z> sa;
  int lane, c, cs, g0, g1, row0;
  bool emit_lane;
  ColWindow<4> cw;

  __device__ __forceinline__ Fused2March(const Geom& g_, const Fused2Args& a_, int c0, int g0_, int g1_)
      : g(g_), a(a_), lane(threadIdx.x), c(c0 + (int)threadIdx.x * 4), g0(g0_), g1(g1_), row0(zrow0<Z>(g_)), cw(0, 0) {
    const int W = g.W;
    const bool valid = IX || (c >= 0 && c < W);                // W % 4 == 0: all four cells or none
    cs = valid ? c : (c < 0 ? 0 : W - 4);                      // in-bounds column for addressing
    emit_lane = valid && lane >= 1 && lane <= 30;
    cw = ColWindow<4>(cs, W);
    if (IX) cw.interior_x = cw.interior_p = true;              // what it computes, known at compile time
    sa.p = a.p;
    if (Z) sa.zddt = a.zddt;
  }

  __device__ __forceinline__ int rowoff(int gr) const { return (gr - row0 + kFuseHalo) * g.pitch; }
  __device__ __forceinline__ int xrow(int gr) const { return rowoff(clampi(gr, 1, g.H - 2)); }
  __device__ __forceinline__ int prow(int gr) const { return rowoff(reflecti(gr, g.H)); }

  // the phase term of row gr (ionic.py:70-81), exactly as step_kernel forms it: phi is fetched on
  // demand, only where fib_set_phase flagged the 32-column block.  o*: offsets of my columns of the
  // (reflected) rows gr - 1, gr, gr + 1
  __device__ __forceinline__ bool phase_flag(int gr) const {
    return a.pmask[(gr - row0 + 1) * a.pmask_pitch + (cs >> 5)] != 0;
  }
  __device__ __forceinline__ void add_phase(int oN, int oC, int oS, const float (&n)[6], const float (&x)[6],
                                            const float (&s)[6], float (&lapv)[4]) const {
    float pN[4], pS[4], pC[6];
    VecIO<4>::ld(a.phase + oN, pN);
    VecIO<4>::ld(a.phase + oS, pS);
    load_reflect_row<4>(a.phase, oC - cs, cw, g.W, pC);
#pragma unroll
    for (int l = 0; l < 4; ++l)
      lapv[l] = __fadd_rn(lapv[l], phase_term(n[l + 1], s[l + 1], x[l], x[l + 2], pN[l], pS[l], pC[l], pC[l + 2],
                                              pC[l + 1]));
  }

  // lap9 of my four cells with the same operations in the same order: the vertical sums N + S of a
  // cell are the NW + SW of its right neighbour, and the last three operations run on pairs
  __device__ __forceinline__ void lap4(const float (&n)[6], const float (&x)[6], const float (&s)[6],
                                       float (&lapv)[4]) const {
    float v[6], edges[4], corners[4];
    v[0] = __fadd_rn(n[0], s[0]);
    v[5] = __fadd_rn(n[5], s[5]);
#pragma unroll
    for (int q = 1; q < 5; q += 2) {
      const f2 t = add_rn(f2(n[q], n[q + 1]), f2(s[q], s[q + 1]));
      v[q] = t.x;
      v[q + 1] = t.y;
    }
#pragma unroll
    for (int l = 0; l < 4; ++l) {
      edges[l] = __fadd_rn(__fadd_rn(v[l + 1], x[l]), x[l + 2]);
      corners[l] = __fadd_rn(__fadd_rn(v[l], n[l + 2]), s[l + 2]);
    }
#pragma unroll
    for (int l = 0; l < 4; l += 2) {
      const f2 lap = lap9_combine(f2(edges[l], edges[l + 1]), f2(corners[l], corners[l + 1]), f2(x[l + 1], x[l + 2]));
      lapv[l] = lap.x;
      lapv[l + 1] = lap.y;
    }
  }

  // One trip.  xN, xC: U(t) windows (column-clamped) of rows j-1, j; xS receives row j+1.  wA, wB: U1
  // windows of rows j-2, j-1; wC receives row j.  eB / eC: raw U1 of my first and last column of rows
  // j-1 / j (IX: wB[1], wB[4]).  sP: V1, W1, S1 of row j-1 (advanced and stored by step 2); sQ receives
  // those of row j.  oj = rowoff(j) + cs (interior body only).
  template <bool EDGE>
  __device__ __forceinline__ void trip(int j, int oj, float (&xN)[6], float (&xC)[6], float (&xS)[6],
                                       float (&wA)[6], float (&wB)[6], float (&wC)[6], float (&eB)[2],
                                       float (&eC)[2], float (&sP)[3][4], float (&sQ)[3][4]) const {
    const int W = g.W, H = g.H, pitch = g.pitch;
    if (EDGE) oj = rowoff(j) + cs;
    // ---------------- step 1 on row j ----------------
    load_enforced_row<4>(a.in[0], EDGE ? xrow(j + 1) : oj + pitch - cs, cw, W, xS);
    // the next trip's lines: a trip is ~400 instructions of arithmetic behind five loads, and only
    // 20 warps per SM are resident to cover their latency
    if (!EDGE || j + kFusePFD <= g1) {
      prefetch_l1(a.in[0] + (EDGE ? xrow(j + 1 + kFusePFD) + cs : oj + (1 + kFusePFD) * pitch));
      const int offn = EDGE ? rowoff(min(j + kFusePFD, H - 1)) + cs : oj + kFusePFD * pitch;
#pragma unroll
      for (int k = 0; k < 3; ++k) prefetch_l1(a.in[k + 1] + offn);
    }
    float u1[4] = {0.f, 0.f, 0.f, 0.f};
    if (!EDGE || (j >= 0 && j < H)) {                         // warp-uniform
      float xraw[4];
      if (!cw.interior_x || (EDGE && (j == 0 || j == H - 1))) {
        VecIO<4>::ld(a.in[0] + oj, xraw);
      } else {
#pragma unroll
        for (int l = 0; l < 4; ++l) xraw[l] = xC[l + 1];
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) VecIO<4>::ld(a.in[k + 1] + oj, sQ[k]);
      float lapv[4];
      lap4(xN, xC, xS, lapv);
      if (PHASE && phase_flag(j)) {
        if (EDGE) add_phase(prow(j - 1) + cs, prow(j) + cs, prow(j + 1) + cs, xN, xC, xS, lapv);
        else add_phase(oj - pitch, oj, oj + pitch, xN, xC, xS, lapv);
      }
      Fenton4v::cell4(sa, xraw, &xC[1], lapv, sQ, u1);
    }

    // ---------------- U1 window of row j: neighbours by shuffle, then the column clamp ----------
    const float left = __shfl_up_sync(0xffffffffu, u1[3], 1);
    const float right = __shfl_down_sync(0xffffffffu, u1[0], 1);
    if (!IX) {
      eC[0] = u1[0];
      eC[1] = u1[3];
    }
    if (cw.interior_x) {
      wC[0] = left; wC[1] = u1[0]; wC[2] = u1[1]; wC[3] = u1[2]; wC[4] = u1[3]; wC[5] = right;
    } else {
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        const int src = clampi(cs - 1 + q, 1, W - 2) - cs;    // -1 .. 4
        wC[q] = src < 0 ? left : (src > 3 ? right : pick4(u1, src));
      }
    }

    // ---------------- step 2 on row r = j - 1 ----------------
    const int r = j - 1;
    if (!EDGE || r >= g0) {                                   // warp-uniform; r < g1 because j <= g1
      float nN[6], nC[6], nS[6];
      if (!EDGE || (r >= 2 && r <= H - 3)) {
#pragma unroll
        for (int q = 0; q < 6; ++q) { nN[q] = wA[q]; nC[q] = wB[q]; nS[q] = wC[q]; }
      } else {                                                // row clamp on the two border rows
        const int iN = clampi(r - 1, 1, H - 2) - (r - 1), iC = clampi(r, 1, H - 2) - (r - 1),
                  iS = clampi(r + 1, 1, H - 2) - (r - 1);     // 0 -> wA, 1 -> wB, 2 -> wC
#pragma unroll
        for (int q = 0; q < 6; ++q) {
          nN[q] = iN == 0 ? wA[q] : (iN == 1 ? wB[q] : wC[q]);
          nC[q] = iC == 0 ? wA[q] : (iC == 1 ? wB[q] : wC[q]);
          nS[q] = iS == 0 ? wA[q] : (iS == 1 ? wB[q] : wC[q]);
        }
      }
      const int orr = oj - pitch;                             // my columns of row r
      float u2[4], lapv[4];
      lap4(nN, nC, nS, lapv);
      if (PHASE && phase_flag(r)) {
        if (EDGE) add_phase(prow(r - 1) + cs, prow(r) + cs, prow(r + 1) + cs, nN, nC, nS, lapv);
        else add_phase(orr - pitch, orr, orr + pitch, nN, nC, nS, lapv);
      }
      const float raw2[4] = {IX ? wB[1] : eB[0], wB[2], wB[3], IX ? wB[4] : eB[1]};
      Fenton4v::cell4(sa, raw2, &nC[1], lapv, sP, u2);
      if (emit_lane) {                                        // emitting lanes are valid: cs == c
        VecIO<4>::st(a.out[0] + orr, u2);
#pragma unroll
        for (int k = 0; k < 3; ++k) VecIO<4>::st(a.out[k + 1] + orr, sP[k]);
      }
    }
  }

  __device__ __forceinline__ void run() const {
    float X0[6], X1[6], X2[6];           // U(t) windows
    float W0[6], W1[6], W2[6];           // U1 windows
    float E0[2] = {0.f, 0.f}, E1[2], E2[2];
    float S0[3][4], S1[3][4], S2[3][4];  // V1, W1, S1
#pragma unroll
    for (int q = 0; q < 6; ++q) W0[q] = W1[q] = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int l = 0; l < 4; ++l) S0[k][l] = 0.f;

    int j = g0 - 1;
    load_enforced_row<4>(a.in[0], xrow(j - 1), cw, g.W, X0);
    load_enforced_row<4>(a.in[0], xrow(j), cw, g.W, X1);

    // interior trips [js, je): a multiple of three; the remainder runs through the edge body before them
    const int jf = max(g0 + 1, 3), je = min(g1 - kFusePFD, g.H - 3) + 1, js = jf + max(0, je - jf) % 3;
#pragma unroll 1
    while (j <= g1) {
      if (IX && j == js && js < je) {
        const int pitch = g.pitch, oe = rowoff(je) + cs;
#pragma unroll 1
        for (int oj = rowoff(j) + cs; oj != oe; j += 3, oj += 3 * pitch) {
          trip<false>(j, oj, X0, X1, X2, W0, W1, W2, E0, E1, S0, S1);
          trip<false>(j + 1, oj + pitch, X1, X2, X0, W1, W2, W0, E1, E2, S1, S2);
          trip<false>(j + 2, oj + 2 * pitch, X2, X0, X1, W2, W0, W1, E2, E0, S2, S0);
        }
        j = je;
        continue;
      }
      trip<true>(j, 0, X0, X1, X2, W0, W1, W2, E0, E1, S0, S1);
#pragma unroll
      for (int q = 0; q < 6; ++q) { X0[q] = X1[q]; X1[q] = X2[q]; W0[q] = W1[q]; W1[q] = W2[q]; }
      E0[0] = E1[0];
      E0[1] = E1[1];
#pragma unroll
      for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int l = 0; l < 4; ++l) S0[k][l] = S1[k][l];
      ++j;
    }
  }
};

// the phase-field flavour needs ~20 more registers for the phi windows: one CTA per SM fewer
template <bool PHASE, bool Z>
__global__ void __launch_bounds__(kBX * kFuseBY, (kFuseMinB - (PHASE ? 1 : 0)) * 4 / kFuseBY)
fenton_fused2_kernel(const Geom g, const Fused2Args a) {
  const int c0 = blockIdx.x * kFuseCols - 4;                  // first column of lane 0
  const int blk = blockIdx.y * blockDim.y + threadIdx.y;
  const int g0 = g.row0 + a.lr0 + blk * a.R;                  // my output rows [g0, g1)
  const int g1 = min(g0 + a.R, g.row0 + a.lr0 + a.nrows);
  if (g0 >= g1) return;                                       // warp-uniform
  // lane 0 reads from column c0 - 1 >= 1, lane 31 up to c0 + 128 <= W - 2: no lane clamps
  if (c0 >= 2 && c0 + 128 <= g.W - 2) Fused2March<PHASE, true, Z>(g, a, c0, g0, g1).run();
  else Fused2March<PHASE, false, Z>(g, a, c0, g0, g1).run();
}

// Output rows per warp R.  A row block costs R + 2 first-step rows, so deep marches are cheaper per
// output row, but the grid is only a few waves of 148 SMs x kFuseMinB CTAs at 4096^2 and a
// badly filled last wave costs more than the two extra rows: pick the R in [8, 48] that minimises
// waves x (R + 2) (4096^2: R = 25, two full waves, instead of 1.5 waves at R = 32: 235 -> see
// profiles/r1_tuning_log.md).  The result does not depend on R (same arithmetic per cell).
inline cudaError_t launch_fused2(const Geom& g, Fused2Args a, cudaStream_t st, int sms) {
  if (a.nrows <= 0) return cudaSuccess;
  const long nseg = (g.W + kFuseCols - 1) / kFuseCols;
  constexpr int BY = kFuseBY;
  auto ctas = [&](int R) { return nseg * (((a.nrows + R - 1) / R + BY - 1) / BY) * a.nz; };
  const long slots = (long)sms * ((kFuseMinB - (a.phase ? 1 : 0)) * 4 / BY);
  int R = 8;
  long best = -1;
  for (int r = 8; r <= 48; ++r) {
    const long waves = (ctas(r) + slots - 1) / slots;
    const long cost = waves * (r + 2);
    if (best < 0 || cost < best || (cost == best && r > R)) { best = cost; R = r; }
  }
  a.R = R;
  dim3 block(kBX, BY), grid((unsigned)nseg, (unsigned)(((a.nrows + R - 1) / R + BY - 1) / BY), (unsigned)a.nz);
  if (preload_only()) {
    cudaFuncAttributes fa;
    return a.phase ? cudaFuncGetAttributes(&fa, fenton_fused2_kernel<true, false>)
                   : cudaFuncGetAttributes(&fa, fenton_fused2_kernel<false, false>);
  }
  const int n = snprintf(last_kernel_name(), 160, "fenton_fused2_kernel<PHASE=%d>,R=%d", a.phase ? 1 : 0, R);
  if (a.nz > 1) snprintf(last_kernel_name() + n, 160 - n, ",Z=%d", a.nz);
  if (a.nz > 1) {
    if (a.phase) fenton_fused2_kernel<true, true><<<grid, block, 0, st>>>(g, a);
    else fenton_fused2_kernel<false, true><<<grid, block, 0, st>>>(g, a);
  } else if (a.phase) {
    fenton_fused2_kernel<true, false><<<grid, block, 0, st>>>(g, a);
  } else {
    fenton_fused2_kernel<false, false><<<grid, block, 0, st>>>(g, a);
  }
  return cudaGetLastError();
}

}  // namespace fib
