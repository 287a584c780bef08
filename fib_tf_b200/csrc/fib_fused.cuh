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
constexpr int kFuseMinB = 5;     // resident CTAs per SM without the phase field
constexpr int kFusePFD = 1;      // prefetch distance in rows

struct Fused2Args {
  const float* in[4];   // U, V, W, S at time t   (halo layout, kFuseHalo rows above and below)
  float* out[4];        // the same at time t + 2 dt
  const float* phase;   // phi in the SAME halo layout (kFuseHalo rows), or nullptr
  const unsigned char* pmask;   // [rows + 2][pmask_pitch], local rows -1 .. rows: 1 where the phase term
  int pmask_pitch;              //   of a 32-column block can be non-zero (fib_set_phase)
  int lr0, nrows;       // local OUTPUT row range of this launch
  int R;                // output rows per warp
  Fenton4v::Params p;
};

__device__ __forceinline__ float pick4(const float (&v)[4], int i) {
  return i == 0 ? v[0] : (i == 1 ? v[1] : (i == 2 ? v[2] : v[3]));
}

// the phase-field flavour needs ~20 more registers for the phi windows: one CTA per SM fewer
template <bool PHASE>
__global__ void __launch_bounds__(kBX * kFuseBY, (kFuseMinB - (PHASE ? 1 : 0)) * 4 / kFuseBY)
fenton_fused2_kernel(const Geom g, const Fused2Args a) {
  const int lane = threadIdx.x;
  const int c = blockIdx.x * kFuseCols - 4 + lane * 4;        // first of my four columns
  const int blk = blockIdx.y * blockDim.y + threadIdx.y;
  const int g0 = g.row0 + a.lr0 + blk * a.R;                  // my output rows [g0, g1)
  const int g1 = min(g0 + a.R, g.row0 + a.lr0 + a.nrows);
  if (g0 >= g1) return;                                       // warp-uniform
  const int W = g.W, H = g.H, pitch = g.pitch;
  const bool valid = c >= 0 && c < W;                         // W % 4 == 0: all four cells or none
  const int cs = valid ? c : (c < 0 ? 0 : W - 4);             // in-bounds column for addressing
  const bool emit_lane = valid && lane >= 1 && lane <= 30;
  const ColWindow<4> cw(cs, W);
  auto rowoff = [&](int gr) { return (gr - g.row0 + kFuseHalo) * pitch; };
  auto xrow = [&](int gr) { return rowoff(clampi(gr, 1, H - 2)); };
  auto prow = [&](int gr) { return rowoff(reflecti(gr, H)); };
  // the phase term of row gr (ionic.py:70-81), exactly as step_kernel forms it: phi is fetched
  // on demand, only where fib_set_phase flagged the 32-column block
  auto phase_flag = [&](int gr) { return a.pmask[(gr - g.row0 + 1) * a.pmask_pitch + (cs >> 5)] != 0; };
  auto load_phi = [&](int gr, float (&pN)[4], float (&pS)[4], float (&pC)[6]) {
    VecIO<4>::ld(a.phase + (prow(gr - 1) + cs), pN);
    VecIO<4>::ld(a.phase + (prow(gr + 1) + cs), pS);
    load_reflect_row<4>(a.phase, prow(gr), cw, W, pC);
  };
  StepArgs<Fenton4v> sa;
  sa.p = a.p;

  float xN[6], xC[6], xS[6];            // U(t): enforced rows j-1, j, j+1
  float wA[6], wB[6], wC[6];            // U1 windows (column-clamped) of rows j-2, j-1, j
  float eB[2] = {0.f, 0.f}, eC[2];      // raw U1 of my first and last column, rows j-1, j
  float sP[3][4], sQ[3][4];             // V1, W1, S1 of rows j-1, j
#pragma unroll
  for (int q = 0; q < 6; ++q) wA[q] = wB[q] = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int l = 0; l < 4; ++l) sP[k][l] = 0.f;

  int j = g0 - 1;
  load_enforced_row<4>(a.in[0], xrow(j - 1), cw, W, xN);
  load_enforced_row<4>(a.in[0], xrow(j), cw, W, xC);

#pragma unroll 1
  for (; j <= g1; ++j) {
    // ---------------- step 1 on row j ----------------
    load_enforced_row<4>(a.in[0], xrow(j + 1), cw, W, xS);
    // the next iteration's lines: an iteration is ~800 instructions of arithmetic behind five
    // loads, and only 20 warps per SM are resident to cover their latency
    if (j + kFusePFD <= g1) {
      prefetch_l1(a.in[0] + xrow(j + 1 + kFusePFD) + cs);
      const int offn = rowoff(min(j + kFusePFD, H - 1)) + cs;
#pragma unroll
      for (int k = 0; k < 3; ++k) prefetch_l1(a.in[k + 1] + offn);
    }
    float u1[4] = {0.f, 0.f, 0.f, 0.f};
    if (j >= 0 && j < H) {                                    // warp-uniform
      const int off = rowoff(j) + cs;
      float xraw[4];
      if (!cw.interior_x || j == 0 || j == H - 1) {
        VecIO<4>::ld(a.in[0] + off, xraw);
      } else {
#pragma unroll
        for (int l = 0; l < 4; ++l) xraw[l] = xC[l + 1];
      }
#pragma unroll
      for (int k = 0; k < 3; ++k) VecIO<4>::ld(a.in[k + 1] + off, sQ[k]);
      float pN[4], pS[4], pC[6];
      bool ph = false;
      if (PHASE) {
        ph = phase_flag(j);
        if (ph) load_phi(j, pN, pS, pC);
      }
      float lapv[4];
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        float lap = lap9(xN[l + 1], xS[l + 1], xC[l], xC[l + 2], xN[l], xS[l], xN[l + 2],
                         xS[l + 2], xC[l + 1]);
        if (PHASE && ph)
          lap = __fadd_rn(lap, phase_term(xN[l + 1], xS[l + 1], xC[l], xC[l + 2], pN[l], pS[l],
                                          pC[l], pC[l + 2], pC[l + 1]));
        lapv[l] = lap;
      }
      Fenton4v::cell4(sa, xraw, &xC[1], lapv, sQ, u1);
    }
#pragma unroll
    for (int q = 0; q < 6; ++q) { xN[q] = xC[q]; xC[q] = xS[q]; }

    // ---------------- U1 window of row j: neighbours by shuffle, then the column clamp ----------
    const float left = __shfl_up_sync(0xffffffffu, u1[3], 1);
    const float right = __shfl_down_sync(0xffffffffu, u1[0], 1);
    eC[0] = u1[0];
    eC[1] = u1[3];
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
    if (r >= g0) {                                            // warp-uniform; r < g1 because j <= g1
      float nN[6], nC[6], nS[6];
      if (r >= 2 && r <= H - 3) {
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
      float pN[4], pS[4], pC[6];
      bool ph = false;
      if (PHASE) {
        ph = phase_flag(r);
        if (ph) load_phi(r, pN, pS, pC);
      }
      float u2[4], lapv[4];
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        float lap = lap9(nN[l + 1], nS[l + 1], nC[l], nC[l + 2], nN[l], nS[l], nN[l + 2],
                         nS[l + 2], nC[l + 1]);
        if (PHASE && ph)
          lap = __fadd_rn(lap, phase_term(nN[l + 1], nS[l + 1], nC[l], nC[l + 2], pN[l], pS[l],
                                          pC[l], pC[l + 2], pC[l + 1]));
        lapv[l] = lap;
      }
      const float raw2[4] = {eB[0], wB[2], wB[3], eB[1]};
      Fenton4v::cell4(sa, raw2, &nC[1], lapv, sP, u2);
      if (emit_lane) {
        const int off = rowoff(r) + c;
        VecIO<4>::st(a.out[0] + off, u2);
#pragma unroll
        for (int k = 0; k < 3; ++k) VecIO<4>::st(a.out[k + 1] + off, sP[k]);
      }
    }

    // ---------------- slide ----------------
#pragma unroll
    for (int q = 0; q < 6; ++q) { wA[q] = wB[q]; wB[q] = wC[q]; }
    eB[0] = eC[0];
    eB[1] = eC[1];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int l = 0; l < 4; ++l) sP[k][l] = sQ[k][l];
  }
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
  auto ctas = [&](int R) { return nseg * (((a.nrows + R - 1) / R + BY - 1) / BY); };
  const long slots = (long)sms * ((kFuseMinB - (a.phase ? 1 : 0)) * 4 / BY);
  int R = 8;
  long best = -1;
  for (int r = 8; r <= 48; ++r) {
    const long waves = (ctas(r) + slots - 1) / slots;
    const long cost = waves * (r + 2);
    if (best < 0 || cost < best || (cost == best && r > R)) { best = cost; R = r; }
  }
  a.R = R;
  dim3 block(kBX, BY), grid((unsigned)nseg, (unsigned)(((a.nrows + R - 1) / R + BY - 1) / BY));
  if (preload_only()) {
    cudaFuncAttributes fa;
    return a.phase ? cudaFuncGetAttributes(&fa, fenton_fused2_kernel<true>)
                   : cudaFuncGetAttributes(&fa, fenton_fused2_kernel<false>);
  }
  snprintf(last_kernel_name(), 160, "fenton_fused2_kernel<PHASE=%d>,R=%d", a.phase ? 1 : 0, R);
  if (a.phase) fenton_fused2_kernel<true><<<grid, block, 0, st>>>(g, a);
  else fenton_fused2_kernel<false><<<grid, block, 0, st>>>(g, a);
  return cudaGetLastError();
}

}  // namespace fib
