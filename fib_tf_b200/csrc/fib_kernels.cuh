// fib_kernels.cuh -- the generic fused step kernel: one launch = one explicit time step of one
// shard (or of a row range of it): boundary + Laplacian + phase term + pointwise ionic update.
//
// Work decomposition (HBM-bound stencil + pointwise ODEs; no tensor cores by design):
//   * a thread owns VEC consecutive cells of a row (one 16-B access per plane for VEC=4) and
//     MARCHES down R rows, keeping the 3-row window of the diffusing variable in registers, so
//     each of its rows is fetched once per strip instead of three times;
//   * a warp covers 32*VEC contiguous columns -> every plane access is a full 128-B line per
//     4 lanes, perfectly coalesced; vertically adjacent warps of a CTA share the strip-edge rows
//     through L1;
//   * only the diffusing variable is ping-ponged (xin -> xout); every other plane is updated in
//     place, so the algorithmic traffic is exactly one read + one write per state variable.
#pragma once
#include <stdio.h>
#include <stdlib.h>

#include <type_traits>

#include "fib_stencil.cuh"

namespace fib {

// A model M provides:
//   NS            number of non-diffusing planes
//   NEED_RAW      reaction term reads the un-enforced centre value (Fenton 4v, fenton.py:101)
//   NEED_LAP      step needs the stencil (false for the Courtemanche 'slow' op)
//   STORE_X       step writes the diffusing variable
//   min_blocks(v, ph) resident CTAs per SM the register allocator must leave room for, v cells per thread,
//                 ph = phase-field flavour (needs more registers)
//   PREFETCH      prefetch the next marching row's lines into L1
//   PACKED        with two cells per thread, run them as one f2 pair (packed fp32, fib_math.cuh)
//   stores(k)     plane k is written by this step
//   struct Params (uniform scalars / small tables; lives in the kernel parameter bank)
//   cell(p, xraw, x0, lap, s[NS], xnew)
template <class M>
struct StepArgs {
  const float* xin;              // diffusing variable, halo layout
  float* xout;                   // ping-pong target (halo layout)
  float* s[M::NS > 0 ? M::NS : 1];  // non-diffusing planes (in place)
  const float* phase;            // halo layout, or nullptr
  const unsigned char* pmask;    // [rows][pmask_pitch]: 1 where the phase term of a 32-column block
  int pmask_pitch;               //   can be non-zero (fib_set_phase), 0 where phi is locally constant
  const float* lut;              // Courtemanche table, transposed [30][160] (global), or nullptr
  int lr0, nrows;                // local row range [lr0, lr0+nrows) processed by this launch
  // Replicas (fib_config.replicas): the launch steps nz independent grids of g.H rows, stacked in every
  // plane as one grid of nz * g.H rows; blockIdx.z = the replica.  zddt: per-replica p.ddt, or nullptr
  int nz;
  const float* zddt;
  typename M::Params p;
};

// The kernels' batched flavour (Z = true) takes its arguments as StepArgsZ: the same fields, but the cell
// functions read replica blockIdx.z's diffusion factor from zddt.  The unbatched flavour is the kernel as it
// was before replicas, instruction for instruction.
template <class M>
struct StepArgsZ : StepArgs<M> {};
template <class M, bool Z>
using StepArgsOf = typename std::conditional<Z, StepArgsZ<M>, StepArgs<M>>::type;

// The state rows of replica blockIdx.z start at local row blockIdx.z * g.H of every plane: a block addresses
// row gr of its replica as local row gr - zrow0(g), and never leaves it (the stencil clamps within the
// replica), so a seam needs no halo rows
template <bool Z>
__device__ __forceinline__ int zrow0(const Geom& g) { return Z ? g.row0 - (int)blockIdx.z * g.H : g.row0; }
// the diffusion factor p.ddt = fp32(diff * dt) the cell functions use: replica blockIdx.z's own, folded in double
// on the host, in the batched flavour; A = StepArgs, StepArgsZ or a wrapper with a member `p` only
template <class A>
__device__ __forceinline__ float ddt_of(const A& a) { return a.p.ddt; }
template <class M>
__device__ __forceinline__ float ddt_of(const StepArgsZ<M>& a) { return __ldg(a.zddt + blockIdx.z); }

constexpr int kBX = 32;   // threads along columns (one warp)
__device__ __forceinline__ void prefetch_l1(const float* p) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}
// grids up to this many cells use VEC_SMALL cells per thread (measured crossover for BR: 512^2 -> 1 cell
// per thread 49 vs 43 Gcell-steps/s, 640^2 -> 2 cells per thread 59 vs 53)
constexpr long kSmallGridCells = 320L * 1024;

// Set around a launch wrapper: do not launch, only make sure the kernel is LOADED (the runtime loads
// kernels lazily on first use, and that load waits for copies in flight -- fatal for the pipelined
// upload, whose whole point is to launch behind them; see preload_kernels in fib_capi.cu)
inline bool& preload_only() {
  static thread_local bool on = false;
  return on;
}
// the flavour launched last on this thread (fib_last_kernel): tests use it to prove which
// instantiation -- cells per thread, marching depth -- they compared with the oracle
inline char* last_kernel_name() {
  static thread_local char name[160] = "";
  return name;
}

template <class M, int VEC, int R, int BY, bool PHASE, bool Z>
__global__ void __launch_bounds__(kBX* BY, M::min_blocks(VEC, PHASE))
step_kernel(const Geom g, const StepArgsOf<M, Z> a) {
  const int row0 = zrow0<Z>(g);                                 // g.row0, in this replica's rows
  const int c = (blockIdx.x * kBX + threadIdx.x) * VEC;
  const int strip = blockIdx.y * BY + threadIdx.y;
  const int gr0 = g.row0 + a.lr0 + strip * R;                 // first global row of my strip
  const int gend = min(gr0 + R, g.row0 + a.lr0 + a.nrows);    // one past my last row
  if (c >= g.W || gr0 >= gend) return;

  // All plane offsets are 32-bit ELEMENT indices (one IMAD.WIDE per address); fib_create rejects
  // shards with (rows+2)*pitch >= 2^31.
  const int pitch = g.pitch;
  const ColWindow<VEC> cw(c, g.W);
  // element index of the start of (clamped / reflected) global row `gr` in a halo-layout plane
  auto xrow = [&](int gr) { return (clampi(gr, 1, g.H - 2) - row0 + 1) * pitch; };
  auto prow = [&](int gr) { return (reflecti(gr, g.H) - row0 + 1) * pitch; };

  float xN[VEC + 2], xC[VEC + 2], xS[VEC + 2];
  if (M::NEED_LAP) load_enforced_row<VEC>(a.xin, xrow(gr0 - 1), cw, g.W, xN);
  load_enforced_row<VEC>(a.xin, xrow(gr0), cw, g.W, xC);

  int off = (gr0 - row0) * pitch + c;            // my cell in a non-halo plane; += pitch per row
#pragma unroll
  for (int i = 0; i < R; ++i, off += pitch) {
    const int gr = gr0 + i;
    if (gr < gend) {
      if (M::NEED_LAP) load_enforced_row<VEC>(a.xin, xrow(gr + 1), cw, g.W, xS);
      // next marching row: pull its lines towards L1 while this row computes (4v +2 %, BR +5 %;
      // off for Courtemanche: 21 planes of prefetches evict the L1-resident table, LUT flavour -31 %)
      if (M::PREFETCH && R > 1 && i + 1 < R && gr + 1 < gend) {
#pragma unroll
        for (int k = 0; k < M::NS; ++k) prefetch_l1(a.s[k] + (off + pitch));
        if (M::NEED_LAP) prefetch_l1(a.xin + (xrow(gr + 2) + c));
      }
      // Phase field: the term is identically 0 wherever phi is locally constant (most of the
      // domain: phi == 1 away from the holes), so phi is only fetched for the 32-column blocks
      // that fib_set_phase flagged; there it is read on demand (no marching window).
      float pN[VEC], pS[VEC], pC[VEC + 2];
      bool ph = false;
      if (PHASE && M::NEED_LAP) {
        ph = a.pmask[(gr - row0) * a.pmask_pitch + (c >> 5)] != 0;
        if (ph) {
          VecIO<VEC>::ld(a.phase + (prow(gr - 1) + c), pN);
          VecIO<VEC>::ld(a.phase + (prow(gr + 1) + c), pS);
          load_reflect_row<VEC>(a.phase, prow(gr), cw, g.W, pC);
        }
      }
      // raw centre values: differ from the enforced ones only on the global border ring
      float xraw[VEC];
      if (M::NEED_RAW && (!cw.interior_x || gr == 0 || gr == g.H - 1)) {
        VecIO<VEC>::ld(a.xin + (off + pitch), xraw);
      } else {
#pragma unroll
        for (int l = 0; l < VEC; ++l) xraw[l] = xC[l + 1];
      }
      float sv[M::NS > 0 ? M::NS : 1][VEC];
#pragma unroll
      for (int k = 0; k < M::NS; ++k) VecIO<VEC>::ld(a.s[k] + off, sv[k]);

      float xnew[VEC], lapv[VEC];
#pragma unroll
      for (int l = 0; l < VEC; ++l) {
        float lap = 0.f;
        if (M::NEED_LAP) {
          lap = lap9(xN[l + 1], xS[l + 1], xC[l], xC[l + 2], xN[l], xS[l], xN[l + 2], xS[l + 2],
                     xC[l + 1]);
          if (PHASE && ph)
            lap = __fadd_rn(lap, phase_term(xN[l + 1], xS[l + 1], xC[l], xC[l + 2], pN[l], pS[l],
                                            pC[l], pC[l + 2], pC[l + 1]));
        }
        lapv[l] = lap;
      }
      if constexpr (M::PACKED && VEC % 2 == 0) {
        // the cells of a thread as packed PAIRS: every multiply-add of the ionic update is a single
        // FFMA2 / FMUL2 / FADD2 for two cells (fib_math.cuh); per lane the arithmetic is that of the
        // scalar flavour of the same source
#pragma unroll
        for (int l = 0; l < VEC; l += 2) {
          f2 sp[M::NS > 0 ? M::NS : 1];
#pragma unroll
          for (int k = 0; k < M::NS; ++k) sp[k] = f2(sv[k][l], sv[k][l + 1]);
          f2 xn;
          M::cell(a, f2(xraw[l], xraw[l + 1]), f2(xC[l + 1], xC[l + 2]), f2(lapv[l], lapv[l + 1]), sp, xn);
          xnew[l] = xn.x;
          xnew[l + 1] = xn.y;
#pragma unroll
          for (int k = 0; k < M::NS; ++k) { sv[k][l] = sp[k].x; sv[k][l + 1] = sp[k].y; }
        }
      } else {
#pragma unroll
        for (int l = 0; l < VEC; ++l) {
          float sl[M::NS > 0 ? M::NS : 1];
#pragma unroll
          for (int k = 0; k < M::NS; ++k) sl[k] = sv[k][l];
          M::cell(a, xraw[l], xC[l + 1], lapv[l], sl, xnew[l]);
#pragma unroll
          for (int k = 0; k < M::NS; ++k) sv[k][l] = sl[k];
        }
      }
#pragma unroll
      for (int k = 0; k < M::NS; ++k)
        if (M::stores(k)) VecIO<VEC>::st(a.s[k] + off, sv[k]);
      if (M::STORE_X) VecIO<VEC>::st(a.xout + (off + pitch), xnew);

      if (M::NEED_LAP) {
#pragma unroll
        for (int j = 0; j < VEC + 2; ++j) { xN[j] = xC[j]; xC[j] = xS[j]; }
      } else if (i + 1 < R && gr + 1 < gend) {
        load_enforced_row<VEC>(a.xin, xrow(gr + 1), cw, g.W, xC);
      }
    }
  }
}

template <class M, int VEC, int R, int BY, bool PHASE, bool Z>
inline cudaError_t launch_step_r(const Geom& g, const StepArgs<M>& a, cudaStream_t st) {
  const int ncg = (g.W + VEC - 1) / VEC;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(kBX, BY);
  cfg.gridDim = dim3((ncg + kBX - 1) / kBX, ((a.nrows + R - 1) / R + BY - 1) / BY, a.nz);
  cfg.stream = st;
  if (preload_only()) {
    cudaFuncAttributes fa;
    return cudaFuncGetAttributes(&fa, step_kernel<M, VEC, R, BY, PHASE, Z>);
  }
  const int n = snprintf(last_kernel_name(), 160, "step_kernel<%s,VEC=%d,R=%d,BY=%d,PHASE=%d>", M::name(), VEC, R,
                         BY, PHASE ? 1 : 0);
  if (a.nz > 1) snprintf(last_kernel_name() + n, 160 - n, ",Z=%d", a.nz);
  StepArgsOf<M, Z> az;
  static_cast<StepArgs<M>&>(az) = a;
  return cudaLaunchKernelEx(&cfg, step_kernel<M, VEC, R, BY, PHASE, Z>, g, az);
}

// Picks the marching depth R: as deep as possible while the grid (all replicas) still has >= 4 CTAs per SM
// (148 SMs); small grids (512^2) fall back to R = 1 and are launch-latency bound anyway.
template <class M, int VEC, int BY, bool PHASE, bool Z>
inline cudaError_t launch_step_p(const Geom& g, const StepArgs<M>& a, cudaStream_t st, int sms) {
  const int ncg = (g.W + VEC - 1) / VEC;
  const long bx = (ncg + kBX - 1) / kBX;
  auto blocks = [&](int R) { return bx * (((a.nrows + R - 1) / R + BY - 1) / BY) * a.nz; };
  const long want = 4L * sms;
  if (M::MAX_R >= 8 && M::AUTO_R >= 8 && blocks(8) >= want) return launch_step_r<M, VEC, (M::MAX_R >= 8 ? 8 : 1), BY, PHASE, Z>(g, a, st);
  if (M::MAX_R >= 4 && M::AUTO_R >= 4 && blocks(4) >= want) return launch_step_r<M, VEC, (M::MAX_R >= 4 ? 4 : 1), BY, PHASE, Z>(g, a, st);
  if (M::MAX_R >= 2 && M::AUTO_R >= 2 && blocks(2) >= want) return launch_step_r<M, VEC, (M::MAX_R >= 2 ? 2 : 1), BY, PHASE, Z>(g, a, st);
  return launch_step_r<M, VEC, 1, BY, PHASE, Z>(g, a, st);
}

template <class M>
inline cudaError_t launch_step(const Geom& g, const StepArgs<M>& a, cudaStream_t st, int sms) {
  if (a.nrows <= 0) return cudaSuccess;
  const bool ph = a.phase && M::NEED_LAP;
  // Small grids (e.g. the reference's 512^2 configs) cannot fill 148 SMs with the
  // wide flavour: fall back to one cell per thread there (twice the CTAs, no tail wave).  The
  // choice depends on the GLOBAL grid only (all replicas), so every shard and every row-range launch of a run
  // uses the same flavour as the unsharded run.
  static const long small_cells = getenv("FIB_SMALL_CELLS") ? atol(getenv("FIB_SMALL_CELLS")) : kSmallGridCells;
  const bool small = M::VEC > 1 && M::VEC_SMALL != M::VEC && (long)g.H * g.W * a.nz <= small_cells;
  auto go = [&](auto z) {
    constexpr bool Z = decltype(z)::value;
    if (small) {
      if (ph) return launch_step_p<M, M::VEC_SMALL, M::BY, true, Z>(g, a, st, sms);
      return launch_step_p<M, M::VEC_SMALL, M::BY, false, Z>(g, a, st, sms);
    }
    if (ph) return launch_step_p<M, M::VEC, M::BY, true, Z>(g, a, st, sms);
    return launch_step_p<M, M::VEC, M::BY, false, Z>(g, a, st, sms);
  };
  return a.nz > 1 ? go(std::true_type()) : go(std::false_type());
}

}  // namespace fib
