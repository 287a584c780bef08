// fib_persist.cuh -- the persistent on-chip kernel for the latency regime (the reference's own
// 512 x 512 configurations, BASELINE configs 1 and 2): ONE launch advances a whole run() iteration
// (10 time steps of 4v, 5 of Beeler-Reuter; fenton.py:133-138, br.py:96-107) with the state resident
// on chip between the steps.
//
// Why: a 512^2 state is 4-8 MiB.  One step per launch leaves such a grid launch-latency bound (3.1 us
// per 4v step against 1.3 us of HBM time and ~0.7 us of issue time, profiles/r1_suite.json); k-step
// temporal blocking by halo recomputation would double the arithmetic at this tile size.  Here
// nothing is recomputed and nothing goes through HBM between steps:
//
//   * the grid is cut into row tiles of TH rows x W columns (W <= 512), one tile per CTA, one CTA per SM
//     (cooperative launch: all CTAs are co-resident by construction);
//   * TMA 2-D tile loads (cp.async.bulk.tensor, mbarrier completion) bring the tile into shared memory at
//     the start; the non-diffusing planes then live in REGISTERS (a thread owns one column of its tile)
//     and the diffusing variable in a double-buffered shared-memory tile; TMA tile stores write
//     everything back once at the end;
//   * per step only the two edge rows of the diffusing variable leave the SM, as self-validating
//     8-byte words {value, step number} in a small L2-resident mailbox (the "LL" protocol of NCCL): an
//     aligned 8-byte store is one transaction, so the neighbour simply polls the words it needs until
//     they carry the step it waits for -- no flag, no memory fence, no L1 invalidation on either side.
//     A step first advances the interior rows, which need nothing from outside, and only then the
//     edge rows, so the hand-shake (one L2 store + one L2 load) is hidden behind arithmetic.
//     One __syncthreads per step (the double-buffered shared tile).
//
// Every cell goes through the SAME cell function and the same Laplacian / phase-term code as
// step_kernel (fib_kernels.cuh), with the same clamped index map, and the library is built with
// -fmad=false, so the result is BIT-IDENTICAL to one launch per step (tests/test_gpu_persist.py).
//
// Deadlock safety: inter-CTA waits exist only under a cooperative launch (fib_capi.cu refuses the
// path otherwise); every spin loop is bounded (kSpinLimit polls, ~1 s) and raises *err instead of
// hanging the device.
#pragma once
#include <cuda.h>

#include "fib_activation.cuh"
#include "model_br.cuh"
#include "model_fenton.cuh"

namespace fib {

constexpr int kPersistThreads = 512;      // one thread per column: W <= 512
constexpr int kPersistBox = 256;          // TMA box width (elements; the hardware limit per dimension)
constexpr int kPersistWP = 512 + 64;      // padded row of the diffusing tile: data at +32 floats (128 B)
constexpr unsigned kSpinLimit = 1u << 22;
// mailbox layout: [2 step parities][tiles][2 sides: 0 = top row, 1 = bottom row][kPersistThreads] words
__host__ __device__ constexpr size_t persist_mailbox_words(int tiles) { return (size_t)2 * tiles * 2 * kPersistThreads; }

// ---- PTX wrappers: mbarrier + TMA (SASS: SYNCS / UTMALDG / UTMASTG) ---------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// 2-D tile load global -> shared, completion counted in bytes on `bar`; (x, y) = (column, row)
__device__ __forceinline__ void tma_load_2d(void* dst_smem, const CUtensorMap* map, int x, int y, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
      ::"r"(smem_u32(dst_smem)), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(smem_u32(bar))
      : "memory");
}
// 2-D tile store shared -> global (rows / columns outside the tensor are clipped)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, int x, int y, const void* src_smem) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(src_smem)), "r"(x), "r"(y)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit_wait() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
// one mailbox word: {fp32 value, step number} moved as ONE aligned 8-byte transaction
__device__ __forceinline__ void ll_store(unsigned long long* p, float v, unsigned step) {
  asm volatile("st.relaxed.gpu.global.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(__float_as_uint(v)), "r"(step) : "memory");
}
__device__ __forceinline__ void ll_load(const unsigned long long* p, float& v, unsigned& step) {
  unsigned a, b;
  asm volatile("ld.relaxed.gpu.global.v2.b32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "l"(p) : "memory");
  v = __uint_as_float(a);
  step = b;
}
// ---- arguments --------------------------------------------------------------------------------
constexpr int kPersistMaxIters = 64;      // run() iterations one launch may cover (fib_step with n_iter > 1)

template <int NS>
struct PersistMaps {
  CUtensorMap x[2];     // the diffusing variable's two buffers, owned rows, box {256, TH}
  CUtensorMap s[NS];    // the other planes, box {256, TH}
};

template <class MS, class MF>
struct PersistArgs {
  float* x[2];                 // the same two buffers as plain pointers (halo layout: row g at (g + 1) * pitch)
  int cur;                     // x[cur] holds the state at the start of the launch
  int nsteps;                  // time steps of this launch (dt_per_step)
  int period;                  // time steps per run() iteration (dt_per_step); a launch may cover several iterations
  int slow_first_only;         // 1: only the first step of every iteration is an MS step (br.py's skip schedule), 0: all
  unsigned long long* mail;    // the mailbox (persist_mailbox_words), words {value, step number}
  unsigned base;               // step number of the state at the start of this launch (monotonic over the run)
  int* err;                    // set to 1 if a neighbour wait ran into the spin limit
  unsigned long long* timeline;   // optional (FIB_PERSIST_TIMELINE=1): %globaltimer of the middle tile at kernel
                                  // start, after the TMA loads, after every step, after the TMA stores (ns)
  const float* phase;          // halo layout (one row), or nullptr
  const unsigned char* pmask;  // [rows][pmask_pitch] as in StepArgs
  int pmask_pitch;
  int bw;                      // TMA box width actually encoded (min(256, W rounded up to 4))
  // fib_probe_watch (or ring == nullptr): the thread owning cell (probe_row, probe_col) appends plane
  // probe_var (0 = the diffusing variable, k = state plane k - 1) to the ring after every iteration,
  // exactly what probe_record_kernel does between the iterations of the one-launch-per-step path
  float* ring;
  unsigned long long* ring_count;
  int probe_var, probe_row, probe_col;
  typename MS::Params ps;      // parameters of the MS steps
  typename MF::Params pf;      // parameters of the MF steps
  // fib_activation_watch (ACT instantiations only): the thread owning a cell samples it at the end of every
  // iteration against its last sample in act_prev (global, L2-resident at these sizes: the register file
  // is full), exactly what activation_update_kernel does between the launches of the plain path.  Iteration
  // it of this launch has k - 1 = act_k0 + it; the launch leaves act_k0 + iterations in *act_iter.
  float* act_prev;             // [rows][pitch]
  float* act_maps;             // kActMaps planes of act_plane floats
  size_t act_plane;
  unsigned long long* act_iter;
  unsigned long long act_k0;
  float act_up, act_down;
};

// ---- the kernel ----------------------------------------------------------------------------------
// MS / MF: the cell types of the "slow" and "fast" steps of a schedule (Fenton4v twice; BeelerReuter<C,true>
// and <C,false> for br.py's skip schedule).  TH: rows per tile.  PHASE: phase field present.  ACT: an
// activation map is armed (fib_activation.cuh).
//
// Where the state lives between the steps of a launch:
//   * a thread owns ONE column of its tile: its TH cells of every plane, the diffusing variable included
//     (the raw values), stay in registers;
//   * shared memory holds the ENFORCED diffusing field of the tile plus a one-cell ring, i.e. what the
//     stencil of fib_stencil.cuh reads, Xp[r][c] = X[clamp(r,1,H-2)][clamp(c,1,W-2)], materialised:
//     local row li <-> global row r0 + li - 1, column c at offset 32 + c (columns -1 and W included).
//     Away from the grid's border that is the field itself; on the border the writers duplicate the
//     neighbouring interior value into the ring positions.  Every stencil read is then a plain
//     [li + dr][c + dc] shared-memory load with static offsets -- no clamping, no branches per cell --
//     and the rows of a column are read once per step (marching reuse in registers);
//   * the rows of the neighbour tiles arrive through the mailbox and are written into the ring rows by
//     the thread that will read them (each thread writes the three columns it reads: no barrier).
template <class MS, class MF, int TH, bool PHASE, bool ACT>
__global__ void __launch_bounds__(kPersistThreads, 1)
persist_kernel(const __grid_constant__ PersistMaps<MS::NS> maps, const Geom g, const PersistArgs<MS, MF> a) {
  constexpr int NS = MS::NS;
  static_assert(MS::NS == MF::NS, "slow / fast steps share the state layout");
  static_assert(TH >= 2, "tiles are at least two rows high");
  extern __shared__ __align__(128) unsigned char smem_raw[];
  float* ub = reinterpret_cast<float*>(smem_raw);                 // [2][TH + 2][kPersistWP] enforced field + ring
  float* st = ub + 2 * (TH + 2) * kPersistWP;                     // [NS + 1][2 column blocks][TH][256] TMA staging
  uint64_t* bar = reinterpret_cast<uint64_t*>(st + (NS + 1) * TH * 512);

  const int t = threadIdx.x, tile = blockIdx.x, ntiles = gridDim.x;
  const bool stamp = a.timeline && t == 0 && tile == ntiles / 2;
  auto now = [&](int slot) __attribute__((always_inline)) {
    if (stamp) {
      unsigned long long ns;
      asm volatile("mov.u64 %0, %globaltimer;" : "=l"(ns));
      a.timeline[slot] = ns;
    }
  };
  now(0);
  const int W = g.W, H = g.H, pitch = g.pitch;
  const int r0 = tile * TH;
  const int nrows = min(TH, H - r0);
  const int c = t;
  const bool active = c < W;
  const int nblk = (W + kPersistBox - 1) / kPersistBox;
  // column 0 of local row li of buffer p
  auto urow = [&](int p, int li) __attribute__((always_inline)) { return ub + (p * (TH + 2) + li) * kPersistWP + 32; };
  auto stage = [&](int k, int b) __attribute__((always_inline)) { return st + (k * 2 + b) * TH * kPersistBox; };

  // ---- TMA in: every plane of the tile as {bw, TH} boxes (plane NS = the diffusing variable)
  if (t == 0) {
    mbar_init(bar, 1);
    fence_async_smem();
  }
  __syncthreads();
  if (t == 0) {
    mbar_expect_tx(bar, (uint32_t)((NS + 1) * TH * nblk * a.bw * sizeof(float)));
    for (int b = 0; b < nblk; ++b) {
      tma_load_2d(stage(NS, b), a.cur ? &maps.x[1] : &maps.x[0], b * kPersistBox, r0, bar);
      for (int k = 0; k < NS; ++k) tma_load_2d(stage(k, b), &maps.s[k], b * kPersistBox, r0, bar);
    }
  }
  // meanwhile: which of my cells have a non-trivial phase term (same flags as step_kernel) ...
  unsigned phbits = 0;
  if (PHASE && active) {
#pragma unroll
    for (int i = 0; i < TH; ++i)
      if (i < nrows && a.pmask[(r0 + i) * a.pmask_pitch + (c >> 5)]) phbits |= 1u << i;
  }
  // ... the columns I write (the enforced field duplicates column 1 into 0 and -1, W-2 into W-1 and W) ...
  const int ccl = clampi(c - 1, 1, W - 2), ccc = clampi(c, 1, W - 2), ccr = clampi(c + 1, 1, W - 2);
  const bool wr_own = active && c >= 1 && c <= W - 2, wr_lo = c == 1, wr_hi = c == W - 2;
  auto put = [&](float* row, float v) __attribute__((always_inline)) {
    if (wr_own) row[c] = v;
    if (wr_lo) { row[0] = v; row[-1] = v; }
    if (wr_hi) { row[W - 1] = v; row[W] = v; }
  };
  // ... and which global row local row li shows: src[li] = local index of row clamp(r0 + li - 1, 1, H - 2)
  // (0 = the row above the tile, 1..TH = my rows, TH + 1 = the row below); identity except at the grid's border
  int src[TH + 2];
  bool plain_tile = true;
#pragma unroll
  for (int li = 0; li < TH + 2; ++li) {
    const int gr = r0 + li - 1;
    src[li] = (gr >= -1 && gr <= H) ? clampi(gr, 1, H - 2) - r0 + 1 : -1;
    if (src[li] != li && src[li] >= 0) plain_tile = false;
  }
  const bool need_top = tile > 0, need_bot = tile + 1 < ntiles;
  while (!mbar_try_wait(bar, 0)) {}
  now(1);

  float s[NS][TH], u[TH];
  {
    const int b = c / kPersistBox, cb = c - b * kPersistBox;
#pragma unroll
    for (int i = 0; i < TH; ++i) {
#pragma unroll
      for (int k = 0; k < NS; ++k) s[k][i] = active ? stage(k, b)[i * a.bw + cb] : 0.f;
      u[i] = active ? stage(NS, b)[i * a.bw + cb] : 0.f;
    }
  }

  // the cell functions only look at `.p`: hand them the parameter blocks where they are (kernel
  // parameter space) instead of copies
  struct PS { const typename MS::Params& p; };
  struct PF { const typename MF::Params& p; };
  const PS sa_s{a.ps};
  const PF sa_f{a.pf};

  // rows of the enforced field that show one of MY rows: written from registers (`vals` = my TH values)
  auto write_own = [&](int p, const float (&vals)[TH], int first, int last) __attribute__((always_inline)) {
    if (plain_tile) {
#pragma unroll
      for (int i = 0; i < TH; ++i)
        if (i >= first && i <= last && i < nrows) put(urow(p, i + 1), vals[i]);
    } else {                      // a tile on the grid's border: some rows show a neighbouring row
#pragma unroll
      for (int li = 0; li < TH + 2; ++li)
#pragma unroll
        for (int i = 0; i < TH; ++i)
          if (src[li] == i + 1 && i >= first && i <= last) put(urow(p, li), vals[i]);
    }
  };
  // rows that show a NEIGHBOUR tile's row: each thread writes the three columns it will read itself
  // (the mailbox / plane loads used clamped columns, so these are enforced values already)
  auto write_ring = [&](int p, const float (&rt)[3], const float (&rb)[3]) __attribute__((always_inline)) {
    if (!active) return;
#pragma unroll
    for (int li = 0; li < TH + 2; ++li) {
      if (src[li] == 0) { float* q = urow(p, li) + c; q[-1] = rt[0]; q[0] = rt[1]; q[1] = rt[2]; }
      if (src[li] == TH + 1) { float* q = urow(p, li) + c; q[-1] = rb[0]; q[0] = rb[1]; q[1] = rb[2]; }
    }
  };

  // ---- step 0 input: my rows from registers, the neighbours' rows from the global plane (complete at the
  // start of a launch: previous launch / upload / stimulus -- whatever the mailbox holds)
  {
    const float* xg = a.cur ? a.x[1] : a.x[0];
    float rt[3] = {0.f, 0.f, 0.f}, rb[3] = {0.f, 0.f, 0.f};
    if (active && need_top) {
      const float* q = xg + (size_t)(r0 - 1 + 1) * pitch;
      rt[0] = __ldcg(q + ccl); rt[1] = __ldcg(q + ccc); rt[2] = __ldcg(q + ccr);
    }
    if (active && need_bot) {
      const float* q = xg + (size_t)(r0 + TH + 1) * pitch;
      rb[0] = __ldcg(q + ccl); rb[1] = __ldcg(q + ccc); rb[2] = __ldcg(q + ccr);
    }
    write_own(0, u, 0, TH - 1);
    __syncthreads();              // (the ring rows may overlap rows written above on border tiles: order them)
    write_ring(0, rt, rb);
    __syncthreads();
  }

  // mailbox words of step number n written by `tl`'s side sd (0 = its top row, 1 = its bottom row)
  auto box = [&](unsigned n, int tl, int sd) __attribute__((always_inline)) {
    return a.mail + (((size_t)(n & 1u) * ntiles + tl) * 2 + sd) * kPersistThreads;
  };

  // local rows 1..TH show rows of my own tile (everywhere but on a one-row last tile, whose row H-1 shows H-2)
  bool lazy = true;
#pragma unroll
  for (int li = 1; li <= TH; ++li)
    if (src[li] == 0 || src[li] == TH + 1) lazy = false;
  const bool probe_me = a.ring && active && c == a.probe_col && a.probe_row >= r0 && a.probe_row < r0 + nrows;
  unsigned long long probe_n = probe_me ? *a.ring_count : 0ull;
  int sub = 0;                                               // time step within the current iteration
  unsigned long long act_k = a.act_k0;                       // ACT: k - 1 of the current iteration
  for (int step = 0; step < a.nsteps; ++step) {
    const int p = step & 1;                                  // shared buffer holding the state this step reads
    const bool slow = !a.slow_first_only || sub == 0;
    const unsigned want = a.base + step;                     // step number of that state
    // My six mailbox words (three columns on each side).  All six loads are issued back to back, so one
    // poll costs ONE L2 round trip; the first poll is issued BEFORE the interior rows are advanced and only
    // looked at afterwards, which hides that round trip behind arithmetic when the neighbours are on time.
    float mv[6];
    unsigned mn[6];
    const int mcols[3] = {ccl, ccc, ccr};
    auto ring_poll = [&]() __attribute__((always_inline)) {
#pragma unroll
      for (int sd = 0; sd < 2; ++sd) {
        // the tile above publishes its BOTTOM row (side 1), the tile below its TOP row (side 0)
        const bool need = sd == 0 ? need_top : need_bot;
        const unsigned long long* w = sd == 0 ? box(want, tile - 1, 1) : box(want, tile + 1, 0);
#pragma unroll
        for (int q = 0; q < 3; ++q) {
          if (need) ll_load(w + mcols[q], mv[sd * 3 + q], mn[sd * 3 + q]);
          else { mv[sd * 3 + q] = 0.f; mn[sd * 3 + q] = want; }
        }
      }
    };

    // the three enforced values around my column in local row li
    float T[TH + 2][3];
    auto load_row = [&](int li) __attribute__((always_inline)) {
      const float* q = urow(p, li) + c;
      T[li][0] = q[-1]; T[li][1] = q[0]; T[li][2] = q[1];
    };
    // Laplacian (+ phase term) of my row i: exactly step_kernel's arithmetic on the same values
    auto lap_row = [&](int i) __attribute__((always_inline)) -> float {
      float lap = lap9(T[i][1], T[i + 2][1], T[i + 1][0], T[i + 1][2], T[i][0], T[i + 2][0], T[i][2], T[i + 2][2],
                       T[i + 1][1]);
      if (PHASE && ((phbits >> i) & 1u)) {
        const int gr = r0 + i;
        const float* ph = a.phase;
        const int rN = (reflecti(gr - 1, H) + 1) * pitch, rC = (gr + 1) * pitch, rS = (reflecti(gr + 1, H) + 1) * pitch;
        const float pN = ph[rN + c], pS = ph[rS + c];
        const float pW = ph[rC + clampi(reflecti(c - 1, W), 0, W - 1)], pE = ph[rC + clampi(reflecti(c + 1, W), 0, W - 1)];
        lap = __fadd_rn(lap, phase_term(T[i][1], T[i + 2][1], T[i + 1][0], T[i + 1][2], pN, pS, pW, pE, ph[rC + c]));
      }
      return lap;
    };
    // one cell (row i) / two cells (rows i and j of my column as ONE packed pair, fib_math.cuh) through the
    // model's cell function; u[]: the raw centre values, T[.][1]: the enforced ones.  `lapf` yields the
    // Laplacian(s) when the cell function gets to its last expression (lap_value, fib_math.cuh).
    auto do_row = [&](int i, auto&& lapf) __attribute__((always_inline)) {
      float sl[NS], xnew;
#pragma unroll
      for (int k = 0; k < NS; ++k) sl[k] = s[k][i];
      if (slow) MS::cell(sa_s, u[i], T[i + 1][1], lapf, sl, xnew);
      else MF::cell(sa_f, u[i], T[i + 1][1], lapf, sl, xnew);
#pragma unroll
      for (int k = 0; k < NS; ++k) s[k][i] = sl[k];
      u[i] = xnew;
    };
    auto do_pair = [&](int i, int j, auto&& lapf) __attribute__((always_inline)) {   // j >= nrows: junk lane
      f2 sl[NS], xnew;
#pragma unroll
      for (int k = 0; k < NS; ++k) sl[k] = f2(s[k][i], s[k][j]);
      if (slow) MS::cell(sa_s, f2(u[i], u[j]), f2(T[i + 1][1], T[j + 1][1]), lapf, sl, xnew);
      else MF::cell(sa_f, f2(u[i], u[j]), f2(T[i + 1][1], T[j + 1][1]), lapf, sl, xnew);
#pragma unroll
      for (int k = 0; k < NS; ++k) { s[k][i] = sl[k].x; s[k][j] = sl[k].y; }
      u[i] = xnew.x;
      u[j] = xnew.y;
    };
    constexpr bool kPairs = MS::PACKED && MF::PACKED;

    // interior rows: need nothing from outside the tile.  The FIRST poll of the mailbox goes out in the
    // middle of this phase: late enough for the neighbours' words (stored at the end of their previous
    // step, i.e. about when this step began) to have reached L2, early enough for the round trip to be
    // hidden behind the cell arithmetic.
    const bool poll = step > 0;
    bool polled = false;
    if (active) {
#pragma unroll
      for (int li = 1; li <= TH; ++li) load_row(li);
      if constexpr (kPairs) {
#pragma unroll
        for (int i = 1; i + 1 < TH - 1; i += 2)
          if (i < nrows) {
            const f2 lap(lap_row(i), lap_row(i + 1));
            if (poll && !polled && i + 3 >= TH - 1) ring_poll();       // before the LAST interior pair's cells
            polled |= i + 3 >= TH - 1;
            do_pair(i, i + 1, lap);
          }
      } else {
#pragma unroll
        for (int i = 1; i < TH - 1; ++i)
          if (i < nrows) {
            const float lap = lap_row(i);
            if (poll && !polled && i + 2 >= TH - 1) ring_poll();
            polled |= i + 2 >= TH - 1;
            do_row(i, lap);
          }
      }
      if (poll && !polled) ring_poll();           // (no interior rows: TH = 2, or a short last tile)
    }
    // the neighbours' rows of this step: wait for the mailbox (bounded: raises *err instead of hanging),
    // put them where my stencil reads them
    auto wait_ring = [&]() __attribute__((always_inline)) {
      unsigned spins = 0;
      for (;;) {
        bool ok = true;
#pragma unroll
        for (int q = 0; q < 6; ++q) ok &= mn[q] == want;
        if (ok) break;
        if (++spins > kSpinLimit) { *a.err = 1; break; }
        ring_poll();
      }
      const float rt[3] = {mv[0], mv[1], mv[2]}, rb[3] = {mv[3], mv[4], mv[5]};
      write_ring(p, rt, rb);
    };
    // Edge rows, published to the neighbours straight from registers.  The neighbours' rows are needed for
    // the Laplacian only, and the Laplacian enters a cell in its last expression: on tiles whose own rows
    // are all shown by themselves (`lazy`: every tile but a one-row last tile) the wait sits INSIDE the
    // cell function at that point -- gates, currents and the reaction term of the edge rows are computed
    // while the mailbox words are in flight, and receive -> publish is ring write, Laplacian, two adds.
    if (active) {
      if (poll && !lazy) wait_ring();
      if (!plain_tile && !lazy) {     // the ring write may have refreshed rows loaded earlier
#pragma unroll
        for (int li = 1; li <= TH; ++li) load_row(li);
      }
      auto outer_rows = [&]() __attribute__((always_inline)) {
        if (poll && lazy) wait_ring();
        load_row(0);
        load_row(TH + 1);
      };
      if constexpr (kPairs) {
        do_pair(0, TH - 1, [&]() __attribute__((always_inline)) {
          outer_rows();
          return f2(lap_row(0), lap_row(TH - 1));
        });
      } else {
        do_row(0, [&]() __attribute__((always_inline)) {
          outer_rows();
          return lap_row(0);
        });
        if (TH - 1 < nrows) do_row(TH - 1, lap_row(TH - 1));
      }
      // (the last step's rows are not consumed through the mailbox: the next launch starts from the plane)
      if (need_top) ll_store(box(want + 1, tile, 0) + c, u[0], want + 1);
      if (need_bot) ll_store(box(want + 1, tile, 1) + c, u[TH - 1], want + 1);
      write_own(p ^ 1, u, 0, TH - 1);
    }
    if (++sub == a.period) {    // an iteration ends here
      sub = 0;
      if (probe_me) {
        float v = 0.f;
#pragma unroll
        for (int i = 0; i < TH; ++i)
          if (r0 + i == a.probe_row) {
            v = u[i];
#pragma unroll
            for (int k = 0; k < NS; ++k)
              if (a.probe_var == k + 1) v = s[k][i];
          }
        a.ring[probe_n % FIB_PROBE_RING] = v;
        ++probe_n;
      }
      if constexpr (ACT) {
        if (active) {
          const float k1 = (float)act_k;
#pragma unroll
          for (int i = 0; i < TH; ++i)
            if (i < nrows) {
              const size_t idx = (size_t)(r0 + i) * pitch + c;
              const float pv = a.act_prev[idx];
              a.act_prev[idx] = u[i];
              act_cell(pv, u[i], k1, a.act_up, a.act_down, a.act_maps + idx, a.act_plane);
            }
        }
        ++act_k;
      }
    }
    __syncthreads();            // shared tile of the next step complete, the old one free for reuse
    now(2 + step);
  }
  if (probe_me) *a.ring_count = probe_n;
  if constexpr (ACT) {
    if (tile == 0 && t == 0) *a.act_iter = act_k;
  }

  // ---- TMA out: registers -> staging, then tile stores (rows beyond the grid are clipped)
  if (active) {
    const int b = c / kPersistBox, cb = c - b * kPersistBox;
#pragma unroll
    for (int i = 0; i < TH; ++i) {
#pragma unroll
      for (int k = 0; k < NS; ++k) stage(k, b)[i * a.bw + cb] = s[k][i];
      stage(NS, b)[i * a.bw + cb] = u[i];
    }
  }
  fence_async_smem();
  __syncthreads();
  if (t == 0) {
    const CUtensorMap* mx = ((a.cur + a.nsteps) & 1) ? &maps.x[1] : &maps.x[0];
    for (int b = 0; b < nblk; ++b) {
      tma_store_2d(mx, b * kPersistBox, r0, stage(NS, b));
      for (int k = 0; k < NS; ++k)
        if (MS::stores(k) || MF::stores(k)) tma_store_2d(&maps.s[k], b * kPersistBox, r0, stage(k, b));
    }
    tma_store_commit_wait();
  }
  now(2 + a.nsteps);
}

template <int NS, int TH>
constexpr size_t persist_smem_bytes() {
  return (size_t)(2 * (TH + 2) * kPersistWP + (NS + 1) * TH * 512) * sizeof(float) + 64;
}

}  // namespace fib
