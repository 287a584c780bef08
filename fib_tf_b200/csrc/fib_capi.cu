// fib_capi.cu -- implementation of include/fib_b200.h (the C ABI of libfibb200.so).
// Owns device memory (SoA fp32 planes), the stream / events / CUDA graphs, the step schedule of
// every model and the halo exchange.  sm_100a only; there is no CPU path in this library.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/fib_b200.h"
#include "model_br.cuh"
#include "model_court.cuh"
#include "model_fenton.cuh"
#include "fib_fused.cuh"
#include "fib_persist.cuh"

using namespace fib;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess)                                                                    \
      return fail(FIB_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                  __LINE__);                                                                  \
  } while (0)

// ------------------------------------------------------------------------------------------
// NCCL, resolved at run time (the library has no link-time dependency on libnccl)
// ------------------------------------------------------------------------------------------
struct Uid { char bytes[128]; };   // ncclUniqueId
struct Nccl {
  void* h = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, Uid /*by value*/, int) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  int (*Send)(const void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*Recv)(void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static Nccl g_nccl;

static int nccl_load() {
  if (g_nccl.h) return 0;
  const char* names[] = {getenv("FIB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    if (!n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) return fail(FIB_E_NCCL, "cannot dlopen libnccl.so.2 (%s)", dlerror());
#define SYM(field, name)                                                          \
  *(void**)(&g_nccl.field) = dlsym(h, name);                                      \
  if (!g_nccl.field) return fail(FIB_E_NCCL, "libnccl lacks symbol %s", name);
  SYM(GetUniqueId, "ncclGetUniqueId")
  SYM(CommInitRank, "ncclCommInitRank")
  SYM(CommDestroy, "ncclCommDestroy")
  SYM(Send, "ncclSend")
  SYM(Recv, "ncclRecv")
  SYM(GroupStart, "ncclGroupStart")
  SYM(GroupEnd, "ncclGroupEnd")
  SYM(GetErrorString, "ncclGetErrorString")
#undef SYM
  g_nccl.h = h;
  return 0;
}
#define NC(call)                                                                             \
  do {                                                                                       \
    int r_ = (call);                                                                         \
    if (r_ != 0) return fail(FIB_E_NCCL, "%s failed: %s", #call, g_nccl.GetErrorString(r_)); \
  } while (0)
static const int kNcclFloat = 7;   // ncclFloat32

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
static const char* kFentonVars[] = {"U", "V", "W", "S"};
static const char* kBrVars[] = {"V", "C", "M", "H", "J", "D", "F", "XI"};
static const char* kCourtVars[] = {"V", "_Na_i_", "_m_", "_h_", "_j_", "_K_i_", "_oa_", "_oi_",
                                   "_ua_", "_ui_", "_xr_", "_xs_", "_Ca_i_", "_d_", "_f_", "_f_Ca_",
                                   "_Ca_rel_", "_u_", "_v_", "_w_", "_Ca_up_", "_us_"};

// one captured iteration of `op`: a replay launches `launches` kernels and moves the state from `cur` to `cur_end`
struct GraphKey { int op, cur, cur_end; uint64_t launches; cudaGraphExec_t exec; };

// "The records up to total[k] were produced by the work enqueued before event ev[k]": a fetch of older records
// waits for the covering event only, not for the launches queued behind it.
template <int N>
struct Ledger {
  cudaEvent_t ev[N] = {};
  unsigned long long total[N] = {};
  int next = 0;
  int create() {
    for (auto& e : ev)
      if (!e) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return 0;
  }
  void destroy() {
    for (auto& e : ev)
      if (e) cudaEventDestroy(e);
  }
  int mark(cudaStream_t st, unsigned long long t) {
    CU(cudaEventRecord(ev[next], st));
    total[next] = t;
    next = (next + 1) % N;
    return 0;
  }
  void clear() { for (auto& t : total) t = 0; }
  // the earliest mark that covers the records up to `need`, among those not past `upto`; -1 if there is none
  int covering(unsigned long long need, unsigned long long upto) const {
    int best = -1;
    for (int k = 0; k < N; ++k)
      if (total[k] >= need && total[k] <= upto && (best < 0 || total[k] < total[best])) best = k;
    return best;
  }
};

struct fib_ctx {
  fib_config cfg;
  Geom g;                             // this shard; a batched context: all replicas as one grid of nrep * height rows
  int nrep = 1;                       // replicas (fib_config.replicas)
  float* zddt = nullptr;              // nrep > 1: fp32(diff_b * dt) of every replica (the kernels' StepArgs::zddt)
  int nvars = 0, dt_per_step = 1, sms = 148;
  const char** names = nullptr;
  cudaStream_t stream = nullptr, comm_stream = nullptr, copy_stream = nullptr;
  cudaEvent_t ev_snap_ready = nullptr, ev_snap_done = nullptr;
  float* snap = nullptr;              // device-side staging copy of one plane (async frame grabs)
  bool snap_pending = false;
  cudaEvent_t ev_start = nullptr, ev_stop = nullptr, ev_bnd = nullptr, ev_comm = nullptr,
              ev_group = nullptr;
  float* x[2] = {nullptr, nullptr};   // diffusing variable, ping-pong, halo layout
  int cur = 0;
  int fuse = 1;                       // time steps per launch (cfg.steps_per_launch): 1 or 2
  float* fx[2][4] = {{nullptr}};      // fuse == 2 (fib_fused.cuh): ALL planes ping-ponged, kFuseHalo rows
  float* s[S_COUNT] = {nullptr};      // other planes
  float* phase = nullptr;             // halo layout
  unsigned char* pmask = nullptr;     // [rows][pmask_pitch] non-trivial-phase flags per 32 columns
  int pmask_pitch = 0;
  float* phase2 = nullptr;            // fuse == 2: second copy of phi with kFuseHalo halo rows ...
  unsigned char* pmask2 = nullptr;    // ... and its flags for local rows -1 .. rows: [rows + 2][pmask_pitch]
  float* lut = nullptr;               // 150 x 30, the ABI layout (courtemanche.h order)
  float* lut_t = nullptr;             // 30 x 160 transposed copy the kernels read
  bool have_lut = false, have_cheb = false, halo_dirty = true, comm_pending = false;
  float cheb[12][9];
  uint64_t launches = 0;
  std::vector<GraphKey> graphs;
  double* red = nullptr;              // 2 doubles per replica for reductions
  // ODE iterations enqueued on this context: each observer below counts its own from the value at its arming
  unsigned long long ode_iters = 0;
  unsigned long long since(unsigned long long armed_at) const { return ode_iters - armed_at; }
  // device-side cycle-length probe (fib_probe_watch): one watched cell, a ring of recorded values;
  // fib_replica_probe_watch: the same local cell of every replica, one record of nrep values per iteration
  float* ring = nullptr;              // page-locked, device-visible: a fetch is a stream sync + host reads
  size_t ring_floats = 0;             // allocated
  unsigned long long ring_cap = FIB_PROBE_RING;   // records of the armed watch
  int watch_n = 1;                    // floats per record: 1, or nrep for a replica watch
  bool watch_replicas = false;        // the armed watch is fib_replica_probe_watch's
  unsigned long long* ring_count = nullptr;   // device: the slot the next record goes to
  unsigned long long probe_armed_at = 0;      // records made = since(probe_armed_at)
  unsigned long long ring_fetched = 0;
  Ledger<4> probe_ledger;             // marked after the last few persistent launches (which record in-kernel)
  int watch_var = -1, watch_row = -1, watch_col = -1;
  // activation maps (fib_activation_watch, fib_activation.cuh): armed iff act_maps != nullptr
  float* act_prev = nullptr;          // the last sample of the diffusing variable, [rows][pitch]
  float* act_maps = nullptr;          // kActMaps planes [rows][pitch]
  unsigned long long* act_iter = nullptr;   // device: samples taken since arming (= k - 1 of the next one)
  unsigned long long act_armed_at = 0;      // *act_iter = since(act_armed_at) once the stream has drained
  float act_up = 0.f, act_down = 0.f;
  // frame recorder (fib_frames_watch): armed iff frames != nullptr.  Frame j is the plane at k = fr_first +
  // j * fr_every and lives in slot j % fr_cap; the host knows k, so only recording iterations launch anything.
  float* frames = nullptr;            // [fr_cap][fr_rows][fr_cols]
  int fr_var = 0, fr_first = 0, fr_every = 1, fr_stride = 1, fr_cap = 0;
  int fr_rows = 0, fr_cols = 0, fr_lr0 = 0;   // this shard's frame; fr_lr0 = local row of its first row
  unsigned long long fr_armed_at = 0; // k = since(fr_armed_at)
  unsigned long long fr_fetched = 0;  // frames handed out (or lost to overflow)
  Ledger<256> frame_ledger;           // marked after every launch that records frames
  size_t frame_floats() const { return (size_t)fr_rows * fr_cols; }
  // frames recorded once k iterations have run
  unsigned long long frames_upto(unsigned long long k) const {
    return k < (unsigned long long)fr_first ? 0 : (k - fr_first) / fr_every + 1;
  }
  unsigned long long frames_recorded() const { return frames_upto(since(fr_armed_at)); }
  // checkpoint in flight (fib_checkpoint_begin): ck_parts dense [rows][W] planes, complete at ev_ck on `stream`
  float* ck = nullptr;
  int ck_parts = 0;
  cudaStream_t ck_stream = nullptr;   // fib_checkpoint_read's copies (possibly from another thread)
  cudaEvent_t ev_ck = nullptr;
  float* weights[4] = {nullptr, nullptr, nullptr, nullptr};   // user masks, halo layout like phase
  // pacing (fib_pace_add): entry p stimulates the diffusing variable right after the ODE iterations whose ode_iters
  // is p.at + j * p.every, j < p.count (count 0: every such iteration); dropped once its last beat is enqueued
  struct Pace {
    int id, replica, r0, r1, c0, c1;
    float value, floor_v;
    unsigned long long at, every, count;
    bool fires(unsigned long long n) const {
      return n >= at && (n - at) % every == 0 && (count == 0 || (n - at) / every < count);
    }
    bool done(unsigned long long n) const { return count != 0 && n >= at + (count - 1) * every; }
  };
  std::vector<Pace> paces;
  int pace_ids = 0;                   // ids handed out so far
  // persistent on-chip kernel (fib_persist.cuh): small unsharded 4v / BR grids
  int persist = -1;                   // -1 not decided yet, 0 no, 1 yes
  int persist_th = 0, persist_tiles = 0, persist_bw = 0;
  unsigned long long* pmail = nullptr;   // edge-row mailbox of the persistent kernel, words {value, step number}
  unsigned pbase = 0;
  int pending = 0;                    // ODE iterations accepted by fib_step but not launched yet (see flush_pending)
  // Pipelined upload (fib_set_rect_async of full-width row blocks, in order from one edge of the shard, every
  // plane): the copies run on their own stream; `arrivals` = {the first d_end rows, counted from that edge, of
  // EVERY plane are enqueued up to `ev`}.  Iterations stepped while such a session is open are deferred
  // (unsharded contexts) or asked for explicitly (NCCL shards, fib_step_behind_upload) and then run block by
  // block behind the copies (finish_upload_session).
  struct Arrival { int d_end; cudaEvent_t ev; };   // d = rows counted from the edge the upload started at
  cudaStream_t up_stream = nullptr;
  cudaEvent_t ev_up_begin = nullptr;
  bool up_session = false;
  std::vector<Arrival> arrivals;
  std::vector<int> up_front;          // per plane: the first up_front rows (from the starting edge) are enqueued
  int up_dir = +1;                    // +1: top to bottom, -1: bottom to top (NCCL shards: odd ranks, see below)
  bool pipeline_nccl = true;          // FIB_PIPELINE_NCCL=0: no upload sessions on NCCL-sharded contexts
  std::vector<cudaEvent_t> ev_pool;
  long long pipeline_min_cells = 1ll << 22;   // smaller grids: not worth it (FIB_PIPELINE_MIN_CELLS)
  int pipeline_block_rows = 1024;             // rows per block of the skewed schedule, at least (FIB_PIPELINE_BLOCK_ROWS)
  int* perr = nullptr;                // page-locked, device-visible: raised by a timed-out neighbour wait
  CUtensorMap pmap_x[2], pmap_s[8];
  // NCCL
  void* comm = nullptr;
  int nranks = 1, rank = 0;
  size_t plane_floats() const { return (size_t)g.rows * g.pitch; }
  size_t halo_floats() const { return (size_t)(g.rows + 2) * g.pitch; }
  size_t fused_floats() const { return (size_t)(g.rows + 2 * kFuseHalo) * g.pitch; }
  bool top_is_border() const { return g.row0 == 0; }
  bool bottom_is_border() const { return g.row0 + g.rows == g.H; }
  bool observing() const { return watch_var >= 0 || act_maps || frames || !paces.empty(); }
  // what the step kernels see: ONE replica (the whole shard when nrep == 1), launched nrep times along blockIdx.z
  Geom step_geom() const { return nrep == 1 ? g : Geom{g.H / nrep, g.W, 0, g.H / nrep, g.pitch}; }
};

static void drop_graphs(fib_ctx* c) {
  for (auto& gk : c->graphs) cudaGraphExecDestroy(gk.exec);
  c->graphs.clear();
}

static int check_persist_error(fib_ctx* c);

struct DevGuard {
  int prev = -1;
  explicit DevGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
  ~DevGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ------------------------------------------------------------------------------------------
// small kernels
// ------------------------------------------------------------------------------------------
// ionic.py:144-163: X := max(X, s) with s = value inside the rectangle and floor_v elsewhere.
// fmaxf: tf.maximum on the reference's GPU target returns the non-NaN operand (see clip_tf).
// Over local rows [lr0, lr0 + nrows); the rectangle's rows count within a replica of rh rows (rh = H: the grid).
__global__ void stim_kernel(float* __restrict__ x, Geom g, int halo, int rh, int lr0, int nrows, int r0, int r1,
                            int c0, int c1, float value, float floor_v) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= g.W) return;
  for (int lr = lr0 + (int)blockIdx.y; lr < lr0 + nrows; lr += gridDim.y) {
    const int gr = (g.row0 + lr) % rh;
    const float m = (gr >= r0 && gr < r1 && c >= c0 && c < c1) ? value : floor_v;
    float* p = x + (size_t)(lr + halo) * g.pitch + c;
    const float v = *p;
    *p = fmaxf(v, m);
  }
}

// fib_set_phase: flag the 32-column blocks of each row whose phase term can be non-zero, i.e.
// where phi is not constant over rows r-1..r+1 (REFLECT) x columns c0-1..c0+32 (clipped: the
// reflected columns -1 -> 1 and W -> W-2 lie inside that range).  g: one replica (blockIdx.z), as the step
// kernels see it, so the REFLECT stays inside the replica.
__global__ void phase_mask_kernel(const float* __restrict__ phase, Geom g, unsigned char* __restrict__ mask,
                                  int mpitch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= mpitch) return;
  phase += (size_t)blockIdx.z * g.rows * g.pitch;
  mask += (size_t)blockIdx.z * g.rows * mpitch;
  const int c0 = max(b * 32 - 1, 0), c1 = min(b * 32 + 32, g.W - 1);
  for (int lr = blockIdx.y; lr < g.rows; lr += gridDim.y) {
    const int gr = g.row0 + lr;
    const float first = phase[(size_t)(lr + 1) * g.pitch + c0];
    bool same = true;
    for (int dr = -1; dr <= 1; ++dr) {
      const int rr = reflecti(gr + dr, g.H) - g.row0 + 1;
      for (int c = c0; c <= c1; ++c) same &= (phase[(size_t)rr * g.pitch + c] == first);
    }
    mask[(size_t)lr * mpitch + b] = same ? 0 : 1;
  }
}

// the same flags for the two-steps-per-launch layout: phi with kFuseHalo halo rows, local rows
// -1 .. rows (the first step is recomputed on the neighbours' edge rows); rows outside the grid: 0
__global__ void phase_mask2_kernel(const float* __restrict__ phase, Geom g, unsigned char* __restrict__ mask,
                                   int mpitch) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= mpitch) return;
  phase += (size_t)blockIdx.z * g.rows * g.pitch;
  mask += (size_t)blockIdx.z * g.rows * mpitch;
  const int c0 = max(b * 32 - 1, 0), c1 = min(b * 32 + 32, g.W - 1);
  for (int lr = (int)blockIdx.y - 1; lr <= g.rows; lr += gridDim.y) {
    // the rows just outside a replica are its neighbours' first / last rows: theirs to flag
    if ((lr < 0 && blockIdx.z > 0) || (lr == g.rows && blockIdx.z + 1 < gridDim.z)) continue;
    const int gr = g.row0 + lr;
    bool same = true;
    if (gr >= 0 && gr < g.H) {
      const float first = phase[(size_t)(lr + kFuseHalo) * g.pitch + c0];
      for (int dr = -1; dr <= 1; ++dr) {
        const int rr = reflecti(gr + dr, g.H) - g.row0 + kFuseHalo;
        for (int c = c0; c <= c1; ++c) same &= (phase[(size_t)rr * g.pitch + c] == first);
      }
    }
    mask[(size_t)(lr + 1) * mpitch + b] = same ? 0 : 1;
  }
}

// Sums over row blocks of `rows` rows: block row blockIdx.y = z covers local rows [z * rows, (z + 1) * rows) and
// adds into out[2z], out[2z + 1] (one block row over the shard: the whole-context sum; nrep: one per replica).
__global__ void wsum_kernel(const float* __restrict__ x, const float* __restrict__ w, Geom g,
                            int xhalo, int rows, double* out) {
  double sx = 0.0, sw = 0.0;
  const int r0 = (int)blockIdx.y * rows;
  out += 2 * blockIdx.y;
  for (int lr = r0 + (int)blockIdx.x; lr < r0 + rows; lr += gridDim.x)
    for (int c = threadIdx.x; c < g.W; c += blockDim.x) {
      const double wv = w ? (double)w[(size_t)(lr + 1) * g.pitch + c] : 1.0;
      sx += wv * (double)x[(size_t)(lr + xhalo) * g.pitch + c];
      sw += wv;
    }
  for (int o = 16; o > 0; o >>= 1) {
    sx += __shfl_down_sync(0xffffffffu, sx, o);
    sw += __shfl_down_sync(0xffffffffu, sw, o);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, sx); atomicAdd(out + 1, sw); }
}

__global__ void nonfinite_kernel(const float* __restrict__ x, Geom g, int xhalo, unsigned long long* out) {
  unsigned long long n = 0;
  for (int lr = blockIdx.x; lr < g.rows; lr += gridDim.x)
    for (int c = threadIdx.x; c < g.W; c += blockDim.x)
      n += !isfinite(x[(size_t)(lr + xhalo) * g.pitch + c]);
  for (int o = 16; o > 0; o >>= 1) n += __shfl_down_sync(0xffffffffu, n, o);
  if ((threadIdx.x & 31) == 0 && n) atomicAdd(out, n);
}

// fib_probe_watch / fib_replica_probe_watch: append one record, the `ncells` watched cells `rep_step` floats apart
// (one per replica), to the ring of `cap` records (a node of the iteration graph).  ONE block: every thread has read
// *count before thread 0 advances it.
__global__ void probe_record_kernel(const float* __restrict__ src, size_t rep_step, int ncells,
                                    float* __restrict__ ring, unsigned long long cap,
                                    unsigned long long* __restrict__ count) {
  const unsigned long long n = *count;
  float* rec = ring + (n % cap) * ncells;
  for (int b = threadIdx.x; b < ncells; b += blockDim.x) rec[b] = src[(size_t)b * rep_step];
  __syncthreads();
  if (threadIdx.x == 0) *count = n + 1;
}

// a host-side write (stimulus, assign) after the iteration: the reference evaluates its probe AFTER
// the driver's loop body (ionic.py:202-216), so the last recorded value follows the write
__global__ void probe_update_kernel(const float* __restrict__ src, size_t rep_step, int ncells,
                                    float* __restrict__ ring, unsigned long long cap,
                                    const unsigned long long* __restrict__ count) {
  const unsigned long long n = *count;
  if (!n) return;
  float* rec = ring + ((n - 1) % cap) * ncells;
  for (int b = threadIdx.x; b < ncells; b += blockDim.x) rec[b] = src[(size_t)b * rep_step];
}

// fib_frames_watch: one frame, a strided gather of a plane's owned rows.  `src` = the first owned row whose
// global index is a multiple of the stride, `src_step` = floats between two frame rows (stride * pitch).
__global__ void frame_record_kernel(const float* __restrict__ src, size_t src_step, int stride, int rows, int cols,
                                    float* __restrict__ dst) {
  const int fc = blockIdx.x * blockDim.x + threadIdx.x;
  if (fc >= cols) return;
  for (int fr = blockIdx.y; fr < rows; fr += gridDim.y)
    dst[(size_t)fr * cols + fc] = src[(size_t)fr * src_step + (size_t)fc * stride];
}

// court_ultra.py:504-509: cells with weight > w_min, and among them those whose normalised value
// (x - sub) / div (the image() of br.py:337-343 / court.py:574-580, same fp32 operations) < cutoff
// (row blocks as in wsum_kernel)
__global__ void count_below_kernel(const float* __restrict__ x, const float* __restrict__ w, Geom g,
                                   int xhalo, int rows, float sub, float div, float cutoff, float w_min,
                                   unsigned long long* out) {
  unsigned long long below = 0, total = 0;
  const int r0 = (int)blockIdx.y * rows;
  out += 2 * blockIdx.y;
  for (int lr = r0 + (int)blockIdx.x; lr < r0 + rows; lr += gridDim.x)
    for (int c = threadIdx.x; c < g.W; c += blockDim.x) {
      const float wv = w ? w[(size_t)(lr + 1) * g.pitch + c] : 1.0f;
      if (wv > w_min) {
        ++total;
        const float img = __fdiv_rn(__fsub_rn(x[(size_t)(lr + xhalo) * g.pitch + c], sub), div);
        below += img < cutoff;
      }
    }
  for (int o = 16; o > 0; o >>= 1) {
    below += __shfl_down_sync(0xffffffffu, below, o);
    total += __shfl_down_sync(0xffffffffu, total, o);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, below); atomicAdd(out + 1, total); }
}

// ---- op-level entry points (fib_op_*): IonicModel's helpers on dense planes ----------------------
__global__ void op_enforce_kernel(const float* __restrict__ x, int h, int w, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= w) return;
  out[(size_t)r * w + c] = x[(size_t)clampi(r, 1, h - 2) * w + clampi(c, 1, w - 2)];   // ionic.py:107-113
}
// mode 0: Xp = REFLECT pad of x (ionic.py:49-50); mode 1: the step kernels' collapsed map on a raw
// plane, Xp[r][c] = x[clamp(r,1,h-2)][clamp(c,1,w-2)] (fib_stencil.cuh); mode 2: phase term only
__global__ void op_laplace_kernel(const float* __restrict__ x, const float* __restrict__ ph, int h, int w,
                                  int mode, float* __restrict__ out) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
  if (c >= w) return;
  auto X = [&](int rr, int cc) {
    const int r2 = mode == 1 ? clampi(rr, 1, h - 2) : reflecti(rr, h);
    const int c2 = mode == 1 ? clampi(cc, 1, w - 2) : reflecti(cc, w);
    return x[(size_t)r2 * w + c2];
  };
  auto P = [&](int rr, int cc) { return ph[(size_t)reflecti(rr, h) * w + reflecti(cc, w)]; };
  float lap = 0.f;
  if (mode != 2)
    lap = lap9(X(r - 1, c), X(r + 1, c), X(r, c - 1), X(r, c + 1), X(r - 1, c - 1), X(r + 1, c - 1),
               X(r - 1, c + 1), X(r + 1, c + 1), X(r, c));
  if (ph) {
    const float t = phase_term(X(r - 1, c), X(r + 1, c), X(r, c - 1), X(r, c + 1), P(r - 1, c), P(r + 1, c),
                               P(r, c - 1), P(r, c + 1), P(r, c));
    lap = mode == 2 ? t : __fadd_rn(lap, t);
  }
  out[(size_t)r * w + c] = lap;
}
__global__ void op_rush_larsen_kernel(const float* __restrict__ g, const float* __restrict__ gi,
                                      const float* __restrict__ tau, size_t n, float neg_dt, int strict,
                                      float* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = strict ? rush_larsen_strict(g[i], gi[i], tau[i], neg_dt) : rush_larsen(g[i], gi[i], tau[i], neg_dt);
}

__global__ void court_inter_kernel(const float* __restrict__ v, int n, float* __restrict__ out,
                                   int ncols) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float q[kInterCols];
  court_inter_dev<true>(v[i], q);
  for (int k = 0; k < ncols; ++k) out[(size_t)i * ncols + k] = q[k];
}

__global__ void lut_transpose_kernel(const float* __restrict__ lut, float* __restrict__ lut_t) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kLutRows) return;
  for (int k = 0; k < kLutCols; ++k) lut_t[k * kLutTStride + i] = lut[i * kLutCols + k];
}

__global__ void court_lut_kernel(float* __restrict__ lut) {   // courtemanche.h:473-479
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= kLutRows) return;
  float q[kInterCols];
  court_inter_dev<false>(static_cast<float>(i - 100), q);
  for (int k = 0; k < kLutCols; ++k) lut[i * kLutCols + k] = q[k];
}

// ------------------------------------------------------------------------------------------
// library
// ------------------------------------------------------------------------------------------
extern "C" int fib_version(void) { return FIB_ABI_VERSION; }
extern "C" const char* fib_last_error(void) { return g_err.c_str(); }
extern "C" int fib_last_kernel(char* buf, size_t n) {
  if (!buf || n == 0) return fail(FIB_E_ARG, "buf is NULL");
  snprintf(buf, n, "%s", last_kernel_name());
  return 0;
}
extern "C" int fib_device_count(int* count) {
  if (!count) return fail(FIB_E_ARG, "count is NULL");
  CU(cudaGetDeviceCount(count));
  return 0;
}

extern "C" int fib_host_alloc(size_t bytes, void** out) {
  if (!out) return fail(FIB_E_ARG, "out is NULL");
  CU(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
  return 0;
}
extern "C" int fib_host_free(void* p) {
  CU(cudaFreeHost(p));
  return 0;
}

static int create_resources(fib_ctx* c);
// fp32(diff_b * dt) of every replica, folded in double as fenton_params / br_params / launch_court fold cfg.diff
static int upload_replica_diff(fib_ctx* c, const double* diff) {
  std::vector<float> ddt(c->nrep);
  for (int b = 0; b < c->nrep; ++b) ddt[b] = (float)(diff[b] * c->cfg.dt);
  CU(cudaMemcpyAsync(c->zddt, ddt.data(), c->nrep * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" int fib_create(const fib_config* cfg, fib_ctx** out) {
  if (!cfg || !out) return fail(FIB_E_ARG, "cfg/out is NULL");
  if (cfg->struct_size != sizeof(fib_config))
    return fail(FIB_E_ARG, "fib_config.struct_size %u != %zu (ABI mismatch)", cfg->struct_size,
                sizeof(fib_config));
  if (cfg->model < FIB_FENTON4V || cfg->model > FIB_COURT_ULTRA)
    return fail(FIB_E_ARG, "unknown model id %d", cfg->model);
  if (cfg->height < 3 || cfg->width < 3)
    return fail(FIB_E_ARG, "grid %dx%d too small: the two-stage boundary needs >= 3x3", cfg->height,
                cfg->width);
  if (!(cfg->dt > 0.0)) return fail(FIB_E_ARG, "dt must be > 0");
  if (cfg->steps_per_launch < 0 || cfg->steps_per_launch > 2)
    return fail(FIB_E_ARG, "steps_per_launch=%d: 0/1 (one step per launch) or 2", cfg->steps_per_launch);
  if (cfg->steps_per_launch == 2 && (cfg->model != FIB_FENTON4V || cfg->width % 4 != 0))
    return fail(FIB_E_ARG, "steps_per_launch=2 needs the Fenton 4v model and a width that is a multiple "
                "of 4 (got model %d, width %d)", cfg->model, cfg->width);
  const int nrep = cfg->replicas < 1 ? 1 : cfg->replicas;
  if (cfg->replicas < 0 || nrep > 65535)
    return fail(FIB_E_ARG, "replicas=%d: 0 or 1 (one grid) up to 65535", cfg->replicas);
  if (nrep > 1 && cfg->rows != 0)
    return fail(FIB_E_ARG, "replicas=%d: a batched context cannot be a row shard (rows must be 0)", nrep);
  int rows = cfg->rows == 0 ? cfg->height : cfg->rows;
  int row0 = cfg->rows == 0 ? 0 : cfg->row0;
  if (row0 < 0 || rows < 1 || row0 + rows > cfg->height)
    return fail(FIB_E_ARG, "shard rows [%d,%d) outside the grid of height %d", row0, row0 + rows,
                cfg->height);
  if (cfg->steps_per_launch == 2 && rows != cfg->height && rows < kFuseHalo)
    return fail(FIB_E_ARG, "steps_per_launch=2: a shard must own at least %d rows (got %d)", kFuseHalo, rows);
  if ((long long)((long long)rows * nrep + 2 * kFuseHalo) * ((cfg->width + 31) / 32 * 32) >= (1LL << 31))
    return fail(FIB_E_ARG, "shard of %lld rows x %d columns exceeds 2^31 cells per plane: the kernels "
                "index planes with 32-bit element offsets; shard the grid over more GPUs, or use fewer replicas",
                (long long)rows * nrep, cfg->width);
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev)
    return fail(FIB_E_CUDA, "device %d not available (%d CUDA devices)", cfg->device, ndev);
  DevGuard dg(cfg->device);

  fib_ctx* c = new fib_ctx();
  c->cfg = *cfg;
  c->nrep = nrep;
  c->g.H = cfg->height * nrep;
  c->g.W = cfg->width;
  c->g.row0 = row0;
  c->g.rows = rows * nrep;
  c->g.pitch = (cfg->width + 31) / 32 * 32;
  // a failure half way (e.g. out of memory at 32768^2 on a busy GPU) must release what exists
  const int rc = create_resources(c);
  if (rc) {
    const std::string why = g_err;
    fib_destroy(c);
    g_err = why;
    return rc;
  }
  *out = c;
  return 0;
}

static int create_resources(fib_ctx* c) {
  const fib_config* cfg = &c->cfg;
  switch (cfg->model) {
    case FIB_FENTON4V: c->nvars = 4; c->dt_per_step = 10; c->names = kFentonVars; break;
    case FIB_BR: c->nvars = 8; c->dt_per_step = 5; c->names = kBrVars; break;
    case FIB_COURT: c->nvars = 21; c->dt_per_step = 1; c->names = kCourtVars; break;
    default:
      c->nvars = (cfg->flags & FIB_F_ULTRA_SLOW) ? 22 : 21;
      c->dt_per_step = 1;
      c->names = kCourtVars;
  }
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, cfg->device));
  c->sms = prop.multiProcessorCount;
  CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->comm_stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->up_stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&c->ck_stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&c->ev_up_begin, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_ck, cudaEventDisableTiming));
  if (const char* e = getenv("FIB_PIPELINE_MIN_CELLS")) c->pipeline_min_cells = atoll(e);
  if (const char* e = getenv("FIB_PIPELINE_BLOCK_ROWS")) c->pipeline_block_rows = max(atoi(e), 1);
  if (const char* e = getenv("FIB_PIPELINE_NCCL")) c->pipeline_nccl = atoi(e) != 0;
  CU(cudaEventCreateWithFlags(&c->ev_snap_ready, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_snap_done, cudaEventDisableTiming));
  CU(cudaEventCreate(&c->ev_start));
  CU(cudaEventCreate(&c->ev_stop));
  CU(cudaEventCreateWithFlags(&c->ev_bnd, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_comm, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&c->ev_group, cudaEventDisableTiming));
  c->fuse = cfg->steps_per_launch == 2 ? 2 : 1;
  if (c->fuse == 2) {
    for (int b = 0; b < 2; ++b)
      for (int v = 0; v < 4; ++v) {
        CU(cudaMalloc(&c->fx[b][v], c->fused_floats() * sizeof(float)));
        CU(cudaMemsetAsync(c->fx[b][v], 0, c->fused_floats() * sizeof(float), c->stream));
      }
  } else {
    for (int b = 0; b < 2; ++b) {
      CU(cudaMalloc(&c->x[b], c->halo_floats() * sizeof(float)));
      CU(cudaMemsetAsync(c->x[b], 0, c->halo_floats() * sizeof(float), c->stream));
    }
    for (int k = 0; k + 1 < c->nvars; ++k) {
      CU(cudaMalloc(&c->s[k], c->plane_floats() * sizeof(float)));
      CU(cudaMemsetAsync(c->s[k], 0, c->plane_floats() * sizeof(float), c->stream));
    }
  }
  CU(cudaMalloc(&c->red, 2 * c->nrep * sizeof(double)));
  if (c->nrep > 1) {
    CU(cudaMalloc(&c->zddt, c->nrep * sizeof(float)));
    const std::vector<double> diff(c->nrep, cfg->diff);
    const int r = upload_replica_diff(c, diff.data());
    if (r) return r;
  }
  if (cfg->model >= FIB_COURT) {
    CU(cudaMalloc(&c->lut, sizeof(float) * kLutRows * kLutCols));
    CU(cudaMalloc(&c->lut_t, sizeof(float) * kLutCols * kLutTStride));
    CU(cudaMemsetAsync(c->lut_t, 0, sizeof(float) * kLutCols * kLutTStride, c->stream));
  }
  memset(c->cheb, 0, sizeof c->cheb);
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int fib_destroy(fib_ctx* c) {
  if (!c) return 0;
  DevGuard dg(c->cfg.device);
  // every handle may still be null: fib_create destroys a partially built context on failure
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->comm_stream) cudaStreamSynchronize(c->comm_stream);
  if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
  if (c->ck) {
    cudaFreeAsync(c->ck, c->stream);
    cudaStreamSynchronize(c->stream);
  }
  if (c->ck_stream) {
    cudaStreamSynchronize(c->ck_stream);
    cudaStreamDestroy(c->ck_stream);
  }
  if (c->ev_ck) cudaEventDestroy(c->ev_ck);
  if (c->up_stream) {
    cudaStreamSynchronize(c->up_stream);
    cudaStreamDestroy(c->up_stream);
  }
  if (c->ev_up_begin) cudaEventDestroy(c->ev_up_begin);
  for (auto& a : c->arrivals) cudaEventDestroy(a.ev);
  for (auto e : c->ev_pool) cudaEventDestroy(e);
  cudaFree(c->snap);
  if (c->ev_snap_ready) cudaEventDestroy(c->ev_snap_ready);
  if (c->ev_snap_done) cudaEventDestroy(c->ev_snap_done);
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  for (auto& gk : c->graphs) cudaGraphExecDestroy(gk.exec);
  for (int b = 0; b < 2; ++b) cudaFree(c->x[b]);
  for (int b = 0; b < 2; ++b)
    for (int v = 0; v < 4; ++v) cudaFree(c->fx[b][v]);
  for (int k = 0; k < S_COUNT; ++k) cudaFree(c->s[k]);
  cudaFree(c->phase);
  cudaFree(c->pmask);
  cudaFree(c->phase2);
  cudaFree(c->pmask2);
  cudaFree(c->lut);
  cudaFree(c->lut_t);
  cudaFree(c->red);
  cudaFree(c->zddt);
  cudaFreeHost(c->ring);
  c->probe_ledger.destroy();
  cudaFree(c->ring_count);
  cudaFree(c->act_prev);
  cudaFree(c->act_maps);
  cudaFree(c->act_iter);
  cudaFree(c->frames);
  c->frame_ledger.destroy();
  cudaFree(c->pmail);
  if (c->perr) cudaFreeHost(c->perr);
  for (int k = 0; k < 4; ++k) cudaFree(c->weights[k]);
  for (cudaEvent_t e : {c->ev_start, c->ev_stop, c->ev_bnd, c->ev_comm, c->ev_group})
    if (e) cudaEventDestroy(e);
  if (c->stream) cudaStreamDestroy(c->stream);
  if (c->comm_stream) cudaStreamDestroy(c->comm_stream);
  cudaGetLastError();      // a failed creation may have left a sticky-free error behind
  delete c;
  return 0;
}

extern "C" int fib_num_vars(const fib_ctx* c) { return c ? c->nvars : fail(FIB_E_ARG, "ctx is NULL"); }
extern "C" const char* fib_var_name(const fib_ctx* c, int var) {
  return (c && var >= 0 && var < c->nvars) ? c->names[var] : nullptr;
}
extern "C" int fib_var_index(const fib_ctx* c, const char* name) {
  if (!c || !name) return fail(FIB_E_ARG, "ctx/name is NULL");
  for (int i = 0; i < c->nvars; ++i)
    if (!strcmp(c->names[i], name)) return i;
  return fail(FIB_E_ARG, "unknown state variable '%s'", name);
}
extern "C" int fib_dt_per_step(const fib_ctx* c) { return c ? c->dt_per_step : fail(FIB_E_ARG, "ctx is NULL"); }

// A plane of the CURRENT state: start of its allocation and the number of halo rows above the
// first owned row (1 for the diffusing variable, 0 for the in-place planes, kFuseHalo for every
// plane of the two-steps-per-launch layout).
struct PlaneRef { float* base; int halo; };
static PlaneRef plane_of(fib_ctx* c, int var) {
  if (c->fuse == 2) return {c->fx[c->cur][var], kFuseHalo};
  return var == 0 ? PlaneRef{c->x[c->cur], 1} : PlaneRef{c->s[var - 1], 0};
}
static float* owned_rows(fib_ctx* c, int var) {
  const PlaneRef p = plane_of(c, var);
  return p.base + (size_t)p.halo * c->g.pitch;
}
// the watched cell of the probe (of replica 0 for a replica watch), and the floats between two replicas' cells
static const float* watch_src(fib_ctx* c) {
  return owned_rows(c, c->watch_var) + (size_t)(c->watch_row - c->g.row0) * c->g.pitch + c->watch_col;
}
static size_t replica_step(const fib_ctx* c) { return (size_t)(c->g.H / c->nrep) * c->g.pitch; }
static int probe_threads(const fib_ctx* c) { return min(c->watch_n, 1024); }

// a host write into `var` invalidates the neighbours' copies of the rows they hold as halo, and
// the last record the cycle-length probe made if it watches this plane (enqueue-only)
static void mark_written(fib_ctx* c, int var) {
  if (var == 0 || c->fuse == 2) c->halo_dirty = true;
  if (var == c->watch_var) {
    probe_update_kernel<<<1, probe_threads(c), 0, c->stream>>>(watch_src(c), replica_step(c), c->watch_n, c->ring,
                                                               c->ring_cap, c->ring_count);
    c->launches++;
    c->probe_ledger.clear();                    // a recorded value changes after its launch's event
  }
}
// a halo exchange still running on the side stream must land before anything else touches the
// diffusing variable's buffers on the main stream
static cudaError_t wait_comm(fib_ctx* c) {
  if (!c->comm_pending) return cudaSuccess;
  c->comm_pending = false;
  return cudaStreamWaitEvent(c->stream, c->ev_comm, 0);
}

// the stimulus of fib_stimulate_replica on the CURRENT plane `var` (enqueue-only; the caller marks the plane
// written): rows local to a replica, in replica `replica` only or (-1) in every replica
static int launch_stim(fib_ctx* c, int var, int replica, int r0, int r1, int c0, int c1, float value,
                       float floor_v) {
  CU(wait_comm(c));
  const int rh = c->g.H / c->nrep;
  const int lr0 = replica < 0 ? 0 : replica * rh, nrows = replica < 0 ? c->g.rows : rh;
  dim3 block(128), grid((c->g.W + 127) / 128, min(nrows, 65535));
  const PlaneRef pl = plane_of(c, var);
  stim_kernel<<<grid, block, 0, c->stream>>>(pl.base, c->g, pl.halo, rh, lr0, nrows, r0, r1, c0, c1, value,
                                             floor_v);
  CU(cudaGetLastError());
  c->launches++;
  return 0;
}

// The persistent path DEFERS iterations: fib_step only counts them, and they are launched -- up to
// kPersistMaxIters per launch -- by the next call that observes or modifies anything (every entry
// point below starts with FLUSH), or as soon as a full launch's worth has accumulated.  A driver
// loop of fib_step(ctx, op, 1) calls then costs one launch per 64 iterations instead of one each.
static int flush_pending(fib_ctx* c);
#define FLUSH(c)                                                      \
  do {                                                                \
    if ((c)->pending || (c)->up_session) {                            \
      const int fr_ = flush_pending(c);                               \
      if (fr_) return fr_;                                            \
    }                                                                 \
  } while (0)

extern "C" int fib_set_state(fib_ctx* c, int var, const float* host, size_t n) {
  if (!c || !host) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (n != (size_t)c->g.rows * c->g.W)
    return fail(FIB_E_ARG, "fib_set_state: n=%zu, expected rows*width=%zu", n, (size_t)c->g.rows * c->g.W);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(wait_comm(c));
  CU(cudaMemcpy2DAsync(owned_rows(c, var), c->g.pitch * sizeof(float), host, c->g.W * sizeof(float),
                       c->g.W * sizeof(float), c->g.rows, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  mark_written(c, var);
  return 0;
}

extern "C" int fib_get_state(fib_ctx* c, int var, float* host, size_t n) {
  if (!c || !host) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (n != (size_t)c->g.rows * c->g.W)
    return fail(FIB_E_ARG, "fib_get_state: n=%zu, expected rows*width=%zu", n, (size_t)c->g.rows * c->g.W);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaMemcpy2DAsync(host, c->g.W * sizeof(float), owned_rows(c, var), c->g.pitch * sizeof(float),
                       c->g.W * sizeof(float), c->g.rows, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return check_persist_error(c);
}

extern "C" int fib_get_rect(fib_ctx* c, int var, int r0, int r1, int c0, int c1, float* host) {
  if (!c || !host) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (r0 < c->g.row0 || r1 > c->g.row0 + c->g.rows || r0 >= r1 || c0 < 0 || c1 > c->g.W || c0 >= c1)
    return fail(FIB_E_ARG, "rectangle [%d,%d)x[%d,%d) not inside this shard", r0, r1, c0, c1);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  const float* src = owned_rows(c, var) + (size_t)(r0 - c->g.row0) * c->g.pitch + c0;
  CU(cudaMemcpy2DAsync(host, (size_t)(c1 - c0) * sizeof(float), src, c->g.pitch * sizeof(float),
                       (size_t)(c1 - c0) * sizeof(float), r1 - r0, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int fib_snapshot_begin(fib_ctx* c, int var, float* host_pinned, size_t n) {
  if (!c || !host_pinned) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (n != (size_t)c->g.rows * c->g.W)
    return fail(FIB_E_ARG, "fib_snapshot_begin: n=%zu, expected rows*width=%zu", n, (size_t)c->g.rows * c->g.W);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, host_pinned) != cudaSuccess || pa.type != cudaMemoryTypeHost) {
      cudaGetLastError();
      return fail(FIB_E_ARG, "fib_snapshot_begin needs page-locked host memory (fib_host_alloc)");
    }
  }
  if (!c->snap) CU(cudaMalloc(&c->snap, c->plane_floats() * sizeof(float)));
  if (c->snap_pending) CU(cudaStreamWaitEvent(c->stream, c->ev_snap_done, 0));   // staging still in use
  CU(cudaMemcpyAsync(c->snap, owned_rows(c, var), c->plane_floats() * sizeof(float),
                     cudaMemcpyDeviceToDevice, c->stream));
  CU(cudaEventRecord(c->ev_snap_ready, c->stream));
  CU(cudaStreamWaitEvent(c->copy_stream, c->ev_snap_ready, 0));
  CU(cudaMemcpy2DAsync(host_pinned, c->g.W * sizeof(float), c->snap, c->g.pitch * sizeof(float),
                       c->g.W * sizeof(float), c->g.rows, cudaMemcpyDeviceToHost, c->copy_stream));
  CU(cudaEventRecord(c->ev_snap_done, c->copy_stream));
  c->snap_pending = true;
  return 0;
}

extern "C" int fib_snapshot_wait(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (!c->snap_pending) return 0;
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaEventSynchronize(c->ev_snap_done));
  c->snap_pending = false;
  return 0;
}

// the probe ring's storage, at least `floats` (allocations may synchronise with copies in flight: never between
// the blocks of a pipelined upload and the steps behind it; the ring only grows, when no watch is armed)
static int ensure_ring(fib_ctx* c, size_t floats) {
  if (c->ring_floats < floats) {
    cudaFreeHost(c->ring);
    c->ring = nullptr;
    c->ring_floats = 0;
    CU(cudaHostAlloc(&c->ring, floats * sizeof(float), cudaHostAllocMapped | cudaHostAllocPortable));
    c->ring_floats = floats;
  }
  if (!c->ring_count) CU(cudaMalloc(&c->ring_count, sizeof(unsigned long long)));
  return c->probe_ledger.create();
}

static int launch_substep(fib_ctx* c, int op, int sub, int lr0, int nrows);
static int substeps_of(const fib_ctx* c, int op);
// Everything an ODE iteration and its probe record can launch is loaded NOW (lazy loading would do it at
// the first launch and wait for the copies in flight).  Called when a pipelined upload begins.
static int preload_kernels(fib_ctx* c) {
  int r = ensure_ring(c, FIB_PROBE_RING);
  if (r) return r;
  cudaFuncAttributes fa;
  CU(cudaFuncGetAttributes(&fa, probe_record_kernel));
  CU(cudaFuncGetAttributes(&fa, probe_update_kernel));
  const uint64_t l0 = c->launches;
  preload_only() = true;
  const int ns = substeps_of(c, FIB_OP_ODE);
  for (int s = 0; s < ns && !r; s += c->fuse)
    for (int nrows : {c->g.rows, min(c->g.rows, c->pipeline_block_rows)})
      if (!r) r = launch_substep(c, FIB_OP_ODE, s, 0, nrows);
  preload_only() = false;
  c->launches = l0;
  cudaGetLastError();
  return 0;       // best effort: a model that cannot step yet (table not set) reports that from fib_step
}

static int set_rect_impl(fib_ctx* c, int var, int r0, int r1, int c0, int c1, const float* host, bool sync) {
  if (!c || !host) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (r0 < c->g.row0 || r1 > c->g.row0 + c->g.rows || r0 >= r1 || c0 < 0 || c1 > c->g.W || c0 >= c1)
    return fail(FIB_E_ARG, "rectangle [%d,%d)x[%d,%d) not inside this shard", r0, r1, c0, c1);
  DevGuard dg(c->cfg.device);
  if (!sync) {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, host) != cudaSuccess || pa.type != cudaMemoryTypeHost) {
      cudaGetLastError();
      return fail(FIB_E_ARG, "fib_set_rect_async needs page-locked host memory (fib_host_alloc)");
    }
    // A full-width block that continues this plane's upload frontier (or starts one at the first row) of a
    // large unsharded grid goes to the upload stream: iterations stepped before anything looks at the
    // result then run block by block BEHIND the copies instead of after them (finish_upload_session).
    // On an NCCL shard the block order may also run bottom to top (odd ranks do, so that both shards of a seam
    // either begin or end there: fib_step_behind_upload).
    // (a batched context steps whole replicas only: not the row blocks of the skewed schedule)
    const bool eligible = (c->comm ? c->pipeline_nccl : c->g.rows == c->g.H) && c->nrep == 1 && c0 == 0 && c1 == c->g.W &&
                          !c->observing() && (long long)c->g.rows * c->g.W >= c->pipeline_min_cells;
    const int row_end = c->g.row0 + c->g.rows;
    const int dir = c->up_session ? c->up_dir : (r0 == c->g.row0 ? +1 : (r1 == row_end && c->comm ? -1 : 0));
    const int dlo = dir > 0 ? r0 - c->g.row0 : row_end - r1, dhi = dir > 0 ? r1 - c->g.row0 : row_end - r0;
    if (eligible && dir != 0 && !c->pending && dlo == (c->up_session ? c->up_front[var] : 0)) {
      if (!c->up_session) {
        const int pr = preload_kernels(c);
        if (pr) return pr;                                       // (allocation failures only)
        CU(wait_comm(c));
        CU(cudaEventRecord(c->ev_up_begin, c->stream));          // after everything stepped so far
        CU(cudaStreamWaitEvent(c->up_stream, c->ev_up_begin, 0));
        if (c->snap_pending) CU(cudaStreamWaitEvent(c->up_stream, c->ev_snap_done, 0));
        c->up_front.assign(c->nvars, 0);
        c->up_dir = dir;
        c->up_session = true;
      }
      float* dst = owned_rows(c, var) + (size_t)(r0 - c->g.row0) * c->g.pitch;
      CU(cudaMemcpy2DAsync(dst, c->g.pitch * sizeof(float), host, (size_t)c->g.W * sizeof(float),
                           (size_t)c->g.W * sizeof(float), r1 - r0, cudaMemcpyHostToDevice, c->up_stream));
      c->up_front[var] = dhi;
      int done = dhi;
      for (int f : c->up_front) done = min(done, f);
      const int had = c->arrivals.empty() ? 0 : c->arrivals.back().d_end;
      if (done - had >= c->pipeline_block_rows || (done > had && done == c->g.rows)) {
        cudaEvent_t ev = nullptr;
        if (!c->ev_pool.empty()) {
          ev = c->ev_pool.back();
          c->ev_pool.pop_back();
        } else {
          CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        }
        CU(cudaEventRecord(ev, c->up_stream));
        c->arrivals.push_back({done, ev});
      }
      if (var == 0 || c->fuse == 2) c->halo_dirty = true;
      return 0;
    }
  }
  FLUSH(c);
  CU(wait_comm(c));
  float* dst = owned_rows(c, var) + (size_t)(r0 - c->g.row0) * c->g.pitch + c0;
  CU(cudaMemcpy2DAsync(dst, c->g.pitch * sizeof(float), host, (size_t)(c1 - c0) * sizeof(float),
                       (size_t)(c1 - c0) * sizeof(float), r1 - r0, cudaMemcpyHostToDevice, c->stream));
  if (sync) CU(cudaStreamSynchronize(c->stream));
  mark_written(c, var);
  return 0;
}
extern "C" int fib_set_rect(fib_ctx* c, int var, int r0, int r1, int c0, int c1, const float* host) {
  return set_rect_impl(c, var, r0, r1, c0, c1, host, true);
}
extern "C" int fib_set_rect_async(fib_ctx* c, int var, int r0, int r1, int c0, int c1, const float* host) {
  return set_rect_impl(c, var, r0, r1, c0, c1, host, false);
}

extern "C" int fib_set_phase(fib_ctx* c, const float* rows_host, int first_row, int nrows) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaStreamSynchronize(c->stream));
  drop_graphs(c);                       // graphs bake the phase pointer in
  if (!rows_host) {
    CU(cudaFree(c->phase));
    CU(cudaFree(c->pmask));
    CU(cudaFree(c->phase2));
    CU(cudaFree(c->pmask2));
    c->phase = nullptr;
    c->pmask = nullptr;
    c->phase2 = nullptr;
    c->pmask2 = nullptr;
    return 0;
  }
  // one halo row of phi for one step per launch, kFuseHalo for two
  const int hr = c->fuse == 2 ? kFuseHalo : 1;
  const int need0 = max(c->g.row0 - hr, 0), need1 = min(c->g.row0 + c->g.rows + hr, c->g.H);
  if (first_row > need0 || first_row + nrows < need1)
    return fail(FIB_E_ARG, "phase rows [%d,%d) do not cover [%d,%d)", first_row, first_row + nrows,
                need0, need1);
  if (!c->phase) {
    CU(cudaMalloc(&c->phase, c->halo_floats() * sizeof(float)));
    CU(cudaMemsetAsync(c->phase, 0, c->halo_floats() * sizeof(float), c->stream));
  }
  // device row (n0 - row0 + 1) <- host row (n0 - first_row); this copy (one halo row) also serves
  // the reductions (fib_weighted_sum)
  {
    const int n0 = max(c->g.row0 - 1, 0), n1 = min(c->g.row0 + c->g.rows + 1, c->g.H);
    CU(cudaMemcpy2DAsync(c->phase + (size_t)(n0 - c->g.row0 + 1) * c->g.pitch,
                         c->g.pitch * sizeof(float),
                         rows_host + (size_t)(n0 - first_row) * c->g.W, c->g.W * sizeof(float),
                         c->g.W * sizeof(float), n1 - n0, cudaMemcpyHostToDevice, c->stream));
  }
  if (c->fuse == 2) {
    if (!c->phase2) {
      CU(cudaMalloc(&c->phase2, c->fused_floats() * sizeof(float)));
      CU(cudaMemsetAsync(c->phase2, 0, c->fused_floats() * sizeof(float), c->stream));
    }
    CU(cudaMemcpy2DAsync(c->phase2 + (size_t)(need0 - c->g.row0 + kFuseHalo) * c->g.pitch,
                         c->g.pitch * sizeof(float),
                         rows_host + (size_t)(need0 - first_row) * c->g.W, c->g.W * sizeof(float),
                         c->g.W * sizeof(float), need1 - need0, cudaMemcpyHostToDevice, c->stream));
  }
  c->pmask_pitch = (c->g.W + 31) / 32;
  if (!c->pmask) CU(cudaMalloc(&c->pmask, (size_t)c->g.rows * c->pmask_pitch));
  {
    const Geom sg = c->step_geom();
    dim3 block(64), grid((c->pmask_pitch + 63) / 64, min(sg.rows, 65535), c->nrep);
    phase_mask_kernel<<<grid, block, 0, c->stream>>>(c->phase, sg, c->pmask, c->pmask_pitch);
    CU(cudaGetLastError());
    c->launches++;
  }
  if (c->fuse == 2) {
    if (!c->pmask2) CU(cudaMalloc(&c->pmask2, (size_t)(c->g.rows + 2) * c->pmask_pitch));
    const Geom sg = c->step_geom();
    dim3 block(64), grid((c->pmask_pitch + 63) / 64, min(sg.rows + 2, 65535), c->nrep);
    phase_mask2_kernel<<<grid, block, 0, c->stream>>>(c->phase2, sg, c->pmask2, c->pmask_pitch);
    CU(cudaGetLastError());
    c->launches++;
  }
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int fib_set_table(fib_ctx* c, int table, const float* data, size_t n) {
  if (!c || !data) return fail(FIB_E_ARG, "ctx/data is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  if (table == FIB_TABLE_BR_CHEBY) {
    if (n != 12 * 9) return fail(FIB_E_ARG, "BR Chebyshev table must hold 12*9 floats, got %zu", n);
    CU(cudaStreamSynchronize(c->stream));
    memcpy(c->cheb, data, sizeof c->cheb);
    c->have_cheb = true;
    drop_graphs(c);
    return 0;
  }
  if (table == FIB_TABLE_COURT_LUT) {
    if (!c->lut) return fail(FIB_E_STATE, "this model has no lookup table");
    if (n != (size_t)kLutRows * kLutCols)
      return fail(FIB_E_ARG, "Courtemanche LUT must hold 150*30 floats, got %zu", n);
    CU(cudaMemcpyAsync(c->lut, data, n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    lut_transpose_kernel<<<(kLutRows + 63) / 64, 64, 0, c->stream>>>(c->lut, c->lut_t);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    c->launches++;
    c->have_lut = true;
    return 0;
  }
  return fail(FIB_E_ARG, "unknown table id %d", table);
}

extern "C" int fib_get_table(fib_ctx* c, int table, float* data, size_t n) {
  if (!c || !data) return fail(FIB_E_ARG, "ctx/data is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  if (table == FIB_TABLE_BR_CHEBY) {
    if (n != 12 * 9) return fail(FIB_E_ARG, "BR Chebyshev table holds 12*9 floats");
    memcpy(data, c->cheb, sizeof c->cheb);
    return 0;
  }
  if (table == FIB_TABLE_COURT_LUT) {
    if (!c->lut || !c->have_lut) return fail(FIB_E_STATE, "no lookup table has been set or built");
    if (n != (size_t)kLutRows * kLutCols) return fail(FIB_E_ARG, "Courtemanche LUT holds 150*30 floats");
    CU(cudaMemcpyAsync(data, c->lut, n * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return 0;
  }
  return fail(FIB_E_ARG, "unknown table id %d", table);
}

extern "C" int fib_build_lut(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (!c->lut) return fail(FIB_E_STATE, "this model has no lookup table");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  court_lut_kernel<<<(kLutRows + 63) / 64, 64, 0, c->stream>>>(c->lut);
  CU(cudaGetLastError());
  lut_transpose_kernel<<<(kLutRows + 63) / 64, 64, 0, c->stream>>>(c->lut, c->lut_t);
  CU(cudaGetLastError());
  c->launches += 2;
  c->have_lut = true;
  return 0;
}

extern "C" int fib_court_inter(fib_ctx* c, const float* v_host, size_t n, float* out_host) {
  if (!c || !v_host || !out_host) return fail(FIB_E_ARG, "NULL argument");
  if (n == 0) return 0;
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  struct Tmp {
    float* p = nullptr;
    ~Tmp() { cudaFree(p); }
  } tv, tq;
  CU(cudaMalloc(&tv.p, n * sizeof(float)));
  CU(cudaMalloc(&tq.p, n * kInterCols * sizeof(float)));
  float *dv = tv.p, *dq = tq.p;
  CU(cudaMemcpyAsync(dv, v_host, n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  court_inter_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(dv, (int)n, dq, kInterCols);
  CU(cudaGetLastError());
  c->launches++;
  CU(cudaMemcpyAsync(out_host, dq, n * kInterCols * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

// ------------------------------------------------------------------------------------------
// the step schedule
// ------------------------------------------------------------------------------------------
static int substeps_of(const fib_ctx* c, int op) {
  if (op == FIB_OP_ODE) return c->dt_per_step;
  return c->cfg.model == FIB_COURT ? 1 : 0;   // 'slow' is an empty group elsewhere
}

template <class M>
static void fill_common(fib_ctx* c, StepArgs<M>& a, int lr0, int nrows) {
  a.xin = c->x[c->cur];
  a.xout = c->x[c->cur ^ 1];
  for (int k = 0; k < M::NS; ++k) a.s[k] = c->s[k];
  a.phase = c->phase;
  a.pmask = c->pmask;
  a.pmask_pitch = c->pmask_pitch;
  a.lut = c->lut_t;
  a.lr0 = lr0;
  a.nrows = nrows;
  a.nz = c->nrep;
  a.zddt = c->zddt;
}

template <int MODE, bool LUT, bool US>
static cudaError_t launch_court(fib_ctx* c, int lr0, int nrows) {
  using M = Courtemanche<MODE, LUT, US>;
  StepArgs<M> a;
  fill_common<M>(c, a, lr0, nrows);
  const double dt = c->cfg.dt;
  const double dts = (c->cfg.model == FIB_COURT) ? dt * 10 : dt;   // court.py:118-122
  const double chron = (c->cfg.flags & FIB_F_NO_CHRONIC) ? 0.0 : 1.0;
  a.p.dt_fast = (float)dt;
  a.p.neg_dt_fast = (float)(-dt);
  a.p.dt_slow = (float)dts;
  a.p.neg_dt_slow = (float)(-dts);
  a.p.ddt = (float)(c->cfg.diff * dt);
  a.p.e_fCa = (float)expm1((double)(float)(-dts / 2.0));
  a.p.e_u = (float)expm1((double)(float)(-dts / 8.0));
  const bool noclip = c->cfg.flags & FIB_F_NO_CLIP;
  a.p.clip_lo = noclip ? -INFINITY : 0.00001f;
  a.p.clip_hi = noclip ? INFINITY : 0.99999f;
  a.p.k_to = (float)((1.0 - 0.5 * chron) * 100 * 0.1652);
  a.p.k_Kur = (float)((1.0 - 0.5 * chron) * 100);
  a.p.k_CaL = (float)((1.0 - 0.7 * chron) * 100 * 0.12375);
  return launch_step<M>(c->step_geom(), a, c->stream, c->sms);
}

// The tables the model's flags ask for have been set: checked before any step launch, and by fib_step before it
// defers iterations (so that the error reaches the caller that asked for them).
static int check_tables(const fib_ctx* c) {
  const uint32_t fl = c->cfg.flags;
  if (c->cfg.model == FIB_BR && (fl & FIB_F_CHEBY) && !c->have_cheb)
    return fail(FIB_E_STATE, "cheby=True but FIB_TABLE_BR_CHEBY has not been set");
  if (c->cfg.model >= FIB_COURT && (fl & FIB_F_LUT) && !c->have_lut)
    return fail(FIB_E_STATE, "lut=True but no table was set/built");
  return 0;
}

static Fenton4v::Params fenton_params(const fib_ctx* c) {
  return {(float)c->cfg.dt, (float)(c->cfg.diff * c->cfg.dt)};     // dt, ddt
}

// A Beeler-Reuter time step that advances the slow gates by n * dt (n = 0: they stay frozen), br.py:96-107.
template <class P>
static P br_params(const fib_ctx* c, int n) {
  const double dt = c->cfg.dt;
  const bool strict = (c->cfg.flags & FIB_F_CHEBY) && (c->cfg.flags & FIB_F_CHEBY_STRICT);
  P p;
  p.dt = (float)dt;
  p.neg_dt = (float)(-dt);
  p.neg_dt_slow = (float)(-(dt * n));
  p.ddt = (float)(c->cfg.diff * dt);
  // S_i = 2^(i-1) x^i (br.py:289-301): hand the kernel plain monomial coefficients (the strict
  // flavour evaluates the S-basis sum itself and takes the table as it is)
  for (int g = 0; g < 12; ++g)
    for (int i = 0; i < 9; ++i)
      p.poly[g][i] = (i < 2 || strict) ? c->cheb[g][i] : ldexpf(c->cheb[g][i], i - 1);
  return p;
}

// fn(slow, fast): the Beeler-Reuter model types of the flavour the flags select (strict Chebyshev, Chebyshev or
// exact gates), for a time step that advances the slow gates and for one that freezes them
template <class F>
static cudaError_t with_br_flavour(const fib_ctx* c, F&& fn) {
  const uint32_t fl = c->cfg.flags;
  if (!(fl & FIB_F_CHEBY)) return fn(BeelerReuter<0, true>(), BeelerReuter<0, false>());
  if (fl & FIB_F_CHEBY_STRICT) return fn(BeelerReuter<2, true>(), BeelerReuter<2, false>());
  return fn(BeelerReuter<1, true>(), BeelerReuter<1, false>());
}

// One time step `sub` of op over local rows [lr0, lr0+nrows).  Does NOT flip the ping-pong.
static int launch_substep(fib_ctx* c, int op, int sub, int lr0, int nrows) {
  if (nrows <= 0) return 0;
  // a batched context launches whole replicas only (no upload session, no shards): local rows = replica rows
  if (c->nrep > 1 && (lr0 != 0 || nrows != c->g.rows))
    return fail(FIB_E_STATE, "internal: a row range [%d,%d) of a batched context", lr0, lr0 + nrows);
  if (c->nrep > 1) nrows = c->g.rows / c->nrep;
  const int tr = check_tables(c);
  if (tr) return tr;
  const uint32_t fl = c->cfg.flags;
  cudaError_t e = cudaSuccess;
  switch (c->cfg.model) {
    case FIB_FENTON4V: {
      if (c->fuse == 2) {                       // time steps `sub` and `sub + 1` in one launch
        Fused2Args f;
        for (int v = 0; v < 4; ++v) { f.in[v] = c->fx[c->cur][v]; f.out[v] = c->fx[c->cur ^ 1][v]; }
        f.phase = c->phase2;
        f.pmask = c->pmask2;
        f.pmask_pitch = c->pmask_pitch;
        f.lr0 = lr0;
        f.nrows = nrows;
        f.R = 0;
        f.nz = c->nrep;
        f.zddt = c->zddt;
        f.p = fenton_params(c);
        e = launch_fused2(c->step_geom(), f, c->stream, c->sms);
        break;
      }
      StepArgs<Fenton4v> a;
      fill_common<Fenton4v>(c, a, lr0, nrows);
      a.p = fenton_params(c);
      e = launch_step<Fenton4v>(c->step_geom(), a, c->stream, c->sms);
      break;
    }
    case FIB_BR: {
      // br.py:96-107: skip -> solve(n=5) then 4x solve(n=0); else 5x solve(n=1)
      const int n = (fl & FIB_F_SKIP) ? (sub == 0 ? 5 : 0) : 1;
      auto go = [&](auto tag) {
        using M = decltype(tag);
        StepArgs<M> a;
        fill_common<M>(c, a, lr0, nrows);
        a.p = br_params<typename M::Params>(c, n);
        return launch_step<M>(c->step_geom(), a, c->stream, c->sms);
      };
      e = with_br_flavour(c, [&](auto slow, auto fast) { return n > 0 ? go(slow) : go(fast); });
      break;
    }
    case FIB_COURT: {
      const bool lut = fl & FIB_F_LUT;
      if (op == FIB_OP_ODE) e = lut ? launch_court<COURT_FAST, true, false>(c, lr0, nrows)
                                    : launch_court<COURT_FAST, false, false>(c, lr0, nrows);
      else                  e = lut ? launch_court<COURT_SLOW, true, false>(c, lr0, nrows)
                                    : launch_court<COURT_SLOW, false, false>(c, lr0, nrows);
      break;
    }
    default: {
      const bool lut = fl & FIB_F_LUT, us = fl & FIB_F_ULTRA_SLOW;
      if (us) e = lut ? launch_court<COURT_ALL, true, true>(c, lr0, nrows)
                      : launch_court<COURT_ALL, false, true>(c, lr0, nrows);
      else    e = lut ? launch_court<COURT_ALL, true, false>(c, lr0, nrows)
                      : launch_court<COURT_ALL, false, false>(c, lr0, nrows);
    }
  }
  if (e != cudaSuccess) return fail(FIB_E_CUDA, "step kernel launch failed: %s", cudaGetErrorString(e));
  c->launches++;
  return 0;
}

static bool op_writes_x(const fib_ctx* c, int op) { return !(c->cfg.model == FIB_COURT && op == FIB_OP_SLOW); }

// ---- NCCL halo exchange of buffer `buf` (rows just written), on `st` ------------------------
// fuse == 2: kFuseHalo rows of every plane of buffer set `b` (rows are pitch-contiguous)
// `sides`: bit 0 = the seam with rank - 1 (above), bit 1 = the seam with rank + 1 (below)
enum { kSeamUp = 1, kSeamDown = 2, kSeamBoth = 3 };
static int nccl_exchange_fused(fib_ctx* c, int b, cudaStream_t st, int sides) {
  const size_t P = c->g.pitch, n = (size_t)kFuseHalo * P;
  NC(g_nccl.GroupStart());
  for (int v = 0; v < 4; ++v) {
    float* buf = c->fx[b][v];
    if (c->rank > 0 && (sides & kSeamUp)) {
      NC(g_nccl.Send(buf + n, n, kNcclFloat, c->rank - 1, c->comm, st));
      NC(g_nccl.Recv(buf, n, kNcclFloat, c->rank - 1, c->comm, st));
    }
    if (c->rank + 1 < c->nranks && (sides & kSeamDown)) {
      NC(g_nccl.Send(buf + (size_t)c->g.rows * P, n, kNcclFloat, c->rank + 1, c->comm, st));
      NC(g_nccl.Recv(buf + (size_t)c->g.rows * P + n, n, kNcclFloat, c->rank + 1, c->comm, st));
    }
  }
  NC(g_nccl.GroupEnd());
  return 0;
}

static int nccl_exchange(fib_ctx* c, int b, cudaStream_t st, int sides = kSeamBoth) {
  if (c->fuse == 2) return nccl_exchange_fused(c, b, st, sides);
  float* buf = c->x[b];
  const size_t W = c->g.W, P = c->g.pitch;
  NC(g_nccl.GroupStart());
  if (c->rank > 0 && (sides & kSeamUp)) {
    NC(g_nccl.Send(buf + P, W, kNcclFloat, c->rank - 1, c->comm, st));
    NC(g_nccl.Recv(buf, W, kNcclFloat, c->rank - 1, c->comm, st));
  }
  if (c->rank + 1 < c->nranks && (sides & kSeamDown)) {
    NC(g_nccl.Send(buf + (size_t)c->g.rows * P, W, kNcclFloat, c->rank + 1, c->comm, st));
    NC(g_nccl.Recv(buf + (size_t)(c->g.rows + 1) * P, W, kNcclFloat, c->rank + 1, c->comm, st));
  }
  NC(g_nccl.GroupEnd());
  return 0;
}


// ------------------------------------------------------------------------------------------
// the persistent on-chip kernel (fib_persist.cuh): eligibility, tensor maps, launch
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess) {
      cudaGetLastError();
      p = nullptr;
    }
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}
// fp32 plane [rows][W] with row pitch `pitch` floats, box {bw, bh}
static bool make_tile_map(CUtensorMap* m, float* base, int W, int rows, int pitch, int bw, int bh) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)W, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)pitch * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)bw, (cuuint32_t)bh};
  const cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) ==
         CUDA_SUCCESS;
}

template <class MS, class MF, int TH, bool PHASE, bool ACT, bool EVENTS>
static cudaError_t launch_persist_t(fib_ctx* c, const PersistArgs<MS, MF>& a) {
  PersistMaps<MS::NS> maps;
  maps.x[0] = c->pmap_x[0];
  maps.x[1] = c->pmap_x[1];
  for (int k = 0; k < MS::NS; ++k) maps.s[k] = c->pmap_s[k];
  auto kern = persist_kernel<MS, MF, TH, PHASE, ACT, EVENTS>;
  constexpr size_t smem = persist_smem_bytes<MS::NS, TH>();
  static bool attr_set = false;           // per instantiation
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(c->persist_tiles);
  cfg.blockDim = dim3(kPersistThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = c->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;       // all tiles co-resident, or the launch fails
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  snprintf(last_kernel_name(), 160, "persist_kernel<%s,TH=%d,PHASE=%d%s%s%s>", MS::name(), TH, PHASE ? 1 : 0,
           ACT ? ",ACT=1" : "", a.frames ? ",FRAMES=1" : "", a.pace_n ? ",PACE=1" : "");
  return cudaLaunchKernelEx(&cfg, kern, maps, c->g, a);
}

template <class MS, class MF>
static cudaError_t launch_persist_m(fib_ctx* c, PersistArgs<MS, MF>& a, int iters) {
  a.x[0] = c->x[0];
  a.x[1] = c->x[1];
  a.cur = c->cur;
  a.period = substeps_of(c, FIB_OP_ODE);
  a.nsteps = a.period * iters;
  a.mail = c->pmail;
  a.base = c->pbase;
  a.err = c->perr;
  a.phase = c->phase;
  a.pmask = c->pmask;
  a.pmask_pitch = c->pmask_pitch;
  a.bw = c->persist_bw;
  a.ring = c->watch_var >= 0 ? c->ring : nullptr;
  a.ring_count = c->ring_count;
  a.probe_var = c->watch_var;
  a.probe_row = c->watch_row;
  a.probe_col = c->watch_col;
  a.act_prev = c->act_prev;
  a.act_maps = c->act_maps;
  a.act_plane = c->plane_floats();
  a.act_iter = c->act_iter;
  a.act_k0 = c->since(c->act_armed_at);
  a.act_up = c->act_up;
  a.act_down = c->act_down;
  // frames: the first recording iteration of this launch (k = k1 + it0), if there is one
  a.frames = nullptr;
  a.frame_step0 = a.nsteps + 1;
  a.frame_steps = 1;
  if (c->frames) {
    const unsigned long long k1 = c->since(c->fr_armed_at) + 1, f0 = c->fr_first, ev = c->fr_every;
    const unsigned long long kf = k1 <= f0 ? f0 : f0 + (k1 - f0 + ev - 1) / ev * ev;
    if (kf < k1 + (unsigned)iters) {
      a.frames = c->frames;
      a.frame_step0 = (int)(kf - k1 + 1) * a.period;
      a.frame_steps = (int)min(ev, (unsigned long long)kPersistMaxIters) * a.period;
      a.frame_slot0 = (int)((c->frames_upto(kf) - 1) % (unsigned long long)c->fr_cap);
      a.frame_cap = c->fr_cap;
      a.frame_var = c->fr_var;
      a.frame_stride = c->fr_stride;
      a.frame_cols = c->fr_cols;
      a.frame_floats = c->frame_floats();
    }
  }
  // pacing: the entries that fire in this launch, with one bit per iteration (the iteration's ode_iters is
  // ode_iters + 1 + it)
  a.pace_n = 0;
  for (const auto& p : c->paces) {
    unsigned long long mask = 0;
    for (int it = 0; it < iters; ++it)
      if (p.fires(c->ode_iters + 1 + it)) mask |= 1ull << it;
    if (!mask) continue;
    const int e = a.pace_n++;
    a.pace_rect[e][0] = p.r0;
    a.pace_rect[e][1] = p.r1;
    a.pace_rect[e][2] = p.c0;
    a.pace_rect[e][3] = p.c1;
    a.pace_value[e] = p.value;
    a.pace_floor[e] = p.floor_v;
    a.pace_mask[e] = mask;
  }
  const bool ph = c->phase != nullptr, act = c->act_maps != nullptr, fr = a.frames != nullptr || a.pace_n > 0;
  auto flag = [](bool b, auto&& fn) { return b ? fn(std::true_type()) : fn(std::false_type()); };
  auto go = [&](auto th) {
    return flag(ph, [&](auto P) {
      return flag(act, [&](auto A) {
        return flag(fr, [&](auto F) {
          return launch_persist_t<MS, MF, decltype(th)::value, decltype(P)::value, decltype(A)::value,
                                  decltype(F)::value>(c, a);
        });
      });
    });
  };
  switch (c->persist_th) {
    case 2: return go(std::integral_constant<int, 2>());
    case 4: return go(std::integral_constant<int, 4>());
    case 8:
      if constexpr (MS::NS <= 3) return go(std::integral_constant<int, 8>());
    default: return cudaErrorInvalidValue;
  }
}

// Decides once per context (and again after fib_set_phase) whether ODE iterations run as the persistent
// kernel: Fenton 4v (one step per launch layout) or Beeler-Reuter, unsharded, W <= 512, at most 8 (4v) /
// 4 (BR) rows per SM, cooperative launch available.  FIB_PERSIST=0 or FIB_F_NO_PERSIST switch it off.
static void decide_persist(fib_ctx* c) {
  c->persist = 0;
  static const bool env_on = !(getenv("FIB_PERSIST") && atoi(getenv("FIB_PERSIST")) == 0);
  if (!env_on || (c->cfg.flags & FIB_F_NO_PERSIST)) return;
  const int model = c->cfg.model;
  if (!(model == FIB_FENTON4V || model == FIB_BR) || c->fuse != 1) return;
  // one CTA per SM for one grid: a batched context exists to leave that regime
  if (c->comm || c->nrep > 1 || c->g.rows != c->g.H || c->g.W > kPersistThreads) return;
  int coop = 0;
  if (cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, c->cfg.device) != cudaSuccess || !coop) return;
  const int max_th = model == FIB_FENTON4V ? 8 : 4;
  const int need = (c->g.H + c->sms - 1) / c->sms;
  int th = 2;
  while (th < need) th *= 2;
  if (th > max_th) return;
  const int bw = c->g.W >= kPersistBox ? kPersistBox : (c->g.W + 3) / 4 * 4;
  const int P = c->g.pitch;
  bool ok = make_tile_map(&c->pmap_x[0], c->x[0] + P, c->g.W, c->g.H, P, bw, th) &&
            make_tile_map(&c->pmap_x[1], c->x[1] + P, c->g.W, c->g.H, P, bw, th);
  for (int k = 0; ok && k + 1 < c->nvars; ++k) ok = make_tile_map(&c->pmap_s[k], c->s[k], c->g.W, c->g.H, P, bw, th);
  if (!ok) return;
  const int tiles = (c->g.H + th - 1) / th;
  if (!c->pmail) {
    const size_t fbytes = sizeof(unsigned long long) * persist_mailbox_words(c->sms);
    if (cudaMalloc(&c->pmail, fbytes) != cudaSuccess) { cudaGetLastError(); return; }
    cudaMemsetAsync(c->pmail, 0, fbytes, c->stream);       // step number 0 = "nothing published yet"
    if (cudaHostAlloc(&c->perr, sizeof(int), cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); return; }
    *c->perr = 0;
  }
  c->persist_th = th;
  c->persist_tiles = tiles;
  c->persist_bw = bw;
  c->persist = 1;
}

// ------------------------------------------------------------------------------------------
// observers: the probe ring, the activation maps and the frame recorder sample the state at the end of every ODE
// iteration.  Every stepping route calls the two halves of one hook: record_observers inside the iteration (the
// graphs capture it) and end_iterations on the host once the route has enqueued iterations.
// ------------------------------------------------------------------------------------------
// frame j of the current plane into its ring slot, and a ledger mark behind it
static int launch_frame(fib_ctx* c, unsigned long long j) {
  if (c->fr_rows > 0) {
    const float* src = owned_rows(c, c->fr_var) + (size_t)c->fr_lr0 * c->g.pitch;
    float* dst = c->frames + (j % (unsigned long long)c->fr_cap) * c->frame_floats();
    const dim3 grid((c->fr_cols + 127) / 128, min(c->fr_rows, 65535));
    frame_record_kernel<<<grid, 128, 0, c->stream>>>(src, (size_t)c->fr_stride * c->g.pitch, c->fr_stride,
                                                     c->fr_rows, c->fr_cols, dst);
    CU(cudaGetLastError());
    c->launches++;
  }
  return c->frame_ledger.mark(c->stream, c->frames_recorded());
}

// Local rows [lo, hi) of the CURRENT buffers have finished an ODE iteration: the probe records its cell if it lies
// there.  The upload session finishes iterations in row blocks; only the probe can be armed while it is open.
static int observe_rows(fib_ctx* c, int lo, int hi) {
  const int lr = c->watch_row - c->g.row0;
  if (c->watch_var < 0 || lr < lo || lr >= hi) return 0;
  probe_record_kernel<<<1, probe_threads(c), 0, c->stream>>>(watch_src(c), replica_step(c), c->watch_n, c->ring,
                                                             c->ring_cap, c->ring_count);
  CU(cudaGetLastError());
  c->launches++;
  return 0;
}

// The graph-capturable half of the hook, after an iteration of `op` on the CURRENT buffers: the activation update
// and the advance of its device iteration index, then the probe record.
static int record_observers(fib_ctx* c, int op) {
  if (op != FIB_OP_ODE) return 0;
  if (c->act_maps) {
    const size_t n4 = c->plane_floats() / 4;
    const int grid = (int)min((n4 + 255) / 256, (size_t)c->sms * 32);
    activation_update_kernel<<<grid, 256, 0, c->stream>>>(reinterpret_cast<const float4*>(owned_rows(c, 0)),
                                                          reinterpret_cast<float4*>(c->act_prev), c->act_maps, n4,
                                                          c->plane_floats(), c->act_iter, c->act_up, c->act_down);
    activation_advance_kernel<<<1, 1, 0, c->stream>>>(c->act_iter);
    CU(cudaGetLastError());
    c->launches += 2;
  }
  return observe_rows(c, 0, c->g.rows);
}

// The pacing entries that fire after the iteration just counted, in the order they were added: the stimulus of
// each, then the probe's value of this iteration taken again (mark_written), as after a fib_stimulate.
static int fire_paces(fib_ctx* c) {
  bool fired = false;
  for (const auto& p : c->paces)
    if (p.fires(c->ode_iters)) {
      const int r = launch_stim(c, 0, p.replica, p.r0, p.r1, p.c0, p.c1, p.value, p.floor_v);
      if (r) return r;
      fired = true;
    }
  if (fired) mark_written(c, 0);
  return 0;
}

// The host half of the hook: the route has enqueued `n` iterations of `op`, after their record_observers nodes or,
// `persistent`, as one persistent launch that recorded its probe values and frames and applied its pacing itself.
// Counts them; gathers the frame of a recording iteration (the other routes end one iteration at a time; no recorder
// or pacing is armed behind an upload) or marks the frame ledger behind the launch; then fires the pacing entries
// of the iteration, so that the frame and the activation sample precede the stimulus and the probe follows it;
// marks the probe ledger behind a persistent launch.  A stimulus marks the halos dirty: a sharded route that goes
// on stepping refreshes them first.
static int end_iterations(fib_ctx* c, int op, int n, bool persistent = false) {
  if (op != FIB_OP_ODE) return 0;
  const unsigned long long frames0 = c->frames_recorded();
  c->ode_iters += (unsigned)n;
  int r = 0;
  if (c->frames && c->frames_recorded() != frames0)
    r = persistent ? c->frame_ledger.mark(c->stream, c->frames_recorded()) : launch_frame(c, c->frames_recorded() - 1);
  if (!r && !persistent) r = fire_paces(c);
  if (!r && persistent && c->watch_var >= 0) r = c->probe_ledger.mark(c->stream, c->since(c->probe_armed_at));
  c->paces.erase(std::remove_if(c->paces.begin(), c->paces.end(),
                                [&](const fib_ctx::Pace& p) { return p.done(c->ode_iters); }),
                 c->paces.end());
  return r;
}

// `iters` ODE iterations (dt_per_step time steps each) as ONE launch
static int run_iteration_persist(fib_ctx* c, int iters) {
  const int tr = check_tables(c);
  if (tr) return tr;
  cudaError_t e;
  if (c->cfg.model == FIB_FENTON4V) {
    PersistArgs<Fenton4v, Fenton4v> a;
    a.slow_first_only = 0;
    a.ps = a.pf = fenton_params(c);
    e = launch_persist_m<Fenton4v, Fenton4v>(c, a, iters);
  } else {
    const bool skip = c->cfg.flags & FIB_F_SKIP;
    e = with_br_flavour(c, [&](auto slow, auto fast) {
      using MS = decltype(slow);
      using MF = decltype(fast);
      PersistArgs<MS, MF> a;
      a.slow_first_only = skip ? 1 : 0;                                               // br.py:96-107
      a.ps = br_params<typename MS::Params>(c, skip ? 5 : 1);
      a.pf = br_params<typename MF::Params>(c, 0);
      return launch_persist_m<MS, MF>(c, a, iters);
    });
  }
  if (e != cudaSuccess) {
    // e.g. the tiles cannot all be resident (another context holds SMs): never a partial launch.
    // Fall back to one launch per step for the rest of this context's life.
    cudaGetLastError();
    c->persist = 0;
    return 1;           // caller retries on the plain path; these iterations were not counted
  }
  c->launches++;
  const int ns = substeps_of(c, FIB_OP_ODE) * iters;
  c->pbase += (unsigned)ns;
  if (ns & 1) c->cur ^= 1;
  return end_iterations(c, FIB_OP_ODE, iters, true);
}

static int check_persist_error(fib_ctx* c) {
  if (c->perr && *c->perr) {
    *c->perr = 0;
    return fail(FIB_E_STATE, "persistent kernel: a tile waited for its neighbour beyond the spin limit "
                "(state is invalid); set FIB_PERSIST=0 to use one launch per step");
  }
  return 0;
}

// one iteration as direct launches: what the iteration graphs capture
static int run_iteration_plain(fib_ctx* c, int op) {
  const int ns = substeps_of(c, op);
  for (int s = 0; s < ns; s += c->fuse) {
    int r = launch_substep(c, op, s, 0, c->g.rows);
    if (r) return r;
    if (op_writes_x(c, op)) c->cur ^= 1;
  }
  return record_observers(c, op);
}

// boundary rows first, halo exchange on the side stream overlapped with the interior rows
static int run_iteration_nccl(fib_ctx* c, int op) {
  const int ns = substeps_of(c, op);
  const int rows = c->g.rows;
  const int nb = c->fuse;      // rows the neighbours need from each edge = time steps per launch
  for (int s = 0; s < ns; s += c->fuse) {
    if (!op_writes_x(c, op)) {
      int r = launch_substep(c, op, s, 0, rows);
      if (r) return r;
      continue;
    }
    if (c->comm_pending) {   // halos of x[cur] must have arrived
      CU(cudaStreamWaitEvent(c->stream, c->ev_comm, 0));
      c->comm_pending = false;
    }
    int r;
    if (rows >= 3 * nb) {
      if ((r = launch_substep(c, op, s, 0, nb))) return r;
      if ((r = launch_substep(c, op, s, rows - nb, nb))) return r;
      CU(cudaEventRecord(c->ev_bnd, c->stream));
      CU(cudaStreamWaitEvent(c->comm_stream, c->ev_bnd, 0));
      if ((r = nccl_exchange(c, c->cur ^ 1, c->comm_stream))) return r;
      CU(cudaEventRecord(c->ev_comm, c->comm_stream));
      c->comm_pending = true;
      if ((r = launch_substep(c, op, s, nb, rows - 2 * nb))) return r;
    } else {
      if ((r = launch_substep(c, op, s, 0, rows))) return r;
      if ((r = nccl_exchange(c, c->cur ^ 1, c->stream))) return r;
    }
    c->cur ^= 1;
  }
  return record_observers(c, op);
}

// Every rank must take part in an exchange, but a host write (fib_set_state / fib_set_rect /
// fib_stimulate) is local knowledge: a rank cannot know whether its neighbour's edge rows changed.
// So fib_step ALWAYS refreshes the halos of the current buffer first (one small grouped send/recv
// per fib_step call, idempotent when nothing was written): the decision is the same on all ranks.
static int refresh_halos_nccl(fib_ctx* c) {
  CU(wait_comm(c));
  int r = nccl_exchange(c, c->cur, c->stream);
  if (r) return r;
  c->halo_dirty = false;
  return 0;
}

// n_iter iterations of `op`, enqueued now
static int step_now(fib_ctx* c, int op, int n_iter) {
  if (c->comm) {
    // a pacing stimulus inside this call (halo_dirty) changed edge rows the neighbours hold as halo: every rank
    // registered the same entries, so all of them take the same refresh
    int r = refresh_halos_nccl(c);
    for (int i = 0; i < n_iter && !r; ++i) {
      if (!(r = run_iteration_nccl(c, op))) r = end_iterations(c, op, 1);
      if (!r && c->halo_dirty && i + 1 < n_iter) r = refresh_halos_nccl(c);
    }
    return r;
  }
  if (c->persist == 1 && op == FIB_OP_ODE) {
    // up to kPersistMaxIters iterations per launch (no launch gap, no tile reload between them); a
    // watched probe is recorded by the kernel itself after every iteration
    int i = 0;
    while (i < n_iter) {
      const int batch = min(n_iter - i, kPersistMaxIters);
      int r = run_iteration_persist(c, batch);
      if (r > 0) break;                 // could not launch: plain path from here on
      if (r) return r;
      i += batch;
    }
    if (i == n_iter) return 0;
    n_iter -= i;
  }
  if (c->cfg.flags & FIB_F_NO_GRAPH) {
    int r = 0;
    for (int i = 0; i < n_iter && !r; ++i)
      if (!(r = run_iteration_plain(c, op))) r = end_iterations(c, op, 1);
    return r;
  }
  // CUDA graph of one iteration, cached per (op, ping-pong parity)
  for (int i = 0; i < n_iter; ++i) {
    const GraphKey* gk = nullptr;
    for (auto& k : c->graphs)
      if (k.op == op && k.cur == c->cur) gk = &k;
    if (!gk) {
      // capture one iteration and measure what it launches and where it leaves the state; nothing runs yet
      GraphKey k = {op, c->cur, 0, 0, nullptr};
      const uint64_t l0 = c->launches;
      cudaGraph_t graph = nullptr;
      CU(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
      int r = run_iteration_plain(c, op);
      cudaError_t ce = cudaStreamEndCapture(c->stream, &graph);
      k.cur_end = c->cur;
      k.launches = c->launches - l0;
      c->launches = l0;
      c->cur = k.cur;
      if (r) { if (graph) cudaGraphDestroy(graph); return r; }
      if (ce != cudaSuccess) return fail(FIB_E_CUDA, "graph capture failed: %s", cudaGetErrorString(ce));
      CU(cudaGraphInstantiate(&k.exec, graph, 0));
      CU(cudaGraphDestroy(graph));
      c->graphs.push_back(k);
      gk = &c->graphs.back();
    }
    CU(cudaGraphLaunch(gk->exec, c->stream));
    c->launches += gk->launches;
    c->cur = gk->cur_end;
    const int r = end_iterations(c, op, 1);
    if (r) return r;
  }
  return 0;
}

// Ends a pipelined upload (see set_rect_impl) and runs the `n` ODE iterations deferred meanwhile.
// With blocks ending at rows a_0 < a_1 < .. < a_m = H and nb rows of halo per launch, launch l of block j
// covers rows [a_{j-1} - nb (l+1), a_j - nb (l+1)) (first block from row 0, last block to row H): every row
// gets every launch exactly once and in order, a launch reads only rows its predecessors have brought to
// its time level, and block j's launches wait for block j's copies only -- the same arithmetic on the
// same values as stepping after the whole upload, so the result is bit-identical.
// iterations a session can still defer: launch l of the first block ends at row a_0 - nb (l + 1) > 0
static int upload_room_iters(const fib_ctx* c) {
  if (!c->up_session || c->arrivals.empty()) return 0;
  const int nl = substeps_of(c, FIB_OP_ODE) / c->fuse;
  return max((c->arrivals[0].d_end / c->fuse - 3) / max(nl, 1), 0);
}

// NCCL shards (`comm_skew`, only through fib_step_behind_upload -- every rank must take the same path): the
// skew starts at the edge the upload started at.  Even ranks upload top to bottom and odd ranks bottom to top,
// so both shards of a seam either BEGIN there (their first blocks advance launch by launch in lock step,
// exchanging the seam's halo rows after every launch) or END there (the same for their last blocks); the
// blocks in between need no exchange at all.
static int finish_upload_session(fib_ctx* c, int n, bool comm_skew = false) {
  c->up_session = false;
  std::vector<fib_ctx::Arrival> blocks;
  blocks.swap(c->arrivals);
  auto release = [&]() {
    for (auto& b : blocks) c->ev_pool.push_back(b.ev);
  };
  const int op = FIB_OP_ODE;
  const int nb = c->fuse, nl = substeps_of(c, op) / c->fuse, L = n * nl;
  const int rows = c->g.rows, dir = c->up_dir;
  const bool sharded = c->comm != nullptr;
  bool skew = n > 0 && blocks.size() > 1 && blocks.back().d_end == rows && c->persist != 1 &&
              blocks[0].d_end > nb * (L + 2) && (!sharded || comm_skew);
  for (size_t j = 1; skew && j < blocks.size(); ++j) skew = blocks[j].d_end - blocks[j - 1].d_end > 2 * nb;
  if (!skew) {
    if (!blocks.empty()) CU(cudaStreamWaitEvent(c->stream, blocks.back().ev, 0));
    release();
    if (comm_skew) return fail(FIB_E_STATE, "fib_step_behind_upload: this upload cannot be pipelined (fib_upload_state)");
    return n ? step_now(c, op, n) : 0;
  }
  // the seams of this shard, named by where the upload began
  const int side_start = dir > 0 ? kSeamUp : kSeamDown, side_end = dir > 0 ? kSeamDown : kSeamUp;
  const bool has_up = sharded && c->rank > 0, has_down = sharded && c->rank + 1 < c->nranks;
  const bool seam_start = dir > 0 ? has_up : has_down, seam_end = dir > 0 ? has_down : has_up;
  if (sharded) CU(wait_comm(c));
  const int cur0 = c->cur;
  const bool flips = op_writes_x(c, op);
  int r = 0;
  for (size_t j = 0; j < blocks.size() && !r; ++j) {
    CU(cudaStreamWaitEvent(c->stream, blocks[j].ev, 0));
    const bool first = j == 0, last = j + 1 == blocks.size();
    // the seam's halo rows of the state just uploaded
    if (first && seam_start) r = nccl_exchange(c, cur0, c->stream, side_start);
    if (!r && last && seam_end) r = nccl_exchange(c, cur0, c->stream, side_end);
    for (int l = 0; l < L && !r; ++l) {
      const int dlo = first ? 0 : blocks[j - 1].d_end - nb * (l + 1);
      const int dhi = last ? rows : blocks[j].d_end - nb * (l + 1);
      const int lo = dir > 0 ? dlo : rows - dhi, hi = dir > 0 ? dhi : rows - dlo;
      c->cur = cur0 ^ ((flips && (l & 1)) ? 1 : 0);
      r = launch_substep(c, op, (l % nl) * c->fuse, lo, hi - lo);
      if (!r && flips && first && seam_start) r = nccl_exchange(c, c->cur ^ 1, c->stream, side_start);
      if (!r && flips && last && seam_end) r = nccl_exchange(c, c->cur ^ 1, c->stream, side_end);
      if (!r && (l + 1) % nl == 0) {    // rows [lo, hi) have finished an iteration, in the buffer just written
        if (flips) c->cur ^= 1;
        r = observe_rows(c, lo, hi);
      }
    }
  }
  c->cur = cur0 ^ ((flips && (L & 1)) ? 1 : 0);
  if (sharded && !r) c->halo_dirty = false;
  release();
  return r ? r : end_iterations(c, op, n);
}

static int flush_pending(fib_ctx* c) {
  const int n = c->pending;
  c->pending = 0;
  if (c->up_session) return finish_upload_session(c, n);
  return n ? step_now(c, FIB_OP_ODE, n) : 0;
}

extern "C" int fib_step(fib_ctx* c, int op, int n_iter) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (op != FIB_OP_ODE && op != FIB_OP_SLOW) return fail(FIB_E_ARG, "unknown op %d", op);
  if (n_iter < 0) return fail(FIB_E_ARG, "n_iter < 0");
  if (substeps_of(c, op) == 0 || n_iter == 0) return 0;
  DevGuard dg(c->cfg.device);
  if (!c->comm && c->g.rows != c->g.H)
    return fail(FIB_E_STATE, "a row shard needs fib_comm_init (multi-process) or fib_step_group");
  if (!c->comm && c->persist < 0) decide_persist(c);
  if (c->up_session && !c->comm && op == FIB_OP_ODE && c->persist != 1 && !c->arrivals.empty()) {
    // an upload is still in flight: count the iterations, run them behind the copies when something looks
    // (finish_upload_session); at most as many as the first block's height allows
    if (c->pending + n_iter <= upload_room_iters(c)) {
      c->pending += n_iter;
      return 0;
    }
  }
  if (c->persist == 1 && op == FIB_OP_ODE) {
    // persistent path: count now, launch later (see FLUSH); whatever can fail is checked here
    const int tr = check_tables(c);
    if (tr) return tr;
    while (n_iter > 0) {
      const int take = min(n_iter, kPersistMaxIters - c->pending);
      c->pending += take;
      n_iter -= take;
      if (c->pending == kPersistMaxIters) FLUSH(c);
    }
    return 0;
  }
  FLUSH(c);
  return step_now(c, op, n_iter);
}

// What a caller has to know before it asks for fib_step_behind_upload on NCCL shards (every rank must take the
// same decision, so the host side reduces these over the ranks first: fib_tf_b200/ionic.py run()).
extern "C" int fib_upload_state(const fib_ctx* c, int* open, int* complete, int* direction, int* max_iters) {
  if (!c || !open || !complete || !direction || !max_iters) return fail(FIB_E_ARG, "NULL argument");
  *open = c->up_session ? 1 : 0;
  *complete = (c->up_session && !c->arrivals.empty() && c->arrivals.back().d_end == c->g.rows && c->arrivals.size() > 1) ? 1 : 0;
  *direction = c->up_session ? c->up_dir : 0;
  *max_iters = upload_room_iters(c);
  return 0;
}

// n_iter ODE iterations behind a complete pipelined upload, NOW (enqueue only).  On NCCL shards this is a
// collective with its own exchange pattern: all ranks call it, with the same n_iter, after agreeing that every
// rank has a complete upload whose direction is top-to-bottom on even and bottom-to-top on odd ranks.
extern "C" int fib_step_behind_upload(fib_ctx* c, int n_iter) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (n_iter < 1) return fail(FIB_E_ARG, "n_iter < 1");
  DevGuard dg(c->cfg.device);
  if (!c->up_session) return fail(FIB_E_STATE, "fib_step_behind_upload: no pipelined upload is open");
  if (c->pending) return fail(FIB_E_STATE, "fib_step_behind_upload: iterations are already deferred on this context");
  if (c->comm && ((c->rank % 2 == 0) != (c->up_dir > 0)))
    return fail(FIB_E_STATE, "fib_step_behind_upload: rank %d must upload %s", c->rank,
                c->rank % 2 == 0 ? "top to bottom" : "bottom to top");
  if (n_iter > upload_room_iters(c))
    return fail(FIB_E_STATE, "fib_step_behind_upload: at most %d iterations fit behind this upload", upload_room_iters(c));
  if (!c->comm && c->persist < 0) decide_persist(c);
  return finish_upload_session(c, n_iter, c->comm != nullptr);
}

// ---- in-process shard group: lock-step, device-to-device halo copies ------------------------
static int group_copy_halos(fib_ctx** cs, int n, bool written_buffer) {
  // copies the boundary rows of buffer (cur^1 if written_buffer else cur) into the neighbours'
  // halo rows, each on the SOURCE stream, then records ev_group on every stream.  One row of the
  // diffusing variable, or kFuseHalo rows of every plane in the two-steps-per-launch layout.
  for (int i = 0; i < n; ++i) {
    fib_ctx* c = cs[i];
    DevGuard dg(c->cfg.device);
    const int b = written_buffer ? (c->cur ^ 1) : c->cur;
    const bool fused = c->fuse == 2;
    const int nplanes = fused ? 4 : 1, hr = fused ? kFuseHalo : 1;
    const size_t P = c->g.pitch;
    // one row: W floats; several rows: pitch-contiguous block
    const size_t bytes = (hr == 1 ? (size_t)c->g.W : (size_t)hr * P) * sizeof(float);
    for (int v = 0; v < nplanes; ++v) {
      float* mine = fused ? c->fx[b][v] : c->x[b];
      if (i > 0) {
        fib_ctx* up = cs[i - 1];
        const int ub = written_buffer ? (up->cur ^ 1) : up->cur;
        float* theirs = fused ? up->fx[ub][v] : up->x[ub];
        CU(cudaMemcpyPeerAsync(theirs + (size_t)(up->g.rows + hr) * up->g.pitch, up->cfg.device,
                               mine + (size_t)hr * P, c->cfg.device, bytes, c->stream));
      }
      if (i + 1 < n) {
        fib_ctx* dn = cs[i + 1];
        const int db = written_buffer ? (dn->cur ^ 1) : dn->cur;
        float* theirs = fused ? dn->fx[db][v] : dn->x[db];
        CU(cudaMemcpyPeerAsync(theirs, dn->cfg.device, mine + (size_t)c->g.rows * P, c->cfg.device,
                               bytes, c->stream));
      }
    }
    CU(cudaEventRecord(c->ev_group, c->stream));
  }
  return 0;
}

static int group_wait_neighbours(fib_ctx** cs, int n) {
  for (int i = 0; i < n; ++i) {
    DevGuard dg(cs[i]->cfg.device);
    if (i > 0) CU(cudaStreamWaitEvent(cs[i]->stream, cs[i - 1]->ev_group, 0));
    if (i + 1 < n) CU(cudaStreamWaitEvent(cs[i]->stream, cs[i + 1]->ev_group, 0));
  }
  return 0;
}

extern "C" int fib_step_group(fib_ctx** cs, int n, int op, int n_iter) {
  if (!cs || n < 1) return fail(FIB_E_ARG, "empty shard group");
  if (op != FIB_OP_ODE && op != FIB_OP_SLOW) return fail(FIB_E_ARG, "unknown op %d", op);
  int row = 0;
  for (int i = 0; i < n; ++i) {
    if (!cs[i]) return fail(FIB_E_ARG, "shard %d is NULL", i);
    if (cs[i]->nrep > 1) return fail(FIB_E_ARG, "fib_step_group: shard %d is a batched context", i);
    if (cs[i]->g.row0 != row || cs[i]->g.H != cs[0]->g.H || cs[i]->g.W != cs[0]->g.W ||
        cs[i]->cfg.model != cs[0]->cfg.model || cs[i]->cfg.flags != cs[0]->cfg.flags ||
        cs[i]->fuse != cs[0]->fuse)
      return fail(FIB_E_ARG, "shard %d is not the row-adjacent continuation of shard %d", i, i - 1);
    row += cs[i]->g.rows;
  }
  if (row != cs[0]->g.H) return fail(FIB_E_ARG, "shards cover %d of %d rows", row, cs[0]->g.H);
  for (int i = 0; i < n; ++i) {
    DevGuard dg(cs[i]->cfg.device);
    FLUSH(cs[i]);
  }
  // shards on different devices of this process: direct NVLink copies need peer access
  for (int i = 0; i + 1 < n; ++i) {
    const int a = cs[i]->cfg.device, b = cs[i + 1]->cfg.device;
    if (a == b) continue;
    for (int dir = 0; dir < 2; ++dir) {
      DevGuard dg(dir ? b : a);
      cudaError_t e = cudaDeviceEnablePeerAccess(dir ? a : b, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();     // not fatal: cudaMemcpyPeerAsync then stages through the host
      } else if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
      }
    }
  }
  const int ns = substeps_of(cs[0], op);
  if (ns == 0 || n_iter == 0) return 0;
  int r;
  bool dirty = false;
  for (int i = 0; i < n; ++i) dirty |= cs[i]->halo_dirty;
  if (dirty) {
    if ((r = group_copy_halos(cs, n, false))) return r;
    if ((r = group_wait_neighbours(cs, n))) return r;
    for (int i = 0; i < n; ++i) cs[i]->halo_dirty = false;
  }
  for (int it = 0; it < n_iter; ++it) {
    for (int s = 0; s < ns; s += cs[0]->fuse) {
      for (int i = 0; i < n; ++i) {
        DevGuard dg(cs[i]->cfg.device);
        if ((r = launch_substep(cs[i], op, s, 0, cs[i]->g.rows))) return r;
      }
      if (op_writes_x(cs[0], op)) {
        if ((r = group_copy_halos(cs, n, true))) return r;
        if ((r = group_wait_neighbours(cs, n))) return r;
        for (int i = 0; i < n; ++i) cs[i]->cur ^= 1;
      }
    }
    dirty = false;
    for (int i = 0; i < n; ++i) {
      DevGuard dg(cs[i]->cfg.device);
      if ((r = record_observers(cs[i], op)) || (r = end_iterations(cs[i], op, 1))) return r;
      dirty |= cs[i]->halo_dirty;
    }
    if (dirty && it + 1 < n_iter) {   // a pacing stimulus changed edge rows the neighbours hold as halo
      if ((r = group_copy_halos(cs, n, false))) return r;
      if ((r = group_wait_neighbours(cs, n))) return r;
      for (int i = 0; i < n; ++i) cs[i]->halo_dirty = false;
    }
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// stimulus, probes, reductions
// ------------------------------------------------------------------------------------------
extern "C" int fib_set_replica_diff(fib_ctx* c, const double* diff, size_t n) {
  if (!c || !diff) return fail(FIB_E_ARG, "ctx/diff is NULL");
  if (n != (size_t)c->nrep) return fail(FIB_E_ARG, "fib_set_replica_diff: n=%zu, the context has %d replicas", n, c->nrep);
  if (c->nrep == 1) return fail(FIB_E_STATE, "fib_set_replica_diff: not a batched context (set fib_config.diff)");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  drop_graphs(c);
  return upload_replica_diff(c, diff);
}

extern "C" int fib_stimulate_replica(fib_ctx* c, int replica, int var, int r0, int r1, int c0, int c1, float value,
                                     float floor_v) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (replica < -1 || replica >= c->nrep)
    return fail(FIB_E_ARG, "replica %d out of range -1..%d", replica, c->nrep - 1);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  const int r = launch_stim(c, var, replica, r0, r1, c0, c1, value, floor_v);
  if (r) return r;
  mark_written(c, var);
  return 0;
}

extern "C" int fib_stimulate(fib_ctx* c, int var, int r0, int r1, int c0, int c1, float value,
                             float floor_v) {
  return fib_stimulate_replica(c, -1, var, r0, r1, c0, c1, value, floor_v);
}

extern "C" int fib_pace_add(fib_ctx* c, int r0, int r1, int c0, int c1, float value, float floor_v, int first,
                            int every, int count, int* id) {
  return fib_pace_add_replica(c, -1, r0, r1, c0, c1, value, floor_v, first, every, count, id);
}

extern "C" int fib_pace_add_replica(fib_ctx* c, int replica, int r0, int r1, int c0, int c1, float value,
                                    float floor_v, int first, int every, int count, int* id) {
  if (!c || !id) return fail(FIB_E_ARG, "ctx/id is NULL");
  if (replica < -1 || replica >= c->nrep)
    return fail(FIB_E_ARG, "replica %d out of range -1..%d", replica, c->nrep - 1);
  if (first < 1 || count < 0 || (count != 1 && every < 1))
    return fail(FIB_E_ARG, "fib_pace_add: need first >= 1, count >= 0 and every >= 1 unless count == 1 (got first %d, "
                "every %d, count %d)", first, every, count);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  if ((int)c->paces.size() >= kPaceMax)
    return fail(FIB_E_STATE, "fib_pace_add: at most %d pacing entries per context", kPaceMax);
  fib_ctx::Pace p;
  p.id = c->pace_ids++;
  p.replica = replica;
  p.r0 = r0;
  p.r1 = r1;
  p.c0 = c0;
  p.c1 = c1;
  p.value = value;
  p.floor_v = floor_v;
  p.at = c->ode_iters + (unsigned)first;
  p.every = count == 1 ? 1 : (unsigned)every;
  p.count = (unsigned)count;
  c->paces.push_back(p);
  *id = p.id;
  return 0;
}

extern "C" int fib_pace_remove(fib_ctx* c, int id) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (id >= c->pace_ids) return fail(FIB_E_ARG, "fib_pace_remove: no pacing entry %d was added", id);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  c->paces.erase(std::remove_if(c->paces.begin(), c->paces.end(),
                                [&](const fib_ctx::Pace& p) { return id < 0 || p.id == id; }),
                 c->paces.end());
  return 0;
}

extern "C" int fib_probe(fib_ctx* c, int var, int row, int col, float* out) {
  if (!c || !out) return fail(FIB_E_ARG, "ctx/out is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (row < c->g.row0 || row >= c->g.row0 + c->g.rows || col < 0 || col >= c->g.W)
    return fail(FIB_E_ARG, "probe (%d,%d) is not in this shard", row, col);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaMemcpyAsync(out, owned_rows(c, var) + (size_t)(row - c->g.row0) * c->g.pitch + col,
                     sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

static int reduce_weighted(fib_ctx* c, int var, const float* w, int parts, double* sum_wx, double* sum_w);
// a sum over a batched context would mix its replicas: a silently wrong mean, rho or electrogram
static int refuse_batched_sum(const fib_ctx* c, const char* what) {
  return fail(FIB_E_STATE, "%s sums over the whole context, which holds %d replicas", what, c->nrep);
}

extern "C" int fib_weighted_sum(fib_ctx* c, int var, double* sum_wx, double* sum_w) {
  if (!c || !sum_wx || !sum_w) return fail(FIB_E_ARG, "NULL argument");
  if (c->nrep > 1) return refuse_batched_sum(c, "fib_weighted_sum");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  return reduce_weighted(c, var, c->phase, 1, sum_wx, sum_w);
}

// the reductions' grid: `parts` row blocks of the shard (1, or one per replica), about 4 blocks per SM in all
static dim3 reduce_grid(const fib_ctx* c, int parts) {
  return dim3(min(c->g.rows / parts, max(4 * c->sms / parts, 1)), parts);
}

// sum(w * x) and sum(w) over each of `parts` row blocks of the shard into sum_wx[p], sum_w[p]
static int reduce_weighted(fib_ctx* c, int var, const float* w, int parts, double* sum_wx, double* sum_w) {
  CU(cudaMemsetAsync(c->red, 0, 2 * parts * sizeof(double), c->stream));
  const PlaneRef pl = plane_of(c, var);
  wsum_kernel<<<reduce_grid(c, parts), 256, 0, c->stream>>>(pl.base, w, c->g, pl.halo, c->g.rows / parts, c->red);
  CU(cudaGetLastError());
  c->launches++;
  std::vector<double> h(2 * parts);
  CU(cudaMemcpyAsync(h.data(), c->red, h.size() * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  for (int p = 0; p < parts; ++p) {
    sum_wx[p] = h[2 * p];
    sum_w[p] = h[2 * p + 1];
  }
  return 0;
}

extern "C" int fib_count_nonfinite(fib_ctx* c, int var, uint64_t* count) {
  if (!c || !count) return fail(FIB_E_ARG, "ctx/count is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaMemsetAsync(c->red, 0, 2 * sizeof(double), c->stream));
  const PlaneRef pl = plane_of(c, var);
  nonfinite_kernel<<<min(c->g.rows, 4 * c->sms), 256, 0, c->stream>>>(
      pl.base, c->g, pl.halo, reinterpret_cast<unsigned long long*>(c->red));
  CU(cudaGetLastError());
  c->launches++;
  unsigned long long h = 0;
  CU(cudaMemcpyAsync(&h, c->red, sizeof h, cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  *count = h;
  return 0;
}

extern "C" int fib_set_weights(fib_ctx* c, int slot, const float* rows_host, int first_row, int nrows) {
  if (!c || !rows_host) return fail(FIB_E_ARG, "ctx/rows is NULL");
  if (slot < 0 || slot >= 4) return fail(FIB_E_ARG, "weight slot %d out of range 0..3", slot);
  if (first_row > c->g.row0 || first_row + nrows < c->g.row0 + c->g.rows)
    return fail(FIB_E_ARG, "weight rows [%d,%d) do not cover this shard", first_row, first_row + nrows);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  if (!c->weights[slot]) {
    CU(cudaMalloc(&c->weights[slot], c->halo_floats() * sizeof(float)));
    CU(cudaMemsetAsync(c->weights[slot], 0, c->halo_floats() * sizeof(float), c->stream));
  }
  CU(cudaMemcpy2DAsync(c->weights[slot] + c->g.pitch, c->g.pitch * sizeof(float),
                       rows_host + (size_t)(c->g.row0 - first_row) * c->g.W, c->g.W * sizeof(float),
                       c->g.W * sizeof(float), c->g.rows, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int fib_masked_sum(fib_ctx* c, int var, int slot, double* sum_wx, double* sum_w) {
  if (!c || !sum_wx || !sum_w) return fail(FIB_E_ARG, "NULL argument");
  if (c->nrep > 1) return refuse_batched_sum(c, "fib_masked_sum");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (slot < 0 || slot >= 4 || !c->weights[slot]) return fail(FIB_E_STATE, "weight slot %d is empty", slot);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  return reduce_weighted(c, var, c->weights[slot], 1, sum_wx, sum_w);
}

extern "C" int fib_replica_sums(fib_ctx* c, int var, int slot, double* sum_wx, double* sum_w, size_t n) {
  if (!c || !sum_wx || !sum_w) return fail(FIB_E_ARG, "NULL argument");
  if (n != (size_t)c->nrep) return fail(FIB_E_ARG, "fib_replica_sums: n=%zu, the context has %d replicas", n, c->nrep);
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (slot < -1 || slot >= 4) return fail(FIB_E_ARG, "weight slot %d out of range -1..3", slot);
  if (slot >= 0 && !c->weights[slot]) return fail(FIB_E_STATE, "weight slot %d is empty", slot);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  return reduce_weighted(c, var, slot < 0 ? c->phase : c->weights[slot], c->nrep, sum_wx, sum_w);
}

// The probe ring's records: `ncells` cells per record (1, or one per replica), `cap` records.  Arming either kind
// replaces the other; row < 0 disarms whichever is armed.
static int probe_watch(fib_ctx* c, int var, int row, int col, bool replicas, int ncells, unsigned long long cap) {
  DevGuard dg(c->cfg.device);
  if (c->pending) FLUSH(c);             // (an upload still in flight stays in flight: nothing is read here)
  CU(cudaStreamSynchronize(c->stream));
  drop_graphs(c);                       // the record node is part of the iteration graph
  if (row < 0) {
    c->watch_var = -1;
    return 0;
  }
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  // a replica watch: `row` local to a replica (the shard's own rows when unbatched: the replica is the grid)
  const int rh = replicas ? c->g.H / c->nrep : c->g.H;
  if (row >= rh || row < c->g.row0 || row >= c->g.row0 + c->g.rows || col < 0 || col >= c->g.W)
    return fail(FIB_E_ARG, "probe (%d,%d) is not in this shard%s", row, col, replicas ? " or replica" : "");
  c->watch_var = -1;
  {
    const int er = ensure_ring(c, (size_t)cap * ncells);
    if (er) return er;
  }
  CU(cudaMemsetAsync(c->ring_count, 0, sizeof(unsigned long long), c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->probe_ledger.clear();
  c->probe_armed_at = c->ode_iters;
  c->ring_fetched = 0;
  c->ring_cap = cap;
  c->watch_n = ncells;
  c->watch_replicas = replicas;
  c->watch_var = var;
  c->watch_row = row;
  c->watch_col = col;
  return 0;
}

extern "C" int fib_probe_watch(fib_ctx* c, int var, int row, int col) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  return probe_watch(c, var, row, col, false, 1, FIB_PROBE_RING);
}

// FIB_PROBE_RING records when unbatched: the layout the persistent kernel records into.  Batched: about 16 MiB of
// page-locked memory, at least 256 records.
extern "C" int fib_replica_probe_watch(fib_ctx* c, int var, int row, int col, size_t* capacity) {
  if (!c || !capacity) return fail(FIB_E_ARG, "ctx/capacity is NULL");
  const unsigned long long cap =
      c->nrep == 1 ? FIB_PROBE_RING : min((unsigned long long)FIB_PROBE_RING, max(256ull, (1ull << 22) / c->nrep));
  const int r = probe_watch(c, var, row, col, true, c->nrep, cap);
  if (!r) *capacity = (size_t)cap;
  return r;
}

// records [first, first + n) of a ring of `cap` slots as at most two contiguous pieces: copy(done, slot, len)
// copies `len` records from `slot` on to position `done` of the output
template <class Copy>
static int copy_ring(unsigned long long first, unsigned long long n, unsigned long long cap, Copy&& copy) {
  for (unsigned long long done = 0; done < n;) {
    const unsigned long long pos = (first + done) % cap, len = min(cap - pos, n - done);
    const int r = copy(done, pos, len);
    if (r) return r;
    done += len;
  }
  return 0;
}

static int probe_fetch(fib_ctx* c, bool replicas, float* out, size_t max, size_t* n) {
  if (!c || !n || (!out && max)) return fail(FIB_E_ARG, "NULL argument");
  *n = 0;
  if (c->watch_var < 0 || c->watch_replicas != replicas)
    return fail(FIB_E_STATE, "no probe is being watched (%s)", replicas ? "fib_replica_probe_watch" : "fib_probe_watch");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  // The records land in page-locked host memory.  Asked for fewer records than were made, wait only
  // for the launch that produced the last of them (the later ones keep the GPU busy meanwhile).
  const unsigned long long total = c->since(c->probe_armed_at);
  unsigned long long count = total;
  const int k = total - c->ring_fetched > max ? c->probe_ledger.covering(c->ring_fetched + max, total) : -1;
  if (k >= 0) {
    CU(cudaEventSynchronize(c->probe_ledger.ev[k]));
    count = c->probe_ledger.total[k];
  } else {
    CU(cudaStreamSynchronize(c->stream));
  }
  unsigned long long first = c->ring_fetched;
  if (count - first > c->ring_cap) first = count - c->ring_cap;      // the oldest were overwritten
  const unsigned long long take = min(count - first, (unsigned long long)max);
  const size_t rec = c->watch_n;
  copy_ring(first, take, c->ring_cap, [&](unsigned long long done, unsigned long long pos, unsigned long long len) {
    memcpy(out + done * rec, c->ring + pos * rec, len * rec * sizeof(float));
    return 0;
  });
  c->ring_fetched = first + take;
  *n = (size_t)take;
  return 0;
}

extern "C" int fib_probe_fetch(fib_ctx* c, float* out, size_t max, size_t* n) {
  return probe_fetch(c, false, out, max, n);
}

extern "C" int fib_replica_probe_fetch(fib_ctx* c, float* out, size_t max_records, size_t* n) {
  return probe_fetch(c, true, out, max_records, n);
}

// Activation maps: the sample s[0] is the current plane; the update runs after every ODE iteration from
// here on (record_observers, or inside the persistent kernel).  The iteration graphs are rebuilt with or
// without the update nodes.  A resume (`resume`) starts the counter at k and leaves the sample NaN for
// fib_activation_set to fill.
static int activation_arm(fib_ctx* c, float up, float down, bool resume, unsigned long long k) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (!isfinite(up) || !isfinite(down)) return fail(FIB_E_ARG, "activation levels must be finite (up %g, down %g)", up, down);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(wait_comm(c));
  CU(cudaStreamSynchronize(c->stream));
  drop_graphs(c);
  const size_t plane = c->plane_floats();
  if (!c->act_iter) CU(cudaMalloc(&c->act_iter, sizeof(unsigned long long)));
  if (!c->act_prev) CU(cudaMalloc(&c->act_prev, plane * sizeof(float)));
  if (!c->act_maps) CU(cudaMalloc(&c->act_maps, kActMaps * plane * sizeof(float)));   // last: armed from here
  if (resume)
    CU(cudaMemsetAsync(c->act_prev, 0xff, plane * sizeof(float), c->stream));         // all-ones bits: NaN
  else
    CU(cudaMemcpyAsync(c->act_prev, owned_rows(c, 0), plane * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
  activation_reset_kernel<<<c->sms * 4, 256, 0, c->stream>>>(c->act_maps, plane);
  CU(cudaGetLastError());
  c->launches++;
  CU(cudaMemcpyAsync(c->act_iter, &k, sizeof k, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  c->act_armed_at = c->ode_iters - k;     // since(act_armed_at) == k (modulo 2^64)
  c->act_up = up;
  c->act_down = down;
  return 0;
}
extern "C" int fib_activation_watch(fib_ctx* c, float up, float down) {
  return activation_arm(c, up, down, false, 0);
}
extern "C" int fib_activation_resume(fib_ctx* c, float up, float down, uint64_t k) {
  return activation_arm(c, up, down, true, k);
}

// map `map` (fib_act_map) of an armed context: a plane of the shard's row layout
static bool act_map_valid(int map) { return (map >= 0 && map < kActMaps) || map == FIB_ACT_SAMPLE; }
static float* act_plane(fib_ctx* c, int map) {
  return map == FIB_ACT_SAMPLE ? c->act_prev : c->act_maps + (size_t)map * c->plane_floats();
}

extern "C" int fib_activation_set(fib_ctx* c, int map, const float* host, size_t n) {
  if (!c || !host) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (!act_map_valid(map)) return fail(FIB_E_ARG, "unknown activation map %d", map);
  if (n != (size_t)c->g.rows * c->g.W)
    return fail(FIB_E_ARG, "fib_activation_set: n=%zu, expected rows*width=%zu", n, (size_t)c->g.rows * c->g.W);
  if (!c->act_maps) return fail(FIB_E_STATE, "no activation map is armed (fib_activation_resume)");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaMemcpy2DAsync(act_plane(c, map), c->g.pitch * sizeof(float), host, c->g.W * sizeof(float),
                       c->g.W * sizeof(float), c->g.rows, cudaMemcpyHostToDevice, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return check_persist_error(c);
}

extern "C" int fib_activation_stop(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaStreamSynchronize(c->stream));
  drop_graphs(c);
  CU(cudaFree(c->act_maps));
  CU(cudaFree(c->act_prev));
  CU(cudaFree(c->act_iter));
  c->act_maps = c->act_prev = nullptr;
  c->act_iter = nullptr;
  return check_persist_error(c);
}

extern "C" int fib_activation_get(fib_ctx* c, int map, float* host, size_t n) {
  if (!c || !host) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (!act_map_valid(map)) return fail(FIB_E_ARG, "unknown activation map %d", map);
  if (n != (size_t)c->g.rows * c->g.W)
    return fail(FIB_E_ARG, "fib_activation_get: n=%zu, expected rows*width=%zu", n, (size_t)c->g.rows * c->g.W);
  if (!c->act_maps) return fail(FIB_E_STATE, "no activation map is armed (fib_activation_watch)");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaMemcpy2DAsync(host, c->g.W * sizeof(float), act_plane(c, map),
                       c->g.pitch * sizeof(float), c->g.W * sizeof(float), c->g.rows, cudaMemcpyDeviceToHost,
                       c->stream));
  CU(cudaStreamSynchronize(c->stream));
  return check_persist_error(c);
}

// Frame recorder: a ring of strided frames in device memory.  Nothing joins the iteration graphs: the host
// counts iterations and gathers a frame after the recording ones (end_iterations), or hands the persistent kernel
// the first recording iteration of its launch (launch_persist_m).  A resume (`resume`) starts k at `k`, with the
// frames up to k counted as fetched and none taken now.
static int frames_arm(fib_ctx* c, int var, int first, int every, int stride, int capacity, bool resume,
                      unsigned long long k) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  if (first < 0 || every < 1 || stride < 1 || capacity < 1)
    return fail(FIB_E_ARG, "fib_frames_watch: need first >= 0, every >= 1, stride >= 1 and capacity >= 1 "
                "(got %d, %d, %d, %d)", first, every, stride, capacity);
  if (c->nrep > 1 && (c->g.H / c->nrep) % stride != 0)
    return fail(FIB_E_ARG, "fib_frames_watch: stride %d does not divide the replicas' height %d (each replica's "
                "frame rows start at its row 0)", stride, c->g.H / c->nrep);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaStreamSynchronize(c->stream));         // the old ring may still be written
  CU(cudaFree(c->frames));
  c->frames = nullptr;
  const int gr0 = (c->g.row0 + stride - 1) / stride * stride, row_end = c->g.row0 + c->g.rows;
  c->fr_rows = gr0 < row_end ? (row_end - 1 - gr0) / stride + 1 : 0;
  c->fr_cols = (c->g.W + stride - 1) / stride;
  c->fr_lr0 = gr0 - c->g.row0;
  c->fr_var = var;
  c->fr_first = first;
  c->fr_every = every;
  c->fr_stride = stride;
  c->fr_cap = capacity;
  c->fr_armed_at = c->ode_iters - k;      // since(fr_armed_at) == k (modulo 2^64)
  c->fr_fetched = resume ? c->frames_upto(k) : 0;
  const int er = c->frame_ledger.create();
  if (er) return er;
  c->frame_ledger.clear();
  const size_t bytes = max((size_t)capacity * c->frame_floats() * sizeof(float), sizeof(float));
  if (cudaMalloc(&c->frames, bytes) != cudaSuccess) {
    cudaGetLastError();
    c->frames = nullptr;
    return fail(FIB_E_CUDA, "fib_frames_watch: cannot allocate a ring of %d frames (%zu bytes)", capacity, bytes);
  }                                              // armed from here
  return first == 0 && !resume ? launch_frame(c, 0) : 0;
}
extern "C" int fib_frames_watch(fib_ctx* c, int var, int first, int every, int stride, int capacity) {
  return frames_arm(c, var, first, every, stride, capacity, false, 0);
}
extern "C" int fib_frames_resume(fib_ctx* c, int var, int first, int every, int stride, int capacity, uint64_t k) {
  return frames_arm(c, var, first, every, stride, capacity, true, k);
}

extern "C" int fib_frames_stop(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaFree(c->frames));
  c->frames = nullptr;
  return check_persist_error(c);
}

extern "C" int fib_frames_shape(const fib_ctx* c, int* rows, int* cols) {
  if (!c || !rows || !cols) return fail(FIB_E_ARG, "NULL argument");
  if (!c->frames) return fail(FIB_E_STATE, "no frame recorder is armed (fib_frames_watch)");
  *rows = c->fr_rows;
  *cols = c->fr_cols;
  return 0;
}

extern "C" int fib_frames_fetch(fib_ctx* c, float* host, uint64_t* iters, size_t max, size_t* n) {
  if (!c || !n || ((!host || !iters) && max)) return fail(FIB_E_ARG, "NULL argument");
  *n = 0;
  if (!c->frames) return fail(FIB_E_STATE, "no frame recorder is armed (fib_frames_watch)");
  DevGuard dg(c->cfg.device);
  // Iterations the persistent path has deferred are launched only when the frames already launched do not
  // satisfy the request: a caller that fetches one batch behind never cuts a batch.
  unsigned long long total = c->frames_recorded();
  if (total - c->fr_fetched < max) {
    FLUSH(c);
    total = c->frames_recorded();
  }
  unsigned long long first = c->fr_fetched;
  if (total - first > (unsigned long long)c->fr_cap) first = total - c->fr_cap;   // overwritten
  const unsigned long long take = min(total - first, (unsigned long long)max);
  if (take) {
    // wait for the earliest launch that covers the last frame taken, not for the launches queued behind it
    int k = c->frame_ledger.covering(first + take, total);
    if (k < 0) {                                 // no mark yet behind the launch that recorded them: one now
      const int r = c->frame_ledger.mark(c->stream, total);
      if (r) return r;
      k = c->frame_ledger.covering(first + take, total);
    }
    CU(cudaStreamWaitEvent(c->copy_stream, c->frame_ledger.ev[k], 0));
    // the frames taken cannot be overwritten by work already enqueued: that only writes frames < total, and
    // first >= total - capacity
    const size_t ff = c->frame_floats();
    const int r = copy_ring(first, take, c->fr_cap, [&](unsigned long long done, unsigned long long pos,
                                                        unsigned long long len) {
      if (ff)
        CU(cudaMemcpyAsync(host + done * ff, c->frames + pos * ff, len * ff * sizeof(float), cudaMemcpyDeviceToHost,
                           c->copy_stream));
      return 0;
    });
    if (r) return r;
    CU(cudaStreamSynchronize(c->copy_stream));
    for (unsigned long long i = 0; i < take; ++i) iters[i] = c->fr_first + (first + i) * c->fr_every;
  }
  c->fr_fetched = first + take;
  *n = (size_t)take;
  return check_persist_error(c);
}

// ------------------------------------------------------------------------------------------
// checkpoints: a stream-ordered staging copy of the owned rows, read out on ck_stream
// ------------------------------------------------------------------------------------------
extern "C" int fib_checkpoint_begin(fib_ctx* c, fib_checkpoint_info* info) {
  if (!c || !info) return fail(FIB_E_ARG, "ctx/info is NULL");
  if (info->struct_size != sizeof(fib_checkpoint_info))
    return fail(FIB_E_ARG, "fib_checkpoint_info.struct_size %u != %zu (ABI mismatch)", info->struct_size,
                sizeof(fib_checkpoint_info));
  if (c->ck) return fail(FIB_E_STATE, "a checkpoint is already in flight on this context (fib_checkpoint_end)");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  const size_t plane = (size_t)c->g.rows * c->g.W;
  const int parts = c->nvars + (c->act_maps ? 1 + kActMaps : 0);
  // stream-ordered: neither this allocation nor fib_checkpoint_end's release waits for the stepping
  cudaError_t e = cudaMallocAsync((void**)&c->ck, parts * plane * sizeof(float), c->stream);
  if (e != cudaSuccess) {
    cudaGetLastError();
    c->ck = nullptr;
    return fail(FIB_E_CUDA, "fib_checkpoint_begin: cannot allocate the staging copy of %d planes (%zu bytes): %s",
                parts, parts * plane * sizeof(float), cudaGetErrorString(e));
  }
  c->ck_parts = parts;
  for (int p = 0; p < parts && e == cudaSuccess; ++p) {
    const float* src = p < c->nvars ? owned_rows(c, p) : act_plane(c, p == c->nvars ? FIB_ACT_SAMPLE : p - c->nvars - 1);
    e = cudaMemcpy2DAsync(c->ck + p * plane, c->g.W * sizeof(float), src, c->g.pitch * sizeof(float),
                          c->g.W * sizeof(float), c->g.rows, cudaMemcpyDeviceToDevice, c->stream);
  }
  if (e == cudaSuccess) e = cudaEventRecord(c->ev_ck, c->stream);
  if (e != cudaSuccess) {
    cudaFreeAsync(c->ck, c->stream);
    c->ck = nullptr;
    return fail(FIB_E_CUDA, "fib_checkpoint_begin: staging copy failed: %s", cudaGetErrorString(e));
  }
  const fib_checkpoint_info z = {};
  *info = z;
  info->struct_size = sizeof(fib_checkpoint_info);
  info->nparts = parts;
  info->iterations = c->ode_iters;
  if (c->act_maps) {
    info->act_armed = 1;
    info->act_up = c->act_up;
    info->act_down = c->act_down;
    info->act_k = c->since(c->act_armed_at);
  }
  if (c->frames) {
    info->fr_armed = 1;
    info->fr_var = c->fr_var;
    info->fr_first = c->fr_first;
    info->fr_every = c->fr_every;
    info->fr_stride = c->fr_stride;
    info->fr_capacity = c->fr_cap;
    info->fr_k = c->since(c->fr_armed_at);
  }
  return 0;
}

// May run on another thread than the owner's: it touches only the staged copy, ck_stream and ev_ck, which the
// owner changes only in fib_checkpoint_begin / fib_checkpoint_end.
extern "C" int fib_checkpoint_read(fib_ctx* c, int part, int r0, int r1, float* host) {
  if (!c || !host) return fail(FIB_E_ARG, "ctx/host is NULL");
  if (!c->ck) return fail(FIB_E_STATE, "no checkpoint is in flight (fib_checkpoint_begin)");
  if (part < 0 || part >= c->ck_parts) return fail(FIB_E_ARG, "checkpoint part %d out of range (%d parts)", part, c->ck_parts);
  if (r0 < c->g.row0 || r1 > c->g.row0 + c->g.rows || r0 >= r1)
    return fail(FIB_E_ARG, "rows [%d,%d) not inside this shard [%d,%d)", r0, r1, c->g.row0, c->g.row0 + c->g.rows);
  DevGuard dg(c->cfg.device);
  const size_t W = c->g.W;
  CU(cudaStreamWaitEvent(c->ck_stream, c->ev_ck, 0));
  CU(cudaMemcpyAsync(host, c->ck + (size_t)part * c->g.rows * W + (size_t)(r0 - c->g.row0) * W,
                     (size_t)(r1 - r0) * W * sizeof(float), cudaMemcpyDeviceToHost, c->ck_stream));
  CU(cudaStreamSynchronize(c->ck_stream));
  return 0;
}

extern "C" int fib_checkpoint_end(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  if (!c->ck) return 0;
  DevGuard dg(c->cfg.device);
  // after the staging copy on `stream`; every read of it has returned
  CU(cudaFreeAsync(c->ck, c->stream));
  c->ck = nullptr;
  c->ck_parts = 0;
  return 0;
}

// count_below_kernel over each of `parts` row blocks of the shard (as reduce_weighted) into below[p], total[p]
static int reduce_count_below(fib_ctx* c, int var, float sub, float div, float cutoff, float w_min, int parts,
                              uint64_t* below, uint64_t* total) {
  CU(cudaMemsetAsync(c->red, 0, 2 * parts * sizeof(double), c->stream));
  const PlaneRef pl = plane_of(c, var);
  count_below_kernel<<<reduce_grid(c, parts), 256, 0, c->stream>>>(
      pl.base, c->phase, c->g, pl.halo, c->g.rows / parts, sub, div, cutoff, w_min,
      reinterpret_cast<unsigned long long*>(c->red));
  CU(cudaGetLastError());
  c->launches++;
  std::vector<unsigned long long> h(2 * parts);
  CU(cudaMemcpyAsync(h.data(), c->red, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  CU(cudaStreamSynchronize(c->stream));
  for (int p = 0; p < parts; ++p) {
    below[p] = h[2 * p];
    total[p] = h[2 * p + 1];
  }
  return 0;
}

extern "C" int fib_count_below(fib_ctx* c, int var, float sub, float div, float cutoff, float w_min,
                               uint64_t* below, uint64_t* total) {
  if (!c || !below || !total) return fail(FIB_E_ARG, "NULL argument");
  if (c->nrep > 1) return refuse_batched_sum(c, "fib_count_below");
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  return reduce_count_below(c, var, sub, div, cutoff, w_min, 1, below, total);
}

extern "C" int fib_replica_count_below(fib_ctx* c, int var, float sub, float div, float cutoff, float w_min,
                                       uint64_t* below, uint64_t* total, size_t n) {
  if (!c || !below || !total) return fail(FIB_E_ARG, "NULL argument");
  if (n != (size_t)c->nrep)
    return fail(FIB_E_ARG, "fib_replica_count_below: n=%zu, the context has %d replicas", n, c->nrep);
  if (var < 0 || var >= c->nvars) return fail(FIB_E_ARG, "state variable %d out of range", var);
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  return reduce_count_below(c, var, sub, div, cutoff, w_min, c->nrep, below, total);
}

// ------------------------------------------------------------------------------------------
// op-level entry points (eager, dense host planes)
// ------------------------------------------------------------------------------------------
struct DevBuf {
  float* p = nullptr;
  ~DevBuf() { cudaFree(p); }
};
static int op_device(int device) {
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(FIB_E_CUDA, "device %d not available (%d CUDA devices)", device, ndev);
  return 0;
}

extern "C" int fib_op_enforce_boundary(int device, const float* x, int h, int w, float* out) {
  if (!x || !out) return fail(FIB_E_ARG, "NULL argument");
  if (h < 3 || w < 3) return fail(FIB_E_ARG, "plane %dx%d too small: the boundary needs >= 3x3", h, w);
  if (h > 65535) return fail(FIB_E_ARG, "op-level planes are limited to 65535 rows");
  int r = op_device(device);
  if (r) return r;
  DevGuard dg(device);
  const size_t n = (size_t)h * w;
  DevBuf a, b;
  CU(cudaMalloc(&a.p, n * sizeof(float)));
  CU(cudaMalloc(&b.p, n * sizeof(float)));
  CU(cudaMemcpy(a.p, x, n * sizeof(float), cudaMemcpyHostToDevice));
  op_enforce_kernel<<<dim3((w + 127) / 128, h), 128>>>(a.p, h, w, b.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, b.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int fib_op_laplace(int device, const float* x, const float* phase, int h, int w, int mode, float* out) {
  if (!x || !out) return fail(FIB_E_ARG, "NULL argument");
  if (mode < 0 || mode > 2) return fail(FIB_E_ARG, "unknown mode %d", mode);
  if (mode == 2 && !phase) return fail(FIB_E_ARG, "mode 2 (phase term) needs a phase field");
  if (h < 3 || w < 3) return fail(FIB_E_ARG, "plane %dx%d too small", h, w);
  if (h > 65535) return fail(FIB_E_ARG, "op-level planes are limited to 65535 rows");
  int r = op_device(device);
  if (r) return r;
  DevGuard dg(device);
  const size_t n = (size_t)h * w;
  DevBuf a, b, ph;
  CU(cudaMalloc(&a.p, n * sizeof(float)));
  CU(cudaMalloc(&b.p, n * sizeof(float)));
  CU(cudaMemcpy(a.p, x, n * sizeof(float), cudaMemcpyHostToDevice));
  if (phase) {
    CU(cudaMalloc(&ph.p, n * sizeof(float)));
    CU(cudaMemcpy(ph.p, phase, n * sizeof(float), cudaMemcpyHostToDevice));
  }
  op_laplace_kernel<<<dim3((w + 127) / 128, h), 128>>>(a.p, ph.p, h, w, mode, b.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, b.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

extern "C" int fib_op_rush_larsen(int device, const float* g, const float* g_inf, const float* tau, size_t n,
                                  float dt, int strict, float* out) {
  if (!g || !g_inf || !tau || !out) return fail(FIB_E_ARG, "NULL argument");
  if (n == 0) return 0;
  int r = op_device(device);
  if (r) return r;
  DevGuard dg(device);
  DevBuf a, b, t, o;
  for (DevBuf* d : {&a, &b, &t, &o}) CU(cudaMalloc(&d->p, n * sizeof(float)));
  CU(cudaMemcpy(a.p, g, n * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(b.p, g_inf, n * sizeof(float), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(t.p, tau, n * sizeof(float), cudaMemcpyHostToDevice));
  op_rush_larsen_kernel<<<(unsigned)((n + 255) / 256), 256>>>(a.p, b.p, t.p, n, -dt, strict, o.p);
  CU(cudaGetLastError());
  CU(cudaMemcpy(out, o.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  return 0;
}

// ------------------------------------------------------------------------------------------
// sync / timing
// ------------------------------------------------------------------------------------------
extern "C" int fib_sync(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaStreamSynchronize(c->stream));
  CU(cudaStreamSynchronize(c->comm_stream));
  CU(cudaStreamSynchronize(c->copy_stream));
  c->snap_pending = false;
  return check_persist_error(c);
}
extern "C" int fib_flush(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  return 0;
}
extern "C" int fib_timer_start(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  CU(cudaEventRecord(c->ev_start, c->stream));
  return 0;
}
extern "C" int fib_timer_stop(fib_ctx* c) {
  if (!c) return fail(FIB_E_ARG, "ctx is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  if (c->comm_pending) CU(cudaStreamWaitEvent(c->stream, c->ev_comm, 0));
  CU(cudaEventRecord(c->ev_stop, c->stream));
  return 0;
}
extern "C" int fib_timer_ms(fib_ctx* c, float* ms) {
  if (!c || !ms) return fail(FIB_E_ARG, "ctx/ms is NULL");
  DevGuard dg(c->cfg.device);
  CU(cudaEventSynchronize(c->ev_stop));
  CU(cudaEventElapsedTime(ms, c->ev_start, c->ev_stop));
  return 0;
}
extern "C" int fib_launch_count(const fib_ctx* c, uint64_t* kernels) {
  if (!c || !kernels) return fail(FIB_E_ARG, "ctx/kernels is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(const_cast<fib_ctx*>(c));       // deferred iterations count once they are launched
  *kernels = c->launches;
  return 0;
}
extern "C" int fib_stream(const fib_ctx* c, void** cuda_stream) {
  if (!c || !cuda_stream) return fail(FIB_E_ARG, "ctx/out is NULL");
  DevGuard dg(c->cfg.device);
  FLUSH(const_cast<fib_ctx*>(c));
  *cuda_stream = (void*)c->stream;
  return 0;
}

// ------------------------------------------------------------------------------------------
// multi-process sharding
// ------------------------------------------------------------------------------------------
extern "C" int fib_comm_unique_id(void* out128) {
  if (!out128) return fail(FIB_E_ARG, "out128 is NULL");
  int r = nccl_load();
  if (r) return r;
  NC(g_nccl.GetUniqueId(out128));
  return 0;
}

extern "C" int fib_comm_init(fib_ctx* c, int nranks, int rank, const void* id128) {
  if (!c || !id128) return fail(FIB_E_ARG, "ctx/id is NULL");
  if (nranks < 1 || rank < 0 || rank >= nranks) return fail(FIB_E_ARG, "bad rank %d of %d", rank, nranks);
  if (c->nrep > 1) return fail(FIB_E_ARG, "fib_comm_init: a batched context (%d replicas) cannot be sharded", c->nrep);
  if (c->comm) return fail(FIB_E_STATE, "communicator already initialised");
  if (nranks == 1) return 0;   // a single shard needs no communicator
  if ((rank == 0) != c->top_is_border() || (rank == nranks - 1) != c->bottom_is_border())
    return fail(FIB_E_ARG, "rank %d of %d does not match shard rows [%d,%d) of %d", rank, nranks,
                c->g.row0, c->g.row0 + c->g.rows, c->g.H);
  int r = nccl_load();
  if (r) return r;
  DevGuard dg(c->cfg.device);
  FLUSH(c);
  Uid uid;
  memcpy(uid.bytes, id128, sizeof uid.bytes);
  NC(g_nccl.CommInitRank(&c->comm, nranks, uid, rank));
  c->nranks = nranks;
  c->rank = rank;
  c->halo_dirty = true;
  c->persist = 0;          // the persistent kernel is for unsharded grids
  // Bring up the connections of every exchange pattern now, outside anybody's timed region: both seams in one
  // group (the per-step exchange) and each seam on its own (fib_step_behind_upload).  The halo rows this moves
  // are refreshed before their first use (halo_dirty).  Collective like the rest of this call; the one-seam
  // exchanges pair rank r's lower seam with rank r+1's upper one, a chain that starts at rank 0.
  int w = nccl_exchange(c, c->cur, c->stream, kSeamBoth);
  if (!w) w = nccl_exchange(c, c->cur, c->stream, kSeamUp);
  if (!w) w = nccl_exchange(c, c->cur, c->stream, kSeamDown);
  if (w) return w;
  CU(cudaStreamSynchronize(c->stream));
  return 0;
}
