/*
 * fib_b200.h -- C ABI of libfibb200.so: a B200-native (sm_100a) explicit time-stepper for
 * 2-D cardiac monodomain models (Fenton 4v, Beeler-Reuter, Courtemanche).
 *
 * The reference (siravan/fib_tf) has NO native boundary: its hot path is a TensorFlow-1.x
 * graph executed once per run() iteration by tf.Session.run (ionic.py:202-204).  This header
 * is the boundary a maintainer binds instead of TensorFlow; every entry point names the
 * reference interface (file:line under /root/reference) whose device work it replaces.
 * The Python side (fib_tf_b200/_capi.py) binds exactly these symbols with ctypes.
 *
 * Conventions
 *   - every function returns 0 on success and a negative fib_status on error; the message
 *     is available from fib_last_error() (thread-local, valid until the next failing call);
 *   - host pointers are borrowed for the duration of the call only; planes are row-major
 *     [rows][width] fp32 with no padding on the host side;
 *   - all device work is ENQUEUE-ONLY on the context's stream unless stated "synchronous"
 *     (the reference's run() generator hands control back to user code between iterations,
 *     ionic.py:202-204, so the only sync points are state reads, probes and fib_sync);
 *   - one context is not thread-safe (single caller); different contexts are independent;
 *   - there is no CPU fallback: without a CUDA device fib_create fails with FIB_E_CUDA.
 */
#ifndef FIB_B200_H_
#define FIB_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FIB_ABI_VERSION 3

typedef struct fib_ctx fib_ctx;

typedef enum {
  FIB_OK = 0,
  FIB_E_ARG = -1,     /* bad argument / bad ordering of calls              */
  FIB_E_CUDA = -2,    /* CUDA runtime error (message holds the CUDA string) */
  FIB_E_NCCL = -3,    /* NCCL error or libnccl not loadable                 */
  FIB_E_STATE = -4    /* context not in a state that allows the call        */
} fib_status;

/* model ids -- the reference's model classes */
typedef enum {
  FIB_FENTON4V = 0,     /* fenton.py:31   Fenton4v,  4 state planes U V W S            */
  FIB_BR = 1,           /* br.py:30       BeelerReuter, 8 planes V C M H J D F XI     */
  FIB_COURT = 2,        /* court.py:30    Courtemanche, 21 planes, fast/slow split    */
  FIB_COURT_ULTRA = 3   /* court_ultra.py:32  all states every step (+ optional _us_) */
} fib_model;

/* flag bits of fib_config.flags */
#define FIB_F_CHEBY      0x01u  /* BR: degree-8 polynomial gates   (br.py:207-252, config 'cheby') */
#define FIB_F_SKIP       0x02u  /* BR: multi-rate slow gates        (br.py:96-107,  config 'skip')  */
#define FIB_F_LUT        0x04u  /* Courtemanche: V-only intermediates from the 150x30 table,
                                   truncating lookup i=int(V+100) clamped (courtemanche.h:354-357) */
#define FIB_F_ULTRA_SLOW 0x08u  /* court_ultra.py:81-82,198-199,221-222: 22nd state '_us_'         */
#define FIB_F_NO_CHRONIC 0x10u  /* Courtemanche: chronic-AF remodelling OFF (court.py:41 sets it ON) */
#define FIB_F_NO_GRAPH   0x20u  /* launch kernels directly instead of replaying a CUDA graph         */
#define FIB_F_NO_CLIP    0x40u  /* Courtemanche: no [1e-5, 0.99999] clip of the Rush-Larsen gates, as in
                                   the native integrate_gate (courtemanche.h:287-292); court.py clips   */

#define FIB_F_CHEBY_STRICT 0x80u /* BR + FIB_F_CHEBY: evaluate the polynomial gates in the reference's own
                                   operation order (fp32 division for x, S_i recurrence, left-to-right
                                   d_i*S_i sum, unfused Rush-Larsen with IEEE division and libm expm1f;
                                   br.py:215,289-301,327-331, ionic.py:115-123) instead of Horner's scheme */
#define FIB_F_NO_PERSIST 0x100u /* never use the persistent on-chip kernel (fib_persist.cuh) for small grids */

typedef struct {
  uint32_t struct_size;      /* = sizeof(fib_config), for ABI evolution                              */
  int32_t  model;            /* fib_model                                                            */
  int32_t  height, width;    /* GLOBAL grid, config 'height'/'width' (ionic.py:35-37); both >= 3     */
  double   dt;               /* config 'dt'   (ms); kept double: the reference folds diff*dt and dt*n
                                in Python doubles before rounding to fp32 (fenton.py:103, br.py:197) */
  double   diff;             /* config 'diff'                                                        */
  uint32_t flags;            /* FIB_F_*                                                              */
  int32_t  device;           /* CUDA device ordinal                                                  */
  int32_t  row0, rows;       /* this shard = global rows [row0, row0+rows); rows == 0 -> whole grid   */
  int32_t  steps_per_launch; /* temporal blocking: time steps per kernel launch.  0/1 = one; 2 = two
                                (Fenton 4v only, width % 4 == 0; results are
                                bit-identical to one step per launch; shards exchange two halo rows
                                of every plane per launch).  Must divide dt_per_step (SURVEY fact 4) */
  int32_t  reserved[6];
} fib_config;

/* ops of fib_step -- the reference's session ops */
typedef enum {
  FIB_OP_ODE = 0,   /* model._ode_op: one run() iteration = dt_per_step time steps
                       (fenton.py:135-145: 10, br.py:96-120: 5, court.py:91-102: 1)                  */
  FIB_OP_SLOW = 1   /* model._ops['slow'] (court.py:103): the 17 slow states, step 10*dt, evaluated
                       on the CURRENT state; a no-op for every other model (court_ultra.py:108)      */
} fib_op;

/* table ids of fib_set_table / fib_get_table */
typedef enum {
  FIB_TABLE_BR_CHEBY = 0,   /* float[12][9]: rows 2g = inf, 2g+1 = tau of gate g in (xi,m,h,j,d,f);
                               coefficients d_i of the scaled monomials S_i (br.py:303-331)          */
  FIB_TABLE_COURT_LUT = 1   /* float[150][30]: courtemanche.h:105-134 column order, row i = V i-100 mV */
} fib_table;

/* ---- library ----------------------------------------------------------------------- */
int         fib_version(void);            /* FIB_ABI_VERSION of the loaded library                   */
const char *fib_last_error(void);
int         fib_device_count(int *count); /* cudaGetDeviceCount; FIB_E_CUDA if no driver/device       */

/* ---- life cycle: replaces tf.Session()/tf.Variable creation in define() ---------------
 * (fenton.py:126-131, br.py:85-94, court.py:85-89) */
int fib_create(const fib_config *cfg, fib_ctx **out);
int fib_destroy(fib_ctx *ctx);

/* ---- model description ----------------------------------------------------------------- */
int         fib_num_vars(const fib_ctx *ctx);               /* 4 / 8 / 21 / 21|22                   */
const char *fib_var_name(const fib_ctx *ctx, int var);      /* reference names: "U","V",..,"_Na_i_"  */
int         fib_var_index(const fib_ctx *ctx, const char *name);   /* <0 if unknown                 */
int         fib_dt_per_step(const fib_ctx *ctx);            /* model.dt_per_step                     */

/* ---- state I/O: replaces tf.Variable(initial) and Variable.eval() ----------------------
 * (fenton.py:128-131,152-153; br.py:86-93,341; court.py:89; ionic.py:226-229).
 * `n` must equal rows*width of THIS shard.  Synchronous. */
int fib_set_state(fib_ctx *ctx, int var, const float *host, size_t n);
int fib_get_state(fib_ctx *ctx, int var, float *host, size_t n);
/* sub-rectangle read / write of the local shard (frame grabs, strided probes, strip-wise upload
 * of grids too large to stage on the host in one piece); global coordinates, dense host block */
int fib_get_rect(fib_ctx *ctx, int var, int r0, int r1, int c0, int c1, float *host);
int fib_set_rect(fib_ctx *ctx, int var, int r0, int r1, int c0, int c1, const float *host);
/* enqueue-only variant of fib_set_rect: `host_pinned` (page-locked, fib_host_alloc) must stay valid and
 * unchanged until the next fib_sync / synchronous call; the copy is ordered before every later call on
 * this context.  Lets a caller stream a large initial state strip by strip without a round trip each.
 * Pipelined upload: full-width blocks of a large unsharded grid, enqueued top to bottom with every plane
 * of a block before the next block, are copied on a stream of their own, and ODE iterations stepped
 * before anything reads or writes the state run block by block BEHIND the copies -- launch l of the block
 * ending at row a covers rows [a' - h(l+1), a - h(l+1)) (a' = end of the block above, h = time steps per
 * launch), so every launch reads only rows already at its time level.  Same arithmetic on the same
 * values: the result is bit-identical to copying everything first (tests/test_gpu_pipelined_upload.py);
 * the 16 GiB upload of the 32768^2 benchmark state hides behind the first ten iterations. */
int fib_set_rect_async(fib_ctx *ctx, int var, int r0, int r1, int c0, int c1, const float *host_pinned);

/* asynchronous frame grab (the cube.npy writer of fenton.py:179-187 without stalling the stepper):
 * fib_snapshot_begin enqueues a device-side copy of the plane (ordered after everything already
 * enqueued) and its transfer to `host_pinned` (page-locked, rows*width floats) on a separate copy
 * stream, then returns; later fib_step calls overlap with the transfer.  fib_snapshot_wait blocks
 * until the host buffer is complete.  One snapshot may be in flight per context. */
int fib_snapshot_begin(fib_ctx *ctx, int var, float *host_pinned, size_t n);
int fib_snapshot_wait(fib_ctx *ctx);

/* ---- phase field: replaces self.phi = tf.Variable(self.phase) (ionic.py:55-58) ---------
 * `rows_host` holds global rows [first_row, first_row+nrows) of the [H][W] phase field and must
 * cover this shard plus one row either side -- two rows with steps_per_launch = 2 -- clipped to the
 * grid (passing the whole field with first_row = 0 always works).  NULL removes the field. */
int fib_set_phase(fib_ctx *ctx, const float *rows_host, int first_row, int nrows);

/* ---- tables ------------------------------------------------------------------------------ */
int fib_set_table(fib_ctx *ctx, int table, const float *data, size_t n);
int fib_get_table(fib_ctx *ctx, int table, float *data, size_t n);
/* Courtemanche: fill the LUT on the device by evaluating the kernel's own calc_inter at
 * V = i-100 mV, i = 0..149 (courtemanche.h:473-479 init_table). */
int fib_build_lut(fib_ctx *ctx);
/* Courtemanche calc_inter(V) (court.py:273-429 / courtemanche.h:159-285) for n voltages:
 * out[n][32]; columns 0..29 in courtemanche.h:105-134 order, 30 = us_infinity, 31 = tau_us
 * (court_ultra.py:445-450).  Synchronous.  Backs Courtemanche.calc_inter(V, np) / _Inter. */
int fib_court_inter(fib_ctx *ctx, const float *v_host, size_t n, float *out_host);

/* ---- the hot path: replaces sess.run(self.ode_op(i)) (ionic.py:203) and
 * fire_op('slow') (ionic.py:165-169, court.py:103).  Enqueues n_iter iterations.
 * On the persistent on-chip path (small unsharded 4v / BR grids) the iterations are only COUNTED
 * here and launched, up to 64 per launch, by the next call on this context that observes or changes
 * anything (state / probe / reduction reads, writes, fib_sync, the timers, fib_stream, fib_flush) or
 * when 64 have accumulated -- results are the same, a loop of fib_step(ctx, op, 1) just costs one
 * launch per 64 iterations.  Work enqueued on fib_stream() by the caller is ordered after everything
 * stepped before that fib_stream() / fib_flush() call. */
int fib_step(fib_ctx *ctx, int op, int n_iter);
/* launch whatever fib_step has deferred (enqueue only, no synchronisation) */
int fib_flush(fib_ctx *ctx);
/* Pipelined uploads on NCCL shards.  An unsharded context steps behind its upload by itself (fib_set_rect_async);
 * on NCCL shards the skewed schedule needs its own exchange pattern, so it is explicit and COLLECTIVE: every rank
 * uploads its shard block by block -- even ranks top to bottom, odd ranks bottom to top, so that both shards of a
 * seam either begin or end there -- then all ranks agree (host side, e.g. an all-reduce of fib_upload_state's
 * answers: open, complete, direction = +1 / -1, the number of iterations that fit) and call
 * fib_step_behind_upload with the same n_iter.  First blocks advance in lock step with the neighbour that also
 * begins at that seam, exchanging the seam's halo rows after every launch; last blocks likewise; the blocks in
 * between run behind their copies without any exchange.  Without the explicit call a sharded context simply
 * waits for its upload (fib_step).  Bit-identical to upload-then-step (tests/dist_parity.py). */
int fib_upload_state(const fib_ctx *ctx, int *open, int *complete, int *direction, int *max_iters);
int fib_step_behind_upload(fib_ctx *ctx, int n_iter);
/* lock-step stepping of several shards living in ONE process (row-adjacent, ctxs[0] on top):
 * halo rows are exchanged device-to-device after every time step.  Used to emulate the
 * multi-GPU decomposition on one device and for single-process multi-GPU. */
int fib_step_group(fib_ctx **ctxs, int n, int op, int n_iter);

/* name of the step-kernel flavour (model, cells per thread, marching depth, phase flag) launched last
 * by fib_step / fib_step_group on this thread: lets tests prove which instantiation they compared. */
int fib_last_kernel(char *buf, size_t n);

/* ---- stimulus: replaces pot().assign(tf.maximum(pot(), s)) (ionic.py:144-163) -----------
 * X := max(X, inside [r0,r1)x[c0,c1) ? value : floor_v) over the whole plane, GLOBAL coords. */
int fib_stimulate(fib_ctx *ctx, int var, int r0, int r1, int c0, int c1, float value,
                  float floor_v);

/* ---- probes: replaces Variable[r,c] reads (ionic.py:216, court.py:109-110) --------------
 * Synchronous.  FIB_E_ARG if (row,col) is not in this shard. */
int fib_probe(fib_ctx *ctx, int var, int row, int col, float *out);
/* weighted mean of a plane over this shard: sum(w*x), sum(w) (w = phase field, or 1 if none):
 * backs np.average(x, weights=phase) in court_ultra.py:466-480.  Synchronous. */
int fib_weighted_sum(fib_ctx *ctx, int var, double *sum_wx, double *sum_w);
/* failure detection: number of non-finite cells of a plane in this shard (the reference only has a
 * commented-out NaN check, ionic.py:199,208-212).  Synchronous. */
int fib_count_nonfinite(fib_ctx *ctx, int var, uint64_t *count);
/* user weight planes (pseudo-electrogram masks, egm.py:5-12,44-47: np.mean(image * mask)):
 * fib_set_weights uploads global rows [first_row, first_row+nrows) of an [H][W] mask into `slot`
 * (0..3; must cover this shard); fib_masked_sum returns sum(mask*x) and sum(mask) over the shard. */
int fib_set_weights(fib_ctx *ctx, int slot, const float *rows_host, int first_row, int nrows);
int fib_masked_sum(fib_ctx *ctx, int var, int slot, double *sum_wx, double *sum_w);

/* device-side observers (SURVEY 8f1), so that a headless run never moves a frame to the host:
 * fib_probe_watch registers ONE cell (the cycle-length probe image[20, W//2] of ionic.py:216-224; global
 * coordinates, must lie in this shard); from then on every fib_step iteration appends the cell's value to
 * a device ring buffer (inside the iteration's CUDA graph: no host round trip).  fib_probe_fetch copies
 * the values recorded since the last fetch (oldest first, at most `max`) and returns their number in *n;
 * synchronous.  More than FIB_PROBE_RING unfetched values: the oldest are lost, *n reports what is left.
 * row < 0 removes the watch. */
#define FIB_PROBE_RING 4096
int fib_probe_watch(fib_ctx *ctx, int var, int row, int col);
int fib_probe_fetch(fib_ctx *ctx, float *out, size_t max, size_t *n);
/* excitable fraction rho of court_ultra.py:504-509, np.sum(image[phase > w_min] < cutoff) /
 * np.sum(phase > w_min) with image = (x - sub) / div: *below = cells with weight > w_min and image <
 * cutoff, *total = cells with weight > w_min (weight = phase field, 1 if none).  Synchronous. */
int fib_count_below(fib_ctx *ctx, int var, float sub, float div, float cutoff, float w_min,
                    uint64_t *below, uint64_t *total);

/* activation maps (SURVEY 8f1): the activation-time (LAT), repolarisation and cycle-length maps of the whole
 * shard, recorded on the device while stepping, so that APD, cycle length and conduction velocity need no
 * frame on the host.  A map watches the DIFFUSING variable (U of 4v, V of BR / Courtemanche).
 *   samples  s[0] = the plane when fib_activation_watch is called; s[k] (k >= 1) = the plane at the end of
 *            the k-th FIB_OP_ODE iteration enqueued since, taken before anything the caller does between
 *            iterations (fib_stimulate, fib_set_*): a host write shows up in the next sample.  FIB_OP_SLOW
 *            does not write the variable and takes no sample.
 *   events   activation in iteration k:      s[k-1] < up <= s[k],   t = (k-1) + (up - s[k-1]) / (s[k] - s[k-1])
 *            repolarisation in iteration k:  s[k-1] >= down > s[k], t = (k-1) + (s[k-1] - down) / (s[k-1] - s[k])
 *            the event rule of tests/test_spiral_statistics.py events(), in fp32 with one rounding per
 *            operation (no contraction); a NaN sample produces no event.
 *   times    in iterations since arming, fp32.  Iteration indices are exact up to 2^24; the resolution of the
 *            fraction shrinks with k (one ulp of t is ~0.008 iteration at k = 10^5).
 *   maps     FIRST: first activation; LAST: last activation; PREV: the activation before LAST; REPOL: last
 *            repolarisation -- NaN while empty; COUNT: number of activations, as a float.  On an activation
 *            PREV := LAST, LAST := t, COUNT += 1 and FIRST := t if it is NaN; on a repolarisation REPOL := t.
 * Cost: 12 bytes per cell per iteration (the plane and the last sample read, the sample written), plus the
 * map planes at cells with an event.  An armed map keeps fib_set_rect_async blocks out of the pipelined
 * upload (they are copied in order instead).
 * fib_activation_watch arms the map, or re-arms it: everything is reset and s[0] re-taken; FIB_E_ARG if a
 * level is not finite.  fib_activation_stop disarms it and frees the planes.  fib_activation_get copies map
 * `map` (fib_act_map) of this shard, rows*width floats; synchronous; FIB_E_STATE without a watch. */
typedef enum {
  FIB_ACT_FIRST = 0,
  FIB_ACT_LAST = 1,
  FIB_ACT_PREV = 2,
  FIB_ACT_REPOL = 3,
  FIB_ACT_COUNT = 4
} fib_act_map;
int fib_activation_watch(fib_ctx *ctx, float up, float down);
int fib_activation_stop(fib_ctx *ctx);
int fib_activation_get(fib_ctx *ctx, int map, float *host, size_t n);

/* ---- op-level entry points of IonicModel's helpers on dense host planes [h][w] (eager; used by the
 * drop-in IonicModel.enforce_boundary / laplace / phase_field / rush_larsen and by the parity tests that
 * check the stencil arithmetic in isolation).  Synchronous; `device` = CUDA ordinal.
 *   fib_op_enforce_boundary  ionic.py:107-113  border ring := SYMMETRIC pad of the interior
 *   fib_op_laplace           ionic.py:44-60    mode 0: REFLECT-pad `x` by one cell, 9-point stencil
 *                                              (+ phase term ionic.py:70-81 when `phase` != NULL);
 *                                              mode 1: the step kernels' collapsed index map on a RAW
 *                                              plane, = laplace(enforce_boundary(x));
 *                                              mode 2: only the phase-field term (ionic.py:70-81)
 *   fib_op_rush_larsen       ionic.py:115-123  strict != 0: IEEE division, libm expm1f, unfused */
int fib_op_enforce_boundary(int device, const float *x, int h, int w, float *out);
int fib_op_laplace(int device, const float *x, const float *phase, int h, int w, int mode, float *out);
int fib_op_rush_larsen(int device, const float *g, const float *g_inf, const float *tau, size_t n,
                       float dt, int strict, float *out);

/* ---- sync / timing / accounting ------------------------------------------------------------ */
int fib_sync(fib_ctx *ctx);
int fib_timer_start(fib_ctx *ctx);            /* cudaEventRecord on the context's stream        */
int fib_timer_stop(fib_ctx *ctx);
int fib_timer_ms(fib_ctx *ctx, float *ms);    /* synchronises on the stop event                 */
int fib_launch_count(const fib_ctx *ctx, uint64_t *kernels);  /* kernels launched so far        */
int fib_stream(const fib_ctx *ctx, void **cuda_stream);       /* the cudaStream_t, for interop   */

/* ---- pinned host memory for the host<->device legs ---------------------------------------- */
int fib_host_alloc(size_t bytes, void **out);
int fib_host_free(void *p);

/* ---- multi-process row sharding: one process per GPU, halo rows over NCCL ----------------
 * fib_comm_unique_id writes a 128-byte ncclUniqueId (rank 0 calls it; the bytes are
 * broadcast by the host side, e.g. torch.distributed).  After fib_comm_init, fib_step
 * exchanges one halo row of the diffusing variable with rank-1 / rank+1 after every time
 * step (ncclSend/ncclRecv on a side stream, overlapped with the interior rows). */
int fib_comm_unique_id(void *out128);
int fib_comm_init(fib_ctx *ctx, int nranks, int rank, const void *id128);

#ifdef __cplusplus
}
#endif
#endif /* FIB_B200_H_ */
