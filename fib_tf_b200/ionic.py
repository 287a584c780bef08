"""
fib_tf_b200.ionic -- host-side mirror of the reference's IonicModel base class (ionic.py:30-307).

Same public surface (config dict -> attributes, add_hole_to_phase_field, define,
add_pace_op / fire_op, the run() generator, millisecond_to_step, image, pot, ode_op,
jit_scope / context-manager fallback), so the reference's driver loops

    model = Fenton4v(config); model.add_hole_to_phase_field(256, 256, 30); model.define()
    model.add_pace_op('s2', 'luq', 1.0)
    for i in model.run(im):
        if i == s2: model.fire_op('s2')

run unchanged -- but every device operation goes to libfibb200.so (hand-written sm_100a CUDA
kernels behind the C ABI in include/fib_b200.h) instead of a TensorFlow session.  NumPy is used
for set-up only (initial conditions, phase field, Chebyshev fit), exactly where the reference
uses it.  There is no TensorFlow, no XLA and no CPU fallback.

Extra, optional config keys (all default to the reference's behaviour):
    device       CUDA device ordinal (default: LOCAL_RANK when distributed, else 0)
    graph        replay one CUDA graph per run() iteration (default True)
    persist      small unsharded 4v / BR grids (W <= 512, the reference's 512^2 configurations): run an
                 iteration as ONE persistent on-chip kernel, bit-identical to one launch per step
                 (default True; csrc/fib_persist.cuh)
    distributed  row-shard the grid over the torch.distributed world (default False)
    lut          Courtemanche: V-only intermediates from the 150x30 table (default False)
    probe_batch  headless runs with a cl_observer: the cycle-length probe is recorded on the device
                 every iteration and read back `probe_batch` iterations at a time, one batch behind
                 the stepping so the device never idles (default 64; the observer is then called up
                 to twice that many iterations late, with the reference's arguments; 1 = read it
                 back every iteration like the reference)

    replicas     B > 1: step B independent grids of height x width together, one launch per time step for all
                 of them (include/fib_b200.h, Replicas; default 1).  Each replica has its own state, holes
                 (add_hole_to_phase_field(replica=)), stimuli (fire_op / pace with replica=) and `diff`: config
                 'diff' may be a sequence of B floats.  Reads (image(), pot().eval(), _State[n].eval(),
                 activation_maps(), frames()) gain a leading replica axis; assign() takes [H, W] or [B, H, W].
                 Not with `distributed`, run(im), a cl_observer, masked_image_mean() or excitable_fraction(): their
                 per-replica forms are replica_cl_observer, masked_image_means(), excitable_fractions() and
                 weighted_means(), computed on the device.

    upload_window  distributed runs: how many of run()'s first iterations may run behind a pipelined upload
                 (fib_set_rect_async blocks, even ranks top to bottom, odd ranks bottom to top; default 10,
                 0 = never; the ranks agree on the number at the start of run())

Collective calls under config['distributed'] (every rank must make them, in the same order):
define(), run() (each iteration), fire_op(), pace(), stop_pacing(), image(), pot().eval() / _State[..].eval(),
var[r, c].eval(), masked_image_mean(), excitable_fraction(), watch_activation(), activation_maps(),
stop_activation(), frames(), checkpoint(), Checkpoint.wait(), restore(), close().  cl_observer callbacks run on
the rank that owns row 20 only and therefore must not call any of these.
"""
import json
import os
import shutil
import time

import numpy as np

from . import _capi
from . import checkpoint as _ckpt
from .sharding import owner_of_row, partition_rows


class DeviceVar:
    """Stand-in for a tf.Variable holding one state plane: .eval() reads it back
    (fenton.py:152-153, court.py:619), .assign(a) uploads, var[r, c].eval() probes one cell (on a batched model
    the row counts through the replicas: replica b's row r is row b * height + r)."""

    def __init__(self, model, name):
        self._model = model
        self.name = name

    def eval(self):
        return self._model._gather(self._model._ctx.get_state(self.name))

    def local(self):
        return self._model._ctx.get_state(self.name)

    def assign(self, value):
        m = self._model
        m._ctx.set_state(self.name, m._own_rows(value))
        return self

    def __getitem__(self, idx):
        return _Cell(self, int(idx[0]), int(idx[1]))


class _Cell:
    def __init__(self, var, row, col):
        self.var, self.row, self.col = var, row, col

    def eval(self):
        return self.var._model._probe(self.var.name, self.row, self.col)


class IonicModel:
    """Base class for cardiac electrophysiology simulation (mirror of ionic.py:30)."""

    MODEL_ID = None         # set by subclasses

    def __init__(self, config):
        self._nranks = 1
        self._phase_rows, self._phase_full, self._holes = None, None, []
        for key, val in config.items():     # ionic.py:35-37
            if key != 'phase':
                setattr(self, key, val)
        self.replicas = int(config.get('replicas', 1))
        if self.replicas < 1:
            raise ValueError('replicas must be >= 1 (got %d)' % self.replicas)
        if self.replicas > 1 and config.get('distributed'):
            raise ValueError('replicas > 1 cannot be combined with distributed: a batched model runs on one GPU')
        diff = config.get('diff')
        if np.ndim(diff) == 1:
            if len(diff) != self.replicas:
                raise ValueError('diff holds %d values for %d replicas' % (len(diff), self.replicas))
            self.replica_diff = [float(d) for d in diff]
        elif diff is not None:
            self.replica_diff = [float(diff)] * self.replicas
        self._ops = {}
        self.defined = False
        self.dt_per_step = 1
        self.cl_observer = None
        self.replica_cl_observer = None
        self._ctx = None
        self._rank, self._nranks = 0, 1
        if config.get('distributed'):
            import torch.distributed as dist
            if not dist.is_initialized():
                raise RuntimeError("config['distributed'] needs torch.distributed.init_process_group first")
            self._rank, self._nranks = dist.get_rank(), dist.get_world_size()
        parts = partition_rows(self.height, self._nranks)
        self._row0, self._rows = parts[self._rank]
        self._rows *= self.replicas             # a batched model: its replicas' rows one after another
        # host copy of the phase field covers these global rows (everything when not sharded)
        # (two halo rows: what the two-steps-per-launch kernel needs; one would do otherwise)
        self._phase_row0 = max(self._row0 - 2, 0)
        self._phase_row1 = min(self._row0 + self._rows + 2, self.height * self.replicas)
        if config.get('phase') is not None:
            self.phase = config['phase']

    # ---- the reference's stencil helpers, as EAGER device ops on NumPy planes -----------------
    # In the reference these build TensorFlow graph nodes; the fused step kernels never call them.
    # They exist so that the stencil arithmetic can be used and checked in isolation (the same
    # device functions as the step kernels: fib_stencil.cuh / fib_common.cuh).
    def _op_device(self):
        d = self.__dict__.get('device')
        return int(d) if d is not None else 0

    def laplace(self, X0):
        """REFLECT-pad X0 by one cell, 9-point stencil, plus the phase-field correction when a
        phase field is defined (ionic.py:44-60).  X0: [height, width] array -> same shape."""
        return _capi.op_laplace(X0, self._phase_plane(np.shape(X0)), 0, self._op_device())

    def phase_field(self, X):
        """The phase-field correction alone (ionic.py:70-81).  Like the reference it takes the
        REFLECT-padded plane X [height+2, width+2] and returns [height, width]."""
        X = np.asarray(X, dtype=np.float32)
        inner = X[1:-1, 1:-1]
        ph = self._phase_plane(inner.shape)
        if ph is None:
            raise AssertionError('phase_field needs a phase field (add_hole_to_phase_field)')
        if not np.array_equal(np.pad(inner, 1, mode='reflect'), X):
            raise ValueError('phase_field expects the REFLECT-padded plane, as laplace() passes it')
        return _capi.op_laplace(inner, ph, 2, self._op_device())

    def enforce_boundary(self, X):
        """Border ring := SYMMETRIC pad of the interior (ionic.py:107-113)."""
        return _capi.op_enforce_boundary(X, self._op_device())

    def rush_larsen(self, g, g_inf, g_tau, dt, name=None):
        """clip(g + (g - g_inf) * expm1(-dt / g_tau), 1e-5, 0.99999) (ionic.py:115-123)."""
        return _capi.op_rush_larsen(g, g_inf, g_tau, dt, False, self._op_device())

    def _phase_plane(self, shape):
        ph = self.phase
        if ph is None:
            return None
        if tuple(ph.shape) != tuple(shape):
            raise ValueError('plane shape %r does not match the phase field %r' % (tuple(shape), ph.shape))
        return ph

    # ---- the phase field: full grid for the user, local rows for the device -------------------
    @property
    def phase(self):
        """[height, width] phase field or None, as in the reference (drivers do
        `model.image() * model.phase`).  A sharded model keeps only its own rows (+2 halo rows)
        for the device and builds the full-grid array on first use from the recorded holes."""
        rows = self.__dict__.get('_phase_rows')
        if rows is None:
            return None
        if self.replicas > 1:
            return rows.reshape(self.replicas, self.height, self.width)
        if self._nranks == 1:
            return rows
        if self.__dict__.get('_phase_full') is None:
            full = None
            for (x, y, radius, neg) in self._holes:
                full = self._apply_hole(full, 0, self.height, x, y, radius, neg)
            self._phase_full = full
        return self._phase_full

    @phase.setter
    def phase(self, value):
        if value is None:
            self._phase_rows, self._phase_full, self._holes = None, None, []
            return
        a = np.asarray(value, dtype=np.float32)
        if self.replicas > 1:
            if a.shape not in ((self.height, self.width), (self.replicas, self.height, self.width)):
                raise ValueError('phase must be [height, width] or [replicas, height, width] = %r'
                                 % ((self.replicas, self.height, self.width),))
            a = self._own_rows(a)
        elif a.shape != (self.height, self.width):
            raise ValueError('phase must be [height, width] = %r' % ((self.height, self.width),))
        if self.__dict__.get('defined'):
            raise AssertionError('the phase field must be set before calling define')
        self._holes = None                      # no longer described by holes
        self._phase_full = a if self._nranks > 1 else None
        self._phase_rows = a[self._phase_row0:self._phase_row1] if self._nranks > 1 else a

    def _apply_hole(self, phase, r0, r1, x, y, radius, neg):
        """ionic.py:95-105 on global rows [r0, r1)."""
        if phase is None:
            phase = np.ones([r1 - r0, self.width], dtype=np.float32)
        xx, yy = np.meshgrid(np.arange(self.width), np.arange(r0, r1))
        dist = np.hypot(xx - x, yy - y)
        if neg:
            phase *= np.array(0.5 * (np.tanh(0.1 * (radius - dist)) + 1.0), dtype=np.float32)
        else:
            phase *= np.array(0.5 * (np.tanh(dist - radius) + 1.0), dtype=np.float32)
        # floor at 1e-5 to avoid division by 0 in the phase-field term (ionic.py:104-105)
        return np.maximum(phase, 1e-5)

    # ---- geometry (ionic.py:83-105) ----------------------------------------------------------
    def add_hole_to_phase_field(self, x, y, radius, neg=False, replica=None):
        """Adds a circular hole centred at (x, y) = (column, row) to the phase field; with
        neg=True the inside is kept and the outside excluded.  Must precede define().  A batched model:
        in replica `replica` only, or in every replica (None)."""
        if self.defined:
            raise AssertionError('add_hole_to_phase_field should be called before calling define')
        if self._holes is None:
            raise AssertionError('the phase field was assigned directly; holes cannot be added to it')
        if replica is not None or self.replicas > 1:
            B, H = self.replicas, self.height
            if replica is not None and not 0 <= int(replica) < B:
                raise ValueError('replica %r out of range 0..%d' % (replica, B - 1))
            if self._phase_rows is None:
                self._phase_rows = np.ones([B * H, self.width], dtype=np.float32)
            for b in range(B) if replica is None else [int(replica)]:
                self._phase_rows[b * H:(b + 1) * H] = self._apply_hole(self._phase_rows[b * H:(b + 1) * H], 0, H,
                                                                       x, y, radius, neg)
            self._holes.append((x, y, radius, neg))
            return
        self._phase_rows = self._apply_hole(self._phase_rows, self._phase_row0, self._phase_row1,
                                            x, y, radius, neg)
        self._holes.append((x, y, radius, neg))
        self._phase_full = None

    # ---- device context ---------------------------------------------------------------------
    def _make_context(self, flags=0, steps_per_launch=0):
        cfgd = self.__dict__
        device = cfgd.get('device')
        if device is None:
            device = int(os.environ.get('LOCAL_RANK', 0)) if self._nranks > 1 else 0
        if not cfgd.get('graph', True):
            flags |= _capi.F_NO_GRAPH
        if not cfgd.get('persist', True):
            flags |= _capi.F_NO_PERSIST
        sharded = self._nranks > 1
        batched = {'replicas': self.replicas} if self.replicas > 1 else {}
        ctx = _capi.Context(self.MODEL_ID, self.height, self.width, self.dt, self.replica_diff[0], flags=flags,
                            device=device, row0=self._row0 if sharded else 0,
                            rows=self._rows if sharded else 0, steps_per_launch=steps_per_launch, **batched)
        if batched and len(set(self.replica_diff)) > 1:
            ctx.set_replica_diff(self.replica_diff)
        if self._phase_rows is not None:
            ctx.set_phase(np.asarray(self._phase_rows, dtype=np.float32), self._phase_row0)
        if sharded:
            import torch.distributed as dist
            box = [_capi.comm_unique_id() if self._rank == 0 else None]
            dist.broadcast_object_list(box, src=0)
            ctx.comm_init(self._nranks, self._rank, box[0])
        self._ctx = ctx
        return ctx

    # The context, with one twist for NCCL shards: iterations that run() has counted to run behind a
    # pipelined upload (csrc finish_upload_session) are executed by the first thing that touches the context
    # -- every such touch is a collective call under config['distributed'], and every rank holds the same
    # count, so all ranks issue fib_step_behind_upload at the same point of their call sequence.
    @property
    def _ctx(self):
        d = self.__dict__
        n = d.get('_behind', 0)
        if n:
            d['_behind'], d['_behind_limit'] = 0, 0
            d['_ctx_obj'].step_behind_upload(n)
        return d.get('_ctx_obj')

    @_ctx.setter
    def _ctx(self, value):
        self.__dict__['_ctx_obj'] = value

    def _agree_on_upload_window(self, im, batch):
        """How many of run()'s first iterations all ranks will run behind their pipelined uploads (0: none).
        Collective: the answer is the minimum over the ranks, so one rank without a complete upload of the right
        direction (even ranks top to bottom, odd ranks bottom to top) switches it off for everybody."""
        if self._nranks == 1 or im or batch <= 1 or self.ode_op(0) != 0:
            return 0
        import torch
        import torch.distributed as dist
        open_, complete, direction, room = self.__dict__['_ctx_obj'].upload_state()
        ok = open_ and complete and direction == (1 if self._rank % 2 == 0 else -1)
        want = min(room, self.samples, int(self.__dict__.get('upload_window', 10))) if ok else 0
        dev = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend() == 'nccl' else torch.device('cpu')
        t = torch.tensor([want], dtype=torch.int64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return int(t.item())

    def _local_full(self, value):
        """[rows, W] fp32 array filled with `value` for this shard's rows."""
        return np.full([self._rows, self.width], value, dtype=np.float32)

    def _own_rows(self, value):
        """This context's rows of a full-grid array: [height, width] (every replica), or [replicas, height, width]."""
        a = np.asarray(value, dtype=np.float32)
        if self.replicas > 1:
            return np.broadcast_to(a, (self.replicas, self.height, self.width)).reshape(self._rows, self.width)
        return np.broadcast_to(a, (self.height, self.width))[self._row0:self._row0 + self._rows]

    def _gather(self, local):
        if self.replicas > 1:
            return local.reshape(self.replicas, self.height, -1)
        if self._nranks == 1:
            return local
        import torch.distributed as dist
        parts = [None] * self._nranks
        dist.all_gather_object(parts, local)
        return np.concatenate(parts, axis=0)

    def _probe(self, name, row, col):
        """One cell of a state plane; in a sharded run the owner rank reads it and shares it."""
        own = owner_of_row(self.height, self._nranks, row) == self._rank
        v = self._ctx.probe(name, row, col) if own else None
        if self._nranks == 1:
            return v
        import torch.distributed as dist
        vals = [None] * self._nranks
        dist.all_gather_object(vals, v)
        return [x for x in vals if x is not None][0]

    # ---- stimulation (ionic.py:125-169) ------------------------------------------------------
    def add_pace_op(self, name, loc, v):
        """Registers a stimulator: pot := max(pot, s), s = v inside the named region and min_v
        elsewhere.  loc in left/right/top/bottom/luq/llq/ruq/rlq.  Must follow define()."""
        if not self.defined:
            raise AssertionError('add_hole_to_phase_field should be called after calling define')
        H, W = self.height, self.width
        regions = {
            'left': (0, H, 0, 5), 'right': (0, H, W - 5, W), 'top': (0, 5, 0, W),
            'bottom': (H - 5, H, 0, W), 'luq': (1, H // 2, 1, W // 2),
            'llq': (H // 2, H - 1, 1, W // 2), 'ruq': (1, H // 2, W // 2, W - 1),
            'rlq': (H // 2, H - 1, W // 2, W - 1),
        }
        rect = regions.get(loc)
        if rect is None:
            print('undefined pace location')      # ionic.py:161-162: the op still clamps at min_v
            rect = (0, 0, 0, 0)
        self._ops[name] = ('pace', rect, float(v))

    def fire_op(self, name, replica=None):
        """Executes an op registered by add_pace_op (or a model op such as 'slow').  A batched model: a
        stimulus in replica `replica` only, or in every replica (None)."""
        op = self._ops[name]
        if op[0] == 'pace':
            (r0, r1, c0, c1), v = op[1], op[2]
            where = {} if replica is None else {'replica': self._check_replica(replica)}
            self._ctx.stimulate(self._pot_name, max(r0, 0), r1, max(c0, 0), c1, v, float(self.min_v), **where)
        elif op[0] == 'call':
            op[1]()

    def _check_replica(self, replica):
        if not 0 <= int(replica) < self.replicas:
            raise ValueError('replica %r out of range 0..%d' % (replica, self.replicas - 1))
        return int(replica)

    def pace(self, name, at, every=0, count=1, replica=None):
        """Schedules the op `name` registered with add_pace_op on the device: it fires after the absolute ODE
        iterations n = at + 1 + j * every (n counts `iterations`), j = 0 .. count - 1, or until stop_pacing() with
        count = 0.  That is the iteration after which a driver's `for i in run(): if i == at: fire_op(name)` fires,
        in the first run() after define(); `at` usually comes from millisecond_to_step(t).  The stimulus is applied
        while stepping (include/fib_b200.h fib_pace_add): a train needs no call per beat and keeps the persistent
        kernel's batches.  Frames and activation maps see an iteration before its stimulus, the probe after it.
        checkpoint() saves the schedules and restore() continues them.  At most 4 schedules are active at once.
        ValueError if iteration at + 1 has already been stepped.  Collective when distributed.  A batched model:
        the stimulus in replica `replica` only, or in every replica (None)."""
        if not self.defined:
            raise AssertionError('pace should be called after calling define')
        op = self._ops.get(name)
        if op is None or op[0] != 'pace':
            raise ValueError('pace: %r is not an op registered with add_pace_op' % (name,))
        at, every, count = int(at), int(every), int(count)
        if count < 0 or (count != 1 and every < 1):
            raise ValueError('pace: need count >= 0 and every >= 1 unless count == 1 (got every %d, count %d)'
                             % (every, count))
        if at + 1 <= self.iterations:
            raise ValueError('pace: iteration %d (at = %d) has already been stepped (iterations = %d)'
                             % (at + 1, at, self.iterations))
        (r0, r1, c0, c1), v = op[1], op[2]
        entry = {'name': name, 'rect': [max(r0, 0), r1, max(c0, 0), c1], 'value': v, 'floor': float(self.min_v),
                 'next': at + 1, 'every': every, 'count': count}
        where = {}
        if replica is not None:
            entry['replica'] = where['replica'] = self._check_replica(replica)
        entry['id'] = self._ctx.pace_add(*entry['rect'], v, entry['floor'], at + 1 - self.iterations, every, count,
                                         **where)
        self._pacing = self._active_pacing() + [entry]

    def _active_pacing(self):
        """The schedules whose last beat is still to come (the library drops the others by itself)."""
        return [e for e in self.__dict__.get('_pacing') or [] if _ckpt.pacing_state([e], self.iterations)]

    def stop_pacing(self, name=None):
        """Removes the schedules of the op `name`, or every schedule.  Collective when distributed."""
        for e in self.__dict__.get('_pacing') or []:
            if name is None or e['name'] == name:
                self._ctx.pace_remove(e['id'])
        self._pacing = [e for e in self._active_pacing() if name is not None and e['name'] != name]

    # ---- the run() generator (ionic.py:171-245) ----------------------------------------------
    def run(self, im=None, keep_state=False, block=True):
        """Generator: advances the model one iteration (= dt_per_step time steps) per yield.

            for i in model.run(im):
                if i == s2: model.fire_op('s2')

        replica_cl_observer(i, replica, cl), when set, is cl_observer for every replica: each replica's probe cell
        image[20, W//2] is recorded on the device (include/fib_b200.h, fib_replica_probe_watch), and the observer is
        called in order of i, then replica.  Headless, unsharded, and not together with cl_observer.
        """
        if not self.defined:
            raise AssertionError('define() must be called before run()')
        if self.replicas > 1 and (im or self.cl_observer is not None):
            raise ValueError('run(im) and cl_observer watch one cell of one grid: a batched model (replicas = %d) '
                             'has replica_cl_observer and activation maps (watch_activation) instead' % self.replicas)
        rep_obs = self.replica_cl_observer
        if rep_obs is not None and (self.cl_observer is not None or im or self._nranks > 1):
            raise ValueError('replica_cl_observer: a headless run of an unsharded model, without cl_observer')
        then = time.time()
        nrep = self.replicas if rep_obs is not None else 1
        v0 = [self.min_v] * nrep
        last_spike = [0] * nrep
        self.samples = int(self.duration / (self.dt_per_step * self.dt))
        plot_every = max(int(self.dt_per_plot / self.dt_per_step), 1)
        watch = bool(im) or self.cl_observer is not None or rep_obs is not None
        prow, pcol = 20, self.width // 2                         # ionic.py:216
        # Headless watching: the owner rank of row 20 records the probe cell on the device after every
        # iteration (fib_probe_watch: a node of the iteration's CUDA graph) and reads the ring back once
        # per `probe_batch` iterations -- no host round trip per iteration.
        owner = self._row0 <= prow < self._row0 + self._rows
        ring = watch and not im and owner
        batch = max(1, min(int(self.__dict__.get('probe_batch', 64)), _capi.PROBE_RING // 2))
        unread = []                                              # iterations recorded, not yet read

        def crossing(i, v1, b=0):
            if v1 >= 0.5 and v0[b] < 0.5:
                cl = (i - last_spike[b]) * self.dt_per_step * self.dt
                if rep_obs is not None:
                    rep_obs(i, b, cl)
                elif self.cl_observer is None:
                    print('wavefront reaches the middle top point at %d, cycle length is %d' % (i, cl))
                else:
                    self.cl_observer(i, cl)
                last_spike[b] = i
            v0[b] = v1

        def drain(n):
            # the oldest n recorded iterations; the library waits only for the launch that produced
            # them, so the iterations stepped since keep the device busy meanwhile
            fetch = self._ctx.probe_fetch if rep_obs is None else self._ctx.replica_probe_fetch
            vals = fetch(n) if n else []
            if len(vals) != n:
                raise RuntimeError('probe ring returned %d values for %d iterations' % (len(vals), n))
            # replica b's probe cell is row b * height + prow of the model's rows
            w = [self._probe_weight(b * self.height + prow, pcol) for b in range(nrep)]
            for k, rec in zip(unread[:n], vals):
                if k % plot_every == 0:
                    for b, raw in enumerate(np.reshape(rec, nrep)):
                        crossing(k, self._normalise(float(raw)) * w[b], b)
            del unread[:n]

        self._behind, self._behind_limit = 0, self._agree_on_upload_window(im, batch)
        self._upload_window_used = self._behind_limit
        if ring and rep_obs is not None:
            # a batched ring may hold fewer records than run() leaves unread (two batches)
            batch = max(1, min(batch, self._ctx.replica_probe_watch(self._pot_name, prow, pcol) // 2))
        elif ring:
            self._ctx.probe_watch(self._pot_name, prow, pcol)
        try:
            for i in range(self.samples):
                if i < self._behind_limit:
                    self._behind += 1                        # runs behind the upload: see the _ctx property
                    if self._behind == self._behind_limit:
                        self._ctx                            # noqa: B018 (the window is full: go)
                else:
                    self._ctx.step(self.ode_op(i), 1)
                self.iterations += 1
                if self.__dict__.get('_frames') is not None:
                    self._drain_frames()
                yield i
                if ring:
                    unread.append(i)
                    if batch == 1:
                        drain(1)
                    elif len(unread) >= 2 * batch:
                        drain(batch)
                elif im and i % plot_every == 0:
                    image = self.image()
                    if self.phase is not None:
                        image *= self.phase
                    im.imshow(image)
                    crossing(i, image[prow, pcol])
            if ring:
                drain(len(unread))
        finally:
            if ring and self._ctx is not None:
                (self._ctx.probe_watch if rep_obs is None else self._ctx.replica_probe_watch)(self._pot_name, -1, -1)
        if keep_state:                                           # ionic.py:226-229
            self.state = {}
            for s in self._State:
                self.state[s] = self._State[s].eval()
        if getattr(self, 'timeline', False):
            self._write_timeline()
        self._ctx.sync()
        self._release_restore_buffers()
        print('elapsed: %f sec' % (time.time() - then))
        if block and im:
            im.wait()

    def _probe_image(self, row, col):
        v = float(self._ctx.probe(self._pot_name, row, col))
        v = self._normalise(v)
        return v * self._probe_weight(row, col)

    def _probe_weight(self, row, col):
        if self._phase_rows is not None and self._phase_row0 <= row < self._phase_row1:
            return float(self._phase_rows[row - self._phase_row0, col])
        return 1.0

    def _normalise(self, v):
        return (v - self.min_v) / (self.max_v - self.min_v)

    def _write_timeline(self):
        """The reference traces ONE extra iteration after the loop with TF's FULL_TRACE
        (ionic.py:231-241), which also advances the state once more.  Here: CUDA-event timing of
        one extra iteration, written as a chrome-trace JSON to config['timeline_name']."""
        c = self._ctx
        c.sync()
        n0 = c.launch_count()
        c.timer_start()
        c.step(self.ode_op(self.samples), 1)
        self.iterations += 1
        c.timer_stop()
        ms = c.timer_ms()
        ev = [{'name': 'ode_op (%d fused step kernels)' % (c.launch_count() - n0), 'ph': 'X',
               'pid': 0, 'tid': 0, 'ts': 0, 'dur': ms * 1000.0,
               'args': {'cells': self.height * self.width, 'dt_per_step': self.dt_per_step}}]
        with open(self.timeline_name, 'w') as f:
            json.dump({'traceEvents': ev}, f)

    def millisecond_to_step(self, t):
        """Converts t in milliseconds to the iteration count returned by run()."""
        return int(t / (self.dt_per_step * self.dt))

    def define(self, s1=True):
        """Placeholder replaced in subclasses: builds the initial state and the device context."""
        self.defined = True
        self.iterations = 0         # ODE iterations since define(), continued by restore()
        self._pacing = []           # the pace() schedules: name, rect, value, floor, next, every, count, entry id

    def image(self):
        """[height x width] float ndarray in 0..1 encoding the transmembrane potential."""
        pass

    def pot(self):
        """Handle of the transmembrane variable."""
        pass

    def ode_op(self, tick):
        """The op run once per iteration (ionic.py:277-286)."""
        if hasattr(self, '_ode_op'):
            return self._ode_op
        elif tick % self.fast_slow_ratio == 0:
            return self._ode_slow_op
        else:
            return self._ode_fast_op

    # ---- dummy context, as when XLA is unavailable (ionic.py:288-307) ------------------------
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def jit_scope(self):
        return self

    # ---- extras ---------------------------------------------------------------------------------
    def add_probe_mask(self, mask):
        """Registers an [H, W] weight plane on the device (at most 4) and returns its slot; use
        with masked_image_mean().  Backs the pseudo-electrograms of the reference's egm.py.  A batched
        model takes [H, W] (the same mask in every replica) or [B, H, W]; use with masked_image_means()."""
        if not self.defined:
            raise AssertionError('add_probe_mask should be called after calling define')
        slot = len(self.__dict__.setdefault('_mask_slots', []))
        self._ctx.set_weights(slot, self._own_rows(mask), self._row0)
        self._mask_slots.append(slot)
        return slot

    def masked_image_mean(self, slot):
        """np.mean(self.image() * mask) (egm.py:44-47) without moving the frame to the host:
        one weighted reduction on the device (summed over ranks when sharded)."""
        self._refuse_batched_sum('masked_image_mean')
        swx, sw = self._ctx.masked_sum(self._pot_name, slot)
        if self._nranks > 1:
            import torch.distributed as dist
            parts = [None] * self._nranks
            dist.all_gather_object(parts, (swx, sw))
            swx, sw = sum(p[0] for p in parts), sum(p[1] for p in parts)
        # image = (V - min_v) / (max_v - min_v) for BR / Courtemanche, V itself for 4v
        if self.MODEL_ID != _capi.FENTON4V:
            swx = (swx - self.min_v * sw) / (self.max_v - self.min_v)
        return swx / (self.height * self.width)

    def excitable_fraction(self, cutoff=0.2, phase_min=1e-3):
        """rho of court_ultra.py:504-509: np.sum(image[phase > phase_min] < cutoff) /
        np.sum(phase > phase_min) with image = self.image(), as one threshold-count reduction on the
        device (summed over ranks when sharded) -- no frame leaves the GPU."""
        self._refuse_batched_sum('excitable_fraction')
        if self.MODEL_ID == _capi.FENTON4V:
            sub, div = 0.0, 1.0
        else:
            sub, div = float(self.min_v), float(self.max_v - self.min_v)
        below, total = self._ctx.count_below(self._pot_name, sub, div, cutoff, phase_min)
        if self._nranks > 1:
            import torch.distributed as dist
            parts = [None] * self._nranks
            dist.all_gather_object(parts, (below, total))
            below, total = sum(p[0] for p in parts), sum(p[1] for p in parts)
        return below / total if total else float('nan')

    def _refuse_batched_sum(self, what):
        if self.replicas > 1:
            raise ValueError('%s sums over the whole grid, and this model holds %d replicas: use its per-replica form '
                             '(masked_image_means, excitable_fractions, weighted_means)' % (what, self.replicas))

    # ---- per-replica observers: one value per replica, [B] (B = 1 on an unbatched model) ------------------------
    def _refuse_distributed(self, what):
        if self._nranks > 1:
            raise ValueError('%s: per-replica observers need an unsharded model (the scalar forms cover sharded '
                             'runs)' % what)

    def masked_image_means(self, slot):
        """float64 [B]: masked_image_mean(slot) of every replica, np.mean(image()[b] * mask[b]), from one
        reduction per replica on the device (include/fib_b200.h, fib_replica_sums)."""
        self._refuse_distributed('masked_image_means')
        swx, sw = self._ctx.replica_sums(self._pot_name, slot)
        if self.MODEL_ID != _capi.FENTON4V:
            swx = (swx - self.min_v * sw) / (self.max_v - self.min_v)
        return swx / (self.height * self.width)

    def excitable_fractions(self, cutoff=0.2, phase_min=1e-3):
        """float64 [B]: excitable_fraction(cutoff, phase_min) of every replica (NaN where no cell has phase >
        phase_min), from one threshold count per replica on the device (fib_replica_count_below)."""
        self._refuse_distributed('excitable_fractions')
        if self.MODEL_ID == _capi.FENTON4V:
            sub, div = 0.0, 1.0
        else:
            sub, div = float(self.min_v), float(self.max_v - self.min_v)
        below, total = self._ctx.replica_count_below(self._pot_name, sub, div, cutoff, phase_min)
        return np.where(total > 0, below / np.maximum(total, 1), np.nan)

    def weighted_means(self, name):
        """float64 [B]: the phase-weighted mean of state `name` in every replica, np.average(x[b],
        weights=phase[b]) (the plain mean without a phase field) -- the means of court_ultra.py's cl_observer."""
        self._refuse_distributed('weighted_means')
        swx, sw = self._ctx.replica_sums(name, -1)
        return swx / sw

    def watch_activation(self, up=None, down=None):
        """Arms the device-side activation maps of the transmembrane variable (include/fib_b200.h,
        fib_activation_watch): from now on, after every iteration, every cell records its up-crossings of
        `up` and down-crossings of `down` (raw units of the potential; both default to min_v + 0.5 (max_v -
        min_v), the reference's cycle-length probe level of 0.5 on the normalised image), linearly
        interpolated between consecutive iterations.  Calling it again resets the maps."""
        if not self.defined:
            raise AssertionError('watch_activation should be called after calling define')
        mid = float(self.min_v) + 0.5 * (float(self.max_v) - float(self.min_v))
        self._ctx.activation_watch(mid if up is None else float(up), mid if down is None else float(down))

    def activation_maps(self):
        """{name: [height, width] float64} in ms since watch_activation():
            first, last, previous  the first, the last and the one-before-last activation time
            repol                  the last repolarisation time
            count                  the number of activations
            apd                    repol - last where repol > last (the last beat has repolarised), else NaN
            cycle                  last - previous
        Empty times are NaN.  Conduction velocity follows from differences of `last` (or `first`) between
        cells; cycle-length and APD heterogeneity from `cycle` and `apd`."""
        ms = self.dt_per_step * self.dt
        c = self._ctx
        raw = {k: self._gather(c.activation_get(m)).astype(np.float64)
               for k, m in (('first', _capi.ACT_FIRST), ('last', _capi.ACT_LAST), ('previous', _capi.ACT_PREV),
                            ('repol', _capi.ACT_REPOL), ('count', _capi.ACT_COUNT))}
        out = {k: v * ms for k, v in raw.items() if k != 'count'}
        out['count'] = raw['count']
        with np.errstate(invalid='ignore'):
            out['apd'] = np.where(out['repol'] > out['last'], out['repol'] - out['last'], np.nan)
        out['cycle'] = out['last'] - out['previous']
        return out

    def stop_activation(self):
        """Disarms the activation maps and frees their device memory."""
        self._ctx.activation_stop()

    # The persistent kernel launches 64 iterations at a time (csrc fib_step); run() fetches frames one such batch
    # behind the stepping, so a fetch never waits for the launch in flight and never cuts a batch.
    FRAME_BATCH = 64

    @classmethod
    def default_frame_capacity(cls, every):
        """Ring frames that run()'s drain never overflows: it leaves at most two batches of iterations unfetched,
        which hold at most 2 * (ceil(64 / every) + 1) frames."""
        return 2 * (-(-cls.FRAME_BATCH // int(every)) + 1)

    def record_frames(self, every, stride=1, first=1, name=None, capacity=None):
        """Arms the device-side frame recorder (include/fib_b200.h, fib_frames_watch): plane `name` (default: the
        potential) at every `stride`-th row and column, recorded on the device at the end of iterations k = first,
        first + every, ... counted from this call (k = 0 is the plane now), into a ring of `capacity` frames.
        run() drains the ring by itself; frames() returns the movie.  first = 1, every = 10 are the reference
        drivers' cadence (`cube[i // 10]` grabbed after the iteration run() yields as i = 0, 10, ...).
        Calling it again starts a new movie."""
        if not self.defined:
            raise AssertionError('record_frames should be called after calling define')
        every, stride, first = int(every), int(stride), int(first)
        if every < 1 or stride < 1 or first < 0:
            raise ValueError('record_frames: need every >= 1, stride >= 1 and first >= 0')
        capacity = self.default_frame_capacity(every) if capacity is None else int(capacity)
        name = self._pot_name if name is None else name
        self._ctx.frames_watch(name, first, every, stride, capacity)
        self._frames = {'name': name, 'first': first, 'every': every, 'stride': stride, 'capacity': capacity,
                        'k': 0, 'upto': 0, 'iters': [], 'cube': []}

    def _drain_frames(self):
        """After an ODE iteration of run(): every FRAME_BATCH iterations, fetch the frames of the batch before
        the last one (they are in launched work, so the library neither flushes nor waits for the last launch)."""
        f = self._frames
        f['k'] += 1
        B = self.FRAME_BATCH
        if f['k'] % B or f['k'] < 2 * B:
            return
        limit = f['k'] - B
        upto = 0 if limit < f['first'] else (limit - f['first']) // f['every'] + 1
        if upto > f['upto']:
            iters, cube = self._ctx.frames_fetch(upto - f['upto'])
            f['iters'].append(iters)
            f['cube'].append(cube)
            f['upto'] = upto

    def frames(self):
        """(iters, cube): the frames recorded since record_frames() or the last frames() call.  iters[n] (int64)
        are the k of the frames; cube is [n, ceil(height / stride), ceil(width / stride)] float32, the potential
        normalised exactly like image() (raw U for 4v, (V - min_v) / (max_v - min_v) otherwise), any other
        variable raw.  Frames lost to a ring overflow show as gaps in iters.  Collective when distributed: the
        shards' rows are gathered in rank order."""
        f = self.__dict__.get('_frames')
        if f is None:
            raise AssertionError('frames() needs record_frames() first')
        rows, cols = self._ctx.frames_shape()
        self._fetch_frames()
        iters = np.concatenate(f['iters']).astype(np.int64)
        cube = np.concatenate(f['cube']) if f['cube'] else np.empty((0, rows, cols), np.float32)
        f['iters'], f['cube'] = [], []
        if self._nranks > 1:
            import torch.distributed as dist
            parts = [None] * self._nranks
            dist.all_gather_object(parts, cube)
            cube = np.concatenate(parts, axis=1)
        if self.replicas > 1:
            cube = cube.reshape(len(cube), self.replicas, rows // self.replicas, cols)
        if f['name'] == self._pot_name and self.MODEL_ID != _capi.FENTON4V:
            cube = self._normalise(cube)
        return iters, cube

    def _fetch_frames(self):
        """Moves every frame recorded so far from the ring into the host list."""
        f = self._frames
        while True:
            iters, cube = self._ctx.frames_fetch(self.FRAME_BATCH)
            f['iters'].append(iters)
            f['cube'].append(cube)
            if len(iters) < self.FRAME_BATCH:
                break
        f['upto'] = 0 if f['k'] < f['first'] else (f['k'] - f['first']) // f['every'] + 1

    def stop_frames(self):
        """Disarms the frame recorder and frees its ring; frames not yet returned by frames() are dropped."""
        self._ctx.frames_stop()
        self._frames = None

    def nonfinite_cells(self):
        """{variable: count} of NaN/Inf cells in this shard (empty dict when the state is healthy):
        the NaN watch the reference left commented out (ionic.py:199,208-212), as one small
        reduction per plane on the device."""
        out = {}
        for name in self._ctx.var_names:
            n = self._ctx.count_nonfinite(name)
            if n:
                out[name] = n
        return out

    def image_async(self, pinned_out):
        """Starts an asynchronous grab of the raw transmembrane plane of this shard into a pinned
        array (fib_tf_b200._capi.pinned_empty) and returns at once; image_wait() completes it and
        returns the frame normalised like image().  Lets a driver save frames (cube.npy,
        fenton.py:179-187) without stalling the time stepping."""
        self._ctx.snapshot_begin(self._pot_name, pinned_out)
        self._snap = pinned_out

    def image_wait(self):
        self._ctx.snapshot_wait()
        a = getattr(self, '_snap', None)
        if a is None:
            raise RuntimeError('image_wait() without a preceding image_async()')
        return a if self.MODEL_ID == _capi.FENTON4V else self._normalise(a)

    # ---- checkpoint and restart (fib_tf_b200/checkpoint.py) -----------------------------------
    def checkpoint(self, path):
        """Saves the state after the iterations stepped so far, the armed activation map and frame recorder, and
        the pacing schedules still to fire, to the directory `path` while stepping continues: stages a device copy of every shard behind the work
        already enqueued and returns a Checkpoint at once; writer threads fill the files meanwhile.  Frames
        recorded so far move to the host list first (frames() returns them; they are not saved).  The previous
        checkpoint at `path` stays readable until Checkpoint.wait() replaces it, atomically where the file
        system allows.  Collective when distributed."""
        if not self.defined:
            raise AssertionError('checkpoint should be called after calling define')
        self._finish_checkpoint()
        if self.__dict__.get('_frames') is not None:
            self._fetch_frames()
        path = os.path.abspath(path)
        partial = path + '.partial'
        if self._rank == 0 and os.path.exists(partial):
            shutil.rmtree(partial)
        if self._rank == 0:
            os.makedirs(partial)
        if self._nranks > 1:
            import torch.distributed as dist
            dist.barrier()
        ck = Checkpoint(self, path, partial, _ckpt.save_shard(self._ctx, partial, self._own_phase_rows()),
                        self.iterations, _ckpt.pacing_state(self.__dict__.get('_pacing') or [], self.iterations))
        self._ckpt = ck
        return ck

    def _own_phase_rows(self):
        """This shard's rows of the phase field, or None."""
        if self._phase_rows is None:
            return None
        lo = self._row0 - self._phase_row0
        return self._phase_rows[lo:lo + self._rows]

    def _finish_checkpoint(self):
        ck = self.__dict__.get('_ckpt')
        if ck is not None:
            ck.wait()

    def restore(self, path):
        """Instead of define(): builds the device context exactly as define() does, then loads the checkpoint
        at `path` -- saved on any number of ranks -- with the armed observers and the pacing schedules resumed, and continues
        `iterations` from it.  ValueError if this model's config or phase field would compute differently.
        A large grid with no observer steps its first iterations behind its own upload.  Collective when
        distributed."""
        man = _ckpt.load_manifest(path)
        ctx = self._create()
        own = self._own_phase_rows()
        try:
            _ckpt.check_compatible(man, ctx, own)
            _ckpt.check_phase(path, man, ctx, own)
            self._pacing = _ckpt.resume_pacing(ctx, man.get('pacing', []), man['iterations'])
            self._restore_pinned = _ckpt.restore_context(ctx, path, bottom_up=self._rank % 2 == 1, man=man)
        except BaseException:
            self.close()
            self.defined = False
            raise
        self.iterations = man['iterations']
        fr = man['frames']
        if fr['armed']:
            k = fr['k']
            self._frames = {'name': fr['var'], 'first': fr['first'], 'every': fr['every'], 'stride': fr['stride'],
                            'capacity': fr['capacity'], 'k': k, 'iters': [], 'cube': [],
                            'upto': 0 if k < fr['first'] else (k - fr['first']) // fr['every'] + 1}
        return man

    def _release_restore_buffers(self):
        """The host copies of a restore, once a synchronous call has consumed them."""
        _ckpt.release(self.__dict__.get('_restore_pinned') or [])

    def sync(self):
        self._ctx.sync()
        self._release_restore_buffers()

    def close(self):
        try:
            self._finish_checkpoint()
        finally:
            if self._ctx is not None:
                self._ctx.close()
                self._ctx = None
            self._release_restore_buffers()


class Checkpoint:
    """A save started by IonicModel.checkpoint(); wait() completes it."""

    def __init__(self, model, path, partial, writer, iterations, pacing=()):
        self.model, self.path, self.partial, self.writer = model, path, partial, writer
        self.iterations, self.pacing = iterations, list(pacing)
        self.done = False

    def wait(self):
        """Joins the writers, agrees with the other ranks that every shard was saved, then rank 0 writes the
        manifest and puts the checkpoint at `path`.  RuntimeError if any rank failed; the previous checkpoint
        at `path` is then left as it was.  Collective when distributed."""
        if self.done:
            return self
        self.done = True
        m = self.model
        if m.__dict__.get('_ckpt') is self:
            m._ckpt = None
        ok = self.writer.join()
        mine = (ok, None if ok else repr(self.writer.error), self.writer.record, self.writer.info)
        parts = [mine]
        if m._nranks > 1:
            import torch.distributed as dist
            parts = [None] * m._nranks
            dist.all_gather_object(parts, mine)
        failed = ['rank %d: %s' % (r, p[1]) for r, p in enumerate(parts) if not p[0]]
        err = None
        if m._rank == 0:
            try:
                if failed:
                    shutil.rmtree(self.partial, ignore_errors=True)
                else:
                    man = _ckpt.manifest(self.writer.ctx, parts[0][3], [p[2] for p in parts], self.iterations,
                                         self.pacing)
                    _ckpt.write_manifest(self.partial, man)
                    _ckpt.publish(self.partial, self.path)
            except Exception as e:
                err = repr(e)
        if m._nranks > 1:
            import torch.distributed as dist
            box = [err]
            dist.broadcast_object_list(box, src=0)
            err = box[0]
        if failed:
            raise RuntimeError('checkpoint %s was not saved: %s' % (self.path, '; '.join(failed)))
        if err is not None:
            raise RuntimeError('checkpoint %s was not published: %s' % (self.path, err))
        return self
