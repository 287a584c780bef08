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

    upload_window  distributed runs: how many of run()'s first iterations may run behind a pipelined upload
                 (fib_set_rect_async blocks, even ranks top to bottom, odd ranks bottom to top; default 10,
                 0 = never; the ranks agree on the number at the start of run())

Collective calls under config['distributed'] (every rank must make them, in the same order):
define(), run() (each iteration), fire_op(), image(), pot().eval() / _State[..].eval(),
var[r, c].eval(), masked_image_mean(), excitable_fraction(), watch_activation(), activation_maps(),
stop_activation(), close().  cl_observer callbacks run on
the rank that owns row 20 only and therefore must not call any of these.
"""
import json
import os
import time

import numpy as np

from . import _capi
from .sharding import owner_of_row, partition_rows


class DeviceVar:
    """Stand-in for a tf.Variable holding one state plane: .eval() reads it back
    (fenton.py:152-153, court.py:619), .assign(a) uploads, var[r, c].eval() probes one cell."""

    def __init__(self, model, name):
        self._model = model
        self.name = name

    def eval(self):
        return self._model._gather(self._model._ctx.get_state(self.name))

    def local(self):
        return self._model._ctx.get_state(self.name)

    def assign(self, value):
        m = self._model
        a = np.broadcast_to(np.asarray(value, dtype=np.float32), (m.height, m.width))
        m._ctx.set_state(self.name, a[m._row0:m._row0 + m._rows])
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
        self._ops = {}
        self.defined = False
        self.dt_per_step = 1
        self.cl_observer = None
        self._ctx = None
        self._rank, self._nranks = 0, 1
        if config.get('distributed'):
            import torch.distributed as dist
            if not dist.is_initialized():
                raise RuntimeError("config['distributed'] needs torch.distributed.init_process_group first")
            self._rank, self._nranks = dist.get_rank(), dist.get_world_size()
        parts = partition_rows(self.height, self._nranks)
        self._row0, self._rows = parts[self._rank]
        # host copy of the phase field covers these global rows (everything when not sharded)
        # (two halo rows: what the two-steps-per-launch kernel needs; one would do otherwise)
        self._phase_row0 = max(self._row0 - 2, 0)
        self._phase_row1 = min(self._row0 + self._rows + 2, self.height)
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
        if a.shape != (self.height, self.width):
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
    def add_hole_to_phase_field(self, x, y, radius, neg=False):
        """Adds a circular hole centred at (x, y) = (column, row) to the phase field; with
        neg=True the inside is kept and the outside excluded.  Must precede define()."""
        if self.defined:
            raise AssertionError('add_hole_to_phase_field should be called before calling define')
        if self._holes is None:
            raise AssertionError('the phase field was assigned directly; holes cannot be added to it')
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
        ctx = _capi.Context(self.MODEL_ID, self.height, self.width, self.dt, self.diff, flags=flags,
                            device=device, row0=self._row0 if sharded else 0,
                            rows=self._rows if sharded else 0, steps_per_launch=steps_per_launch)
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

    def _gather(self, local):
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

    def fire_op(self, name):
        """Executes an op registered by add_pace_op (or a model op such as 'slow')."""
        op = self._ops[name]
        if op[0] == 'pace':
            (r0, r1, c0, c1), v = op[1], op[2]
            self._ctx.stimulate(self._pot_name, max(r0, 0), r1, max(c0, 0), c1, v, float(self.min_v))
        elif op[0] == 'call':
            op[1]()

    # ---- the run() generator (ionic.py:171-245) ----------------------------------------------
    def run(self, im=None, keep_state=False, block=True):
        """Generator: advances the model one iteration (= dt_per_step time steps) per yield.

            for i in model.run(im):
                if i == s2: model.fire_op('s2')
        """
        if not self.defined:
            raise AssertionError('define() must be called before run()')
        then = time.time()
        v0 = self.min_v
        last_spike = 0
        self.samples = int(self.duration / (self.dt_per_step * self.dt))
        plot_every = max(int(self.dt_per_plot / self.dt_per_step), 1)
        watch = bool(im) or self.cl_observer is not None
        prow, pcol = 20, self.width // 2                         # ionic.py:216
        # Headless watching: the owner rank of row 20 records the probe cell on the device after every
        # iteration (fib_probe_watch: a node of the iteration's CUDA graph) and reads the ring back once
        # per `probe_batch` iterations -- no host round trip per iteration.
        owner = self._row0 <= prow < self._row0 + self._rows
        ring = watch and not im and owner
        batch = max(1, min(int(self.__dict__.get('probe_batch', 64)), _capi.PROBE_RING // 2))
        unread = []                                              # iterations recorded, not yet read

        def crossing(i, v1):
            nonlocal v0, last_spike
            if v1 >= 0.5 and v0 < 0.5:
                cl = (i - last_spike) * self.dt_per_step * self.dt
                if self.cl_observer is None:
                    print('wavefront reaches the middle top point at %d, cycle length is %d' % (i, cl))
                else:
                    self.cl_observer(i, cl)
                last_spike = i
            v0 = v1

        def drain(n):
            # the oldest n recorded iterations; the library waits only for the launch that produced
            # them, so the iterations stepped since keep the device busy meanwhile
            vals = self._ctx.probe_fetch(n) if n else []
            if len(vals) != n:
                raise RuntimeError('probe ring returned %d values for %d iterations' % (len(vals), n))
            w = self._probe_weight(prow, pcol)
            for k, raw in zip(unread[:n], vals):
                if k % plot_every == 0:
                    crossing(k, self._normalise(float(raw)) * w)
            del unread[:n]

        self._behind, self._behind_limit = 0, self._agree_on_upload_window(im, batch)
        self._upload_window_used = self._behind_limit
        if ring:
            self._ctx.probe_watch(self._pot_name, prow, pcol)
        try:
            for i in range(self.samples):
                if i < self._behind_limit:
                    self._behind += 1                        # runs behind the upload: see the _ctx property
                    if self._behind == self._behind_limit:
                        self._ctx                            # noqa: B018 (the window is full: go)
                else:
                    self._ctx.step(self.ode_op(i), 1)
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
                self._ctx.probe_watch(self._pot_name, -1, -1)
        if keep_state:                                           # ionic.py:226-229
            self.state = {}
            for s in self._State:
                self.state[s] = self._State[s].eval()
        if getattr(self, 'timeline', False):
            self._write_timeline()
        self._ctx.sync()
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
        with masked_image_mean().  Backs the pseudo-electrograms of the reference's egm.py."""
        if not self.defined:
            raise AssertionError('add_probe_mask should be called after calling define')
        slot = len(self.__dict__.setdefault('_mask_slots', []))
        m = np.asarray(mask, dtype=np.float32)
        self._ctx.set_weights(slot, m[self._row0:self._row0 + self._rows], self._row0)
        self._mask_slots.append(slot)
        return slot

    def masked_image_mean(self, slot):
        """np.mean(self.image() * mask) (egm.py:44-47) without moving the frame to the host:
        one weighted reduction on the device (summed over ranks when sharded)."""
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

    def sync(self):
        self._ctx.sync()

    def close(self):
        if self._ctx is not None:
            self._ctx.close()
            self._ctx = None
