"""
ctypes binding of libfibb200.so (include/fib_b200.h) -- the only way the Python host code
reaches the GPU.  There is no CPU fallback: if the shared library is missing or no CUDA device
is usable, importing / creating a context fails loudly.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# FIB_B200_LIB selects another build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get('FIB_B200_LIB') or os.path.join(_HERE, 'libfibb200.so')

# model ids / flags / ops / tables: keep in sync with include/fib_b200.h
FENTON4V, BR, COURT, COURT_ULTRA = 0, 1, 2, 3
F_CHEBY, F_SKIP, F_LUT, F_ULTRA_SLOW, F_NO_CHRONIC, F_NO_GRAPH = 0x01, 0x02, 0x04, 0x08, 0x10, 0x20
F_NO_CLIP = 0x40
F_CHEBY_STRICT, F_NO_PERSIST = 0x80, 0x100
PROBE_RING = 4096
OP_ODE, OP_SLOW = 0, 1
TABLE_BR_CHEBY, TABLE_COURT_LUT = 0, 1
ACT_FIRST, ACT_LAST, ACT_PREV, ACT_REPOL, ACT_COUNT = 0, 1, 2, 3, 4
ABI_VERSION = 3
INTER_COLS = 32

# courtemanche.h:105-134 column order (+ the two court_ultra.py:445-450 extras)
INTER_NAMES = (
    'd_infinity', 'f_infinity', 'tau_w', 'tau_d', 'tau_f', 'w_infinity', 'm_inf', 'h_inf', 'j_inf',
    'tau_oa', 'tau_oi', 'tau_ua', 'tau_ui', 'tau_xr', 'tau_xs', 'tau_m', 'tau_h', 'tau_j',
    'oa_infinity', 'oi_infinity', 'ua_infinity', 'ui_infinity', 'xr_infinity', 'xs_infinity',
    'g_Kur', 'f_NaK', 'i_NaCaa', 'i_NaCab', 'i_K1a', 'i_Kra', 'us_infinity', 'tau_us')


class FibError(RuntimeError):
    pass


class FibConfig(C.Structure):
    _fields_ = [
        ('struct_size', C.c_uint32), ('model', C.c_int32),
        ('height', C.c_int32), ('width', C.c_int32),
        ('dt', C.c_double), ('diff', C.c_double),
        ('flags', C.c_uint32), ('device', C.c_int32),
        ('row0', C.c_int32), ('rows', C.c_int32),
        ('steps_per_launch', C.c_int32), ('reserved', C.c_int32 * 6),
    ]


_P = C.c_void_p
_FP = C.POINTER(C.c_float)
_SIGNATURES = {
    'fib_version': (C.c_int, []),
    'fib_last_error': (C.c_char_p, []),
    'fib_device_count': (C.c_int, [C.POINTER(C.c_int)]),
    'fib_create': (C.c_int, [C.POINTER(FibConfig), C.POINTER(_P)]),
    'fib_destroy': (C.c_int, [_P]),
    'fib_num_vars': (C.c_int, [_P]),
    'fib_var_name': (C.c_char_p, [_P, C.c_int]),
    'fib_var_index': (C.c_int, [_P, C.c_char_p]),
    'fib_dt_per_step': (C.c_int, [_P]),
    'fib_set_state': (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    'fib_get_state': (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    'fib_get_rect': (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    'fib_snapshot_begin': (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    'fib_snapshot_wait': (C.c_int, [_P]),
    'fib_set_rect': (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    'fib_set_rect_async': (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _P]),
    'fib_last_kernel': (C.c_int, [C.c_char_p, C.c_size_t]),
    'fib_probe_watch': (C.c_int, [_P, C.c_int, C.c_int, C.c_int]),
    'fib_probe_fetch': (C.c_int, [_P, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    'fib_activation_watch': (C.c_int, [_P, C.c_float, C.c_float]),
    'fib_activation_stop': (C.c_int, [_P]),
    'fib_activation_get': (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    'fib_count_below': (C.c_int, [_P, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float,
                                  C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    'fib_op_enforce_boundary': (C.c_int, [C.c_int, _P, C.c_int, C.c_int, _P]),
    'fib_op_laplace': (C.c_int, [C.c_int, _P, _P, C.c_int, C.c_int, C.c_int, _P]),
    'fib_op_rush_larsen': (C.c_int, [C.c_int, _P, _P, _P, C.c_size_t, C.c_float, C.c_int, _P]),
    'fib_set_phase': (C.c_int, [_P, _P, C.c_int, C.c_int]),
    'fib_set_table': (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    'fib_get_table': (C.c_int, [_P, C.c_int, _P, C.c_size_t]),
    'fib_build_lut': (C.c_int, [_P]),
    'fib_court_inter': (C.c_int, [_P, _P, C.c_size_t, _P]),
    'fib_step': (C.c_int, [_P, C.c_int, C.c_int]),
    'fib_step_group': (C.c_int, [C.POINTER(_P), C.c_int, C.c_int, C.c_int]),
    'fib_stimulate': (C.c_int, [_P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float]),
    'fib_probe': (C.c_int, [_P, C.c_int, C.c_int, C.c_int, _FP]),
    'fib_weighted_sum': (C.c_int, [_P, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    'fib_count_nonfinite': (C.c_int, [_P, C.c_int, C.POINTER(C.c_uint64)]),
    'fib_set_weights': (C.c_int, [_P, C.c_int, _P, C.c_int, C.c_int]),
    'fib_masked_sum': (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    'fib_sync': (C.c_int, [_P]),
    'fib_flush': (C.c_int, [_P]),
    'fib_upload_state': (C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'fib_step_behind_upload': (C.c_int, [_P, C.c_int]),
    'fib_timer_start': (C.c_int, [_P]),
    'fib_timer_stop': (C.c_int, [_P]),
    'fib_timer_ms': (C.c_int, [_P, _FP]),
    'fib_launch_count': (C.c_int, [_P, C.POINTER(C.c_uint64)]),
    'fib_stream': (C.c_int, [_P, C.POINTER(_P)]),
    'fib_host_alloc': (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    'fib_host_free': (C.c_int, [_P]),
    'fib_comm_unique_id': (C.c_int, [_P]),
    'fib_comm_init': (C.c_int, [_P, C.c_int, C.c_int, _P]),
}
EXPORTS = tuple(sorted(_SIGNATURES))

_lib = None


def lib():
    """The loaded shared library (loaded once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FibError(
                '%s is missing: build it with `python -m fib_tf_b200.build` (nvcc, sm_100a). '
                'fib_tf_b200 has no CPU fallback.' % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        if L.fib_version() != ABI_VERSION:
            raise FibError('libfibb200.so ABI %d != binding ABI %d' % (L.fib_version(), ABI_VERSION))
        _lib = L
    return _lib


def check(rc):
    if rc < 0:
        raise FibError(lib().fib_last_error().decode('utf-8', 'replace'))
    return rc


def _f32c(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(_P)


def pinned_empty(shape, dtype=np.float32):
    """A NumPy array backed by page-locked host memory (fib_host_alloc)."""
    n = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = _P()
    check(lib().fib_host_alloc(max(n, 1), C.byref(p)))
    buf = (C.c_char * max(n, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[arr.ctypes.data] = p
    return arr


_PINNED = {}


def pinned_free(arr):
    p = _PINNED.pop(arr.ctypes.data, None)
    if p is not None:
        check(lib().fib_host_free(p))


class Context:
    """One shard of one model on one GPU (fib_ctx*)."""

    def __init__(self, model, height, width, dt, diff, flags=0, device=0, row0=0, rows=0,
                 steps_per_launch=0):
        L = lib()
        cfg = FibConfig()
        cfg.struct_size = C.sizeof(FibConfig)
        cfg.model, cfg.height, cfg.width = int(model), int(height), int(width)
        cfg.dt, cfg.diff, cfg.flags, cfg.device = float(dt), float(diff), int(flags), int(device)
        cfg.row0, cfg.rows, cfg.steps_per_launch = int(row0), int(rows), int(steps_per_launch)
        h = _P()
        check(L.fib_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.height, self.width = int(height), int(width)
        self.row0 = int(row0) if rows else 0
        self.rows = int(rows) if rows else int(height)
        self.nvars = L.fib_num_vars(h)
        self.var_names = [L.fib_var_name(h, i).decode() for i in range(self.nvars)]
        self.dt_per_step = L.fib_dt_per_step(h)

    # -- life cycle
    def close(self):
        if getattr(self, '_h', None):
            lib().fib_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def var(self, name_or_index):
        if isinstance(name_or_index, str):
            return check(lib().fib_var_index(self._h, name_or_index.encode()))
        return int(name_or_index)

    # -- state
    def set_state(self, var, host):
        a, p = _f32c(host)
        if a.shape != (self.rows, self.width):
            raise FibError('set_state: array shape %r != shard shape %r' % (a.shape, (self.rows, self.width)))
        check(lib().fib_set_state(self._h, self.var(var), p, a.size))

    def get_state(self, var, out=None):
        if out is None:
            out = np.empty((self.rows, self.width), dtype=np.float32)
        elif (not isinstance(out, np.ndarray) or out.dtype != np.float32 or not out.flags['C_CONTIGUOUS']
              or not out.flags['WRITEABLE'] or out.shape != (self.rows, self.width)):
            raise FibError('get_state: `out` must be a writeable C-contiguous float32 array of shape %r'
                           % ((self.rows, self.width),))
        check(lib().fib_get_state(self._h, self.var(var), out.ctypes.data_as(_P), out.size))
        return out

    def snapshot_begin(self, var, pinned_out):
        """Asynchronous read of a plane into a pinned array (see pinned_empty); overlaps with the
        steps enqueued afterwards.  snapshot_wait() completes it."""
        if pinned_out.dtype != np.float32 or not pinned_out.flags['C_CONTIGUOUS']:
            raise FibError('snapshot target must be a C-contiguous float32 array')
        if pinned_out.shape != (self.rows, self.width):
            raise FibError('snapshot target must have the shard shape %r' % ((self.rows, self.width),))
        # (that the memory is page-locked is checked by the library: cudaPointerGetAttributes)
        check(lib().fib_snapshot_begin(self._h, self.var(var), pinned_out.ctypes.data_as(_P),
                                       pinned_out.size))

    def snapshot_wait(self):
        check(lib().fib_snapshot_wait(self._h))

    def get_rect(self, var, r0, r1, c0, c1):
        out = np.empty((r1 - r0, c1 - c0), dtype=np.float32)
        check(lib().fib_get_rect(self._h, self.var(var), r0, r1, c0, c1, out.ctypes.data_as(_P)))
        return out

    def set_rect(self, var, r0, c0, block):
        a, p = _f32c(block)
        check(lib().fib_set_rect(self._h, self.var(var), r0, r0 + a.shape[0], c0, c0 + a.shape[1], p))

    def set_rect_async(self, var, r0, c0, pinned_block):
        """Enqueue-only upload of a block that lives in page-locked memory (pinned_empty); the block
        must stay unchanged until the next sync()."""
        a = pinned_block
        if a.dtype != np.float32 or not a.flags['C_CONTIGUOUS'] or a.ndim != 2:
            raise FibError('set_rect_async: the block must be a 2-D C-contiguous float32 array')
        check(lib().fib_set_rect_async(self._h, self.var(var), r0, r0 + a.shape[0], c0, c0 + a.shape[1],
                                       a.ctypes.data_as(_P)))

    def set_phase(self, phase_rows, first_row=0):
        if phase_rows is None:
            check(lib().fib_set_phase(self._h, None, 0, 0))
            return
        a, p = _f32c(phase_rows)
        check(lib().fib_set_phase(self._h, p, int(first_row), a.shape[0]))

    def set_table(self, table, data):
        a, p = _f32c(data)
        check(lib().fib_set_table(self._h, table, p, a.size))

    def get_table(self, table, shape):
        out = np.empty(shape, dtype=np.float32)
        check(lib().fib_get_table(self._h, table, out.ctypes.data_as(_P), out.size))
        return out

    def build_lut(self):
        check(lib().fib_build_lut(self._h))

    def court_inter(self, v):
        a, p = _f32c(np.asarray(v, dtype=np.float32).ravel())
        out = np.empty((a.size, INTER_COLS), dtype=np.float32)
        check(lib().fib_court_inter(self._h, p, a.size, out.ctypes.data_as(_P)))
        return out

    # -- stepping
    def step(self, op=OP_ODE, n_iter=1):
        check(lib().fib_step(self._h, op, n_iter))

    def stimulate(self, var, r0, r1, c0, c1, value, floor_v):
        check(lib().fib_stimulate(self._h, self.var(var), r0, r1, c0, c1, value, floor_v))

    def probe(self, var, row, col):
        v = C.c_float()
        check(lib().fib_probe(self._h, self.var(var), row, col, C.byref(v)))
        return np.float32(v.value)

    def probe_watch(self, var, row, col):
        """Record cell (row, col) of `var` into the device ring after every iteration (row < 0: stop)."""
        check(lib().fib_probe_watch(self._h, self.var(var) if row >= 0 else 0, row, col))

    def probe_fetch(self, max_values=PROBE_RING):
        out = np.empty(max_values, dtype=np.float32)
        n = C.c_size_t()
        check(lib().fib_probe_fetch(self._h, out.ctypes.data_as(_P), max_values, C.byref(n)))
        return out[:n.value]

    def activation_watch(self, up, down):
        """Arm (or re-arm) the activation maps of the diffusing variable at levels up / down."""
        check(lib().fib_activation_watch(self._h, up, down))

    def activation_stop(self):
        check(lib().fib_activation_stop(self._h))

    def activation_get(self, which):
        """[rows, W] float32 map ACT_* of this shard, times in iterations since arming."""
        out = np.empty((self.rows, self.width), dtype=np.float32)
        check(lib().fib_activation_get(self._h, which, out.ctypes.data_as(_P), out.size))
        return out

    def count_below(self, var, sub, div, cutoff, w_min):
        a, b = C.c_uint64(), C.c_uint64()
        check(lib().fib_count_below(self._h, self.var(var), sub, div, cutoff, w_min, C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def weighted_sum(self, var):
        a, b = C.c_double(), C.c_double()
        check(lib().fib_weighted_sum(self._h, self.var(var), C.byref(a), C.byref(b)))
        return a.value, b.value

    def count_nonfinite(self, var):
        v = C.c_uint64()
        check(lib().fib_count_nonfinite(self._h, self.var(var), C.byref(v)))
        return int(v.value)

    def set_weights(self, slot, rows, first_row=0):
        a, p = _f32c(rows)
        check(lib().fib_set_weights(self._h, slot, p, int(first_row), a.shape[0]))

    def masked_sum(self, var, slot):
        a, b = C.c_double(), C.c_double()
        check(lib().fib_masked_sum(self._h, self.var(var), slot, C.byref(a), C.byref(b)))
        return a.value, b.value

    def sync(self):
        check(lib().fib_sync(self._h))

    def flush(self):
        """Launch the iterations the persistent path has deferred (enqueue only)."""
        check(lib().fib_flush(self._h))

    def upload_state(self):
        """(open, complete, direction, max_iters) of the pipelined upload in flight (set_rect_async)."""
        a, b, d, m = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        check(lib().fib_upload_state(self._h, C.byref(a), C.byref(b), C.byref(d), C.byref(m)))
        return bool(a.value), bool(b.value), d.value, m.value

    def step_behind_upload(self, n_iter):
        """n_iter ODE iterations behind a complete pipelined upload; collective on NCCL shards."""
        check(lib().fib_step_behind_upload(self._h, int(n_iter)))

    def timer_start(self):
        check(lib().fib_timer_start(self._h))

    def timer_stop(self):
        check(lib().fib_timer_stop(self._h))

    def timer_ms(self):
        v = C.c_float()
        check(lib().fib_timer_ms(self._h, C.byref(v)))
        return float(v.value)

    def launch_count(self):
        v = C.c_uint64()
        check(lib().fib_launch_count(self._h, C.byref(v)))
        return int(v.value)

    def stream(self):
        p = _P()
        check(lib().fib_stream(self._h, C.byref(p)))
        return p.value or 0

    def comm_init(self, nranks, rank, uid_bytes):
        buf = C.create_string_buffer(bytes(uid_bytes), 128)
        check(lib().fib_comm_init(self._h, nranks, rank, buf))


def comm_unique_id():
    buf = C.create_string_buffer(128)
    check(lib().fib_comm_unique_id(buf))
    return buf.raw


def step_group(contexts, op=OP_ODE, n_iter=1):
    arr = (_P * len(contexts))(*[c._h for c in contexts])
    check(lib().fib_step_group(arr, len(contexts), op, n_iter))


def last_kernel():
    """Name of the step-kernel flavour launched last by this thread (fib_last_kernel)."""
    buf = C.create_string_buffer(160)
    check(lib().fib_last_kernel(buf, 160))
    return buf.value.decode()


def _plane(a, name):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2:
        raise FibError('%s: expected a 2-D plane, got shape %r' % (name, a.shape))
    return a


def op_enforce_boundary(x, device=0):
    """IonicModel.enforce_boundary (ionic.py:107-113) on a dense [h, w] plane, on the device."""
    a = _plane(x, 'enforce_boundary')
    out = np.empty_like(a)
    check(lib().fib_op_enforce_boundary(device, a.ctypes.data_as(_P), a.shape[0], a.shape[1],
                                        out.ctypes.data_as(_P)))
    return out


def op_laplace(x, phase=None, mode=0, device=0):
    """IonicModel.laplace (ionic.py:44-60): mode 0 = REFLECT pad + 9-point stencil (+ phase term);
    mode 1 = the step kernels' collapsed index map on a raw plane = laplace(enforce_boundary(x));
    mode 2 = the phase-field term alone (ionic.py:70-81)."""
    a = _plane(x, 'laplace')
    ph = None
    if phase is not None:
        ph = _plane(phase, 'phase')
        if ph.shape != a.shape:
            raise FibError('laplace: phase shape %r != plane shape %r' % (ph.shape, a.shape))
    out = np.empty_like(a)
    check(lib().fib_op_laplace(device, a.ctypes.data_as(_P), ph.ctypes.data_as(_P) if ph is not None else None,
                               a.shape[0], a.shape[1], mode, out.ctypes.data_as(_P)))
    return out


def op_rush_larsen(g, g_inf, tau, dt, strict=False, device=0):
    """IonicModel.rush_larsen (ionic.py:115-123), elementwise on arrays of one shape."""
    g = np.ascontiguousarray(g, dtype=np.float32)
    gi = np.ascontiguousarray(np.broadcast_to(np.asarray(g_inf, np.float32), g.shape))
    t = np.ascontiguousarray(np.broadcast_to(np.asarray(tau, np.float32), g.shape))
    out = np.empty_like(g)
    check(lib().fib_op_rush_larsen(device, g.ctypes.data_as(_P), gi.ctypes.data_as(_P), t.ctypes.data_as(_P),
                                   g.size, float(dt), 1 if strict else 0, out.ctypes.data_as(_P)))
    return out


def device_count():
    n = C.c_int()
    check(lib().fib_device_count(C.byref(n)))
    return n.value
