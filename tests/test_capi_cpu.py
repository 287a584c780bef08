"""CPU: the C-ABI library loads, exports every symbol include/fib_b200.h declares, validates its
arguments, and fails LOUDLY without a GPU (no CPU fallback).  No compute calls here."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from fib_tf_b200 import _capi


def header_symbols():
    text = open(os.path.join(ROOT, 'include', 'fib_b200.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(fib_[a-z_0-9]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    L = _capi.lib()
    names = header_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(L, n), 'libfibb200.so does not export %s' % n
    assert sorted(_capi.EXPORTS) == names, 'ctypes binding and header disagree'
    assert L.fib_version() == _capi.ABI_VERSION


def test_config_struct_matches_header_layout():
    # uint32, int32 x3, double x2, uint32, int32 x4, int32[6]
    assert C.sizeof(_capi.FibConfig) == 4 * 4 + 2 * 8 + 4 * 5 + 4 * 6 + 4   # +4: tail padding to 8
    assert _capi.FibConfig.dt.offset == 16 and _capi.FibConfig.flags.offset == 32


def _cfg(**kw):
    cfg = _capi.FibConfig()
    cfg.struct_size = C.sizeof(_capi.FibConfig)
    cfg.model, cfg.height, cfg.width, cfg.dt, cfg.diff = 0, 16, 16, 0.1, 1.0
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


@pytest.mark.parametrize('kw,needle', [
    (dict(struct_size=8), 'struct_size'),
    (dict(model=9), 'unknown model'),
    (dict(height=2), 'too small'),
    (dict(dt=0.0), 'dt must be'),
    (dict(steps_per_launch=3), 'steps_per_launch'),
    (dict(steps_per_launch=2, model=1), 'steps_per_launch=2 needs'),       # 4v only
    (dict(steps_per_launch=2, width=66), 'steps_per_launch=2 needs'),      # width % 4
    (dict(steps_per_launch=2, row0=10, rows=1), 'at least 2 rows'),
    (dict(row0=10, rows=10), 'outside the grid'),
    (dict(height=70000, width=40000), '2^31'),      # 32-bit element offsets: shard the grid instead
])
def test_create_rejects_bad_arguments(kw, needle):
    L = _capi.lib()
    h = C.c_void_p()
    rc = L.fib_create(C.byref(_cfg(**kw)), C.byref(h))
    assert rc == -1
    assert needle in L.fib_last_error().decode()


def test_null_arguments_are_errors_not_crashes():
    L = _capi.lib()
    assert L.fib_create(None, None) == -1
    assert L.fib_step(None, 0, 1) == -1
    assert L.fib_sync(None) == -1
    assert L.fib_destroy(None) == 0
    # the round-2 entry points: a NULL context is an argument error before any CUDA call
    n = C.c_size_t()
    u = C.c_uint64()
    assert L.fib_flush(None) == -1
    assert L.fib_probe_watch(None, 0, 1, 1) == -1
    assert L.fib_probe_fetch(None, None, 0, C.byref(n)) == -1
    assert L.fib_count_below(None, 0, 0.0, 1.0, 0.2, 1e-3, C.byref(u), C.byref(u)) == -1
    assert L.fib_set_rect_async(None, 0, 0, 1, 0, 1, None) == -1
    assert 'NULL' in L.fib_last_error().decode()


NO_GPU_CHILD = '''
import pytest
from fib_tf_b200 import _capi
with pytest.raises(_capi.FibError) as e:
    _capi.Context(_capi.FENTON4V, 16, 16, 0.1, 1.0)
assert 'cuda' in str(e.value).lower()
from fib_tf_b200.fenton import Fenton4v
m = Fenton4v({'width': 16, 'height': 16, 'dt': 0.1, 'diff': 1.0, 'duration': 1, 'dt_per_plot': 10})
with pytest.raises(_capi.FibError):
    m.define()
'''


def test_no_cpu_fallback_without_gpu():
    """In a child process that sees no GPU (on a GPU machine the devices are hidden from it)."""
    r = subprocess.run([sys.executable, '-c', NO_GPU_CHILD], cwd=ROOT, capture_output=True, text=True,
                       timeout=300, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))
    assert r.returncode == 0, r.stderr[-2000:]


def test_product_never_imports_the_oracle_or_tensorflow():
    pkg = os.path.join(ROOT, 'fib_tf_b200')
    bad = re.compile(r'^\s*(from|import)\s+(oracle|tensorflow|triton|jax)\b|#include\s+"[^"]*oracle', re.M)
    for dirpath, _d, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert not bad.search(src), '%s pulls in the oracle / a forbidden framework' % f
