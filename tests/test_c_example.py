"""The C-ABI boundary used from plain C (examples/c_driver.c): it compiles and links against
libfibb200.so with nothing but the header; without a GPU it fails loudly (exit 2, CUDA message);
on a GPU its result equals the Python drop-in's."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT


def build(tmp_path):
    exe = str(tmp_path / 'c_driver')
    lib = os.path.join(ROOT, 'fib_tf_b200')
    subprocess.check_call(['gcc', '-O2', '-Wall', '-Werror', '-I' + os.path.join(ROOT, 'include'),
                           os.path.join(ROOT, 'examples', 'c_driver.c'), '-L' + lib, '-lfibb200',
                           '-Wl,-rpath,' + lib, '-o', exe])
    return exe


def test_c_example_builds_and_fails_loudly_without_gpu(tmp_path):
    exe = build(tmp_path)
    # (on a GPU machine the devices are hidden from the child)
    r = subprocess.run([exe, '64', '2'], capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))
    assert r.returncode == 2 and 'fib_create' in r.stderr and 'CUDA' in r.stderr


@pytest.mark.gpu
def test_c_example_matches_the_python_drop_in(cuda_device, tmp_path):
    from fib_tf_b200.fenton import Fenton4v
    exe = build(tmp_path)
    out = subprocess.run([exe, '192', '40'], capture_output=True, text=True, check=True).stdout
    fields = dict(kv.split('=') for kv in out.split())
    m = Fenton4v({'width': 192, 'height': 192, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 40,
                  'timeline': False, 'timeline_name': 'x', 'save_graph': False})
    m.define()
    m.add_pace_op('s2', 'luq', 1.0)
    for i in m.run(None):
        if i == 20:
            m.fire_op('s2')
    u = m.image()
    # 192^2 runs as the persistent on-chip kernel, iterations deferred until something looks: the 21
    # before the stimulus are one launch, the 19 after it another (+ the stimulus)
    assert int(fields['kernels']) == 2 + 1
    assert float(fields['probe']) == pytest.approx(float(u[20, 96]), abs=1e-6)
    assert float(fields['sum(U)']) == pytest.approx(float(np.sum(u, dtype=np.float64)), rel=1e-9)
    m.close()
