"""CPU: the JSON-line contract of `bench.py --impl reference` (the arm the driver runs on the GPU
box's host cores): every key of the base contract, the reference-arm additions, one line, and --
under a multi-rank launch -- silence from every rank but 0.  The timed thing here is the oracle's
C/OpenMP port (test infrastructure), which is exactly what that arm is allowed to execute."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEED = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better',
        'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'cpu_baseline', 'impl']


def run(env_extra, *args):
    env = dict(os.environ, **env_extra)
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference'] + list(args),
                       capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    return [l for l in p.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_contract_line():
    lines = run({}, '--steps', '1', '--warmup', '1')
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert [k for k in NEED if k not in d] == []
    assert d['impl'] == 'reference' and d['metric'] == d['unit'] == 'Gcell-steps/s'
    assert d['steps'] == 1 and d['n_gpus'] == 1 and d['higher_is_better'] is True
    assert d['value'] > 0 and d['dtype'] == 'f32' and d['vs_baseline'] is None
    assert 'workload' in d['config'] and '32768' in d['config']['workload']
    cb, e2e = d['cpu_baseline'], d['e2e']
    assert cb['kind'] in ('port', 'reference') and cb['cores'] >= 1 and cb['sample']
    assert cb['value'] == d['value'] == e2e['value'] and e2e['unit'] == d['unit']
    assert e2e['h2d_bytes_per_step'] == 0 and e2e['d2h_bytes_per_step'] == 0


def test_reference_arm_is_rank0_only_under_a_multi_rank_launch():
    lines = run({'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2'}, '--gpus', '2', '--steps', '1', '--warmup', '1')
    assert lines == []


import pytest  # noqa: E402


@pytest.mark.gpu
def test_our_arm_prints_one_contract_line(cuda_device, tmp_path):
    """`python bench.py` at a reduced grid (4096^2, still >> L2): one JSON line with every key of
    the contract, the device-timed value consistent with ms_per_step, a non-trivial e2e leg,
    kernels of this library launched inside the timed region, and the --dump-outputs sample."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--size', '4096', '--steps', '3',
                        '--warmup', '3', '--no-cpu', '--no-suite', '--dump-outputs', str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    # (--no-cpu skips the 20-second cpu_baseline leg; the CPU test above covers that object)
    need = [k for k in NEED if k not in ('impl', 'cpu_baseline')] + ['gpu_launches', 'clocks', 'roofline']
    assert [k for k in need if k not in d] == []
    cells = 4096.0 * 4096.0
    assert abs(d['value'] - cells * 10 / (d['ms_per_step'] * 1e-3) / 1e9) <= 1e-6 * d['value']
    assert d['steps'] == 3 and d['warmup'] == 3 and d['n_gpus'] == 1
    spl = d['config']['time_steps_per_launch']
    assert d['gpu_launches'] == 3 * 10 // spl
    r = d['roofline']
    assert r['bound'] == 'hbm' and r['unit'] == 'GB/s' and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    assert abs(r['achieved'] - 32.0 * d['value']) <= 1e-6 * r['achieved']      # 32 B per cell-step
    e = d['e2e']
    assert 0 < e['value'] < d['value'] and e['h2d_bytes_per_step'] > 0 and e['d2h_bytes_per_step'] > 0
    assert d['clocks']['sm_mhz'] > 0
    rows = np.load(str(tmp_path / 'rows.npy'))
    assert rows.dtype == np.float64 and len(rows) == 64 and np.all(np.diff(rows) > 0)
    for v in ('U', 'V', 'W', 'S'):
        a = np.load(str(tmp_path / (v + '.npy')))
        assert a.dtype == np.float32 and a.shape == (64, 4096) and np.isfinite(a).all(), v
    assert sum(f.stat().st_size for f in tmp_path.iterdir()) <= 64 << 20
