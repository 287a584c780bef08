"""The march of the two-steps-per-launch 4v kernel (csrc/fib_fused.cuh) against one step per launch, bit
for bit, on the geometries that pick its code paths.

A warp marches its output rows [g0, g1).  The trips j in [max(g0 + 1, 3), min(g1 - 2, H - 3)] of a warp
whose columns need no clamp run through the interior body, unrolled by three; the remainder modulo 3,
the first and last trips (which would prefetch beyond the march), the border rows and the edge warps run
through the general body.  On grids that fill at most one wave, launch_fused2 gives every warp R = 8
output rows: an inner warp has 6 interior trips (0 mod 3), the first warp of the grid 4 (1 mod 3), and the
last warp of a grid with H = 8 m + k rows has k - 4, so k = 6, 7, 8 give 2, 0, 1 mod 3 and k = 1 a last
warp of a single row.  At 4096^2 on 148 SMs R = 25 without the phase field (23 interior trips, 2 mod 3)
and R = 32 with it.
A warp owns 128 columns, lanes 1..30 of it 120 output columns: W mod 120 = 4, 8 and 116 make the last
warp partially valid, W <= 128 leaves no warp without a clamp, H = 5 no interior row.  Row shards put
a seam inside a warp's march, and 4096^2 runs long marches."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def cuda(cuda_device):
    import cuda_adapter
    return cuda_adapter


GRIDS = [
    (38, 484, 1),      # last warp k = 6: interior trips 2 mod 3; W mod 120 = 4
    (63, 488, 1),      # k = 7: 0 mod 3; W mod 120 = 8
    (64, 476, 1),      # k = 8: 1 mod 3; W mod 120 = 116
    (41, 484, 1),      # k = 1: a last warp with a single row
    (5, 484, 1),       # no interior row
    (70, 128, 1),      # no warp without the column clamp
    (64, 124, 2),
    (203, 716, 3),     # row shards of 68 / 68 / 67 rows: seams inside a warp's march
    (130, 476, 2),
    (4096, 4096, 1),   # long marches
]


@pytest.mark.parametrize('phase_field', [False, True])
@pytest.mark.parametrize('H,W,nshards', GRIDS)
def test_fused_march_matches_one_step_launches(cuda, H, W, nshards, phase_field):
    from fib_tf_b200 import _capi
    from fib_tf_b200.sharding import partition_rows
    dt, diff = 0.1, 1.5
    rng = np.random.default_rng(H * 7919 + W)
    init = {v: rng.uniform(0.0, 1.0, (H, W)).astype(np.float32) for v in 'UVWS'}
    init['U'][H // 4:H // 2 + 1, W // 3:W // 2] = 0.95

    phase = None
    if phase_field:
        yy, xx = np.mgrid[0:H, 0:W]
        phase = np.ones((H, W))
        # one hole inside, one across the top border and the right edge warps
        for cy, cx, rad in ((H / 2.0, W / 3.0, max(min(H, W) / 6.0, 1.0)), (0.0, W - 6.0, max(min(H, W) / 5.0, 2.0))):
            phase *= 0.5 * (np.tanh(np.hypot(yy - cy, xx - cx) - rad) + 1.0)
        phase = np.maximum(phase, 1e-5).astype(np.float32)

    def make(steps_per_launch, parts=((0, 0),)):
        out = [_capi.Context(_capi.FENTON4V, H, W, dt, diff, flags=_capi.F_NO_GRAPH, row0=r0, rows=n,
                             steps_per_launch=steps_per_launch) for r0, n in parts]
        for s, (r0, n) in zip(out, parts):
            for v, a in init.items():
                s.set_state(v, a if n == 0 else a[r0:r0 + n])
            if phase is not None:
                s.set_phase(phase, 0)
        return out

    ref, = make(1)
    if nshards > 1:
        fused = make(2, parts=partition_rows(H, nshards))
        step = lambda: _capi.step_group(fused, _capi.OP_ODE, 1)
    else:
        fused = make(2)
        step = lambda: fused[0].step(_capi.OP_ODE, 1)
    for _ in range(4):
        ref.step(_capi.OP_ODE, 1)
        step()
    for v in ref.var_names:
        want = ref.get_state(v)
        assert np.isfinite(want).all(), v
        got = np.concatenate([s.get_state(v) for s in fused], axis=0)
        assert np.array_equal(got, want), v
    for c in [ref] + fused:
        c.close()
