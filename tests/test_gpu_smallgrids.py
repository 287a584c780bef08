"""GPU: tiny end-to-end run of EVERY kernel flavour (all models / flags, with and without a phase
field, stimuli, the slow op, reductions, sub-rectangle reads, an uneven in-process shard group) on
degenerate geometries (3x3, widths that are not multiples of the vector width).  compute-sanitizer
is closed on this pool, so bounds are exercised this way: every plane must stay finite and the
run must not fault."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from cuda_adapter import CudaModel  # noqa: E402
from fib_tf_b200 import _capi  # noqa: E402
from fib_tf_b200.sharding import partition_rows  # noqa: E402


@pytest.mark.gpu
def test_every_flavour_on_degenerate_grids(cuda_device):
    base = {'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.0, 'duration': 1, 'timeline': False,
            'timeline_name': 'x', 'save_graph': False, 'skip': False, 'cheby': False, 'ultra_slow': False}
    for (H, W) in ((3, 3), (7, 5), (33, 47), (40, 130)):
        for kind, extra in (('fenton4v', {}), ('br', {}), ('br', {'cheby': True, 'skip': True}),
                            ('court', {}), ('court', {'lut': True}), ('court_ultra', {'ultra_slow': True}),
                            ('court_ultra', {'lut': True}), ('court_ultra', {'lut': True, 'ultra_slow': True})):
            for hole in (False, True):
                cfg = dict(base, width=W, height=H, **extra)
                m = CudaModel(kind, cfg)
                if hole:
                    m.add_hole(W // 2, H // 2, max(min(H, W) // 4, 1))
                m.define()
                m.add_pace('a', 'luq', 1.0)
                m.add_pace('b', 'bottom', 1.0)
                for i in range(3):
                    m.iterate()
                    m.fire('slow') if kind.startswith('court') else None
                    m.fire('a' if i == 0 else 'b')
                for v in m.m._ctx.var_names:
                    assert np.isfinite(m.state[v]).all(), (kind, extra, H, W, hole, v)
                m.m._ctx.weighted_sum(m.m._ctx.var_names[0])
                m.m._ctx.get_rect(m.m._ctx.var_names[0], 0, 1, 0, W)
                m.close()
    # shard group with uneven shards
    H, W = 23, 37
    parts = partition_rows(H, 4)
    sh = [_capi.Context(_capi.BR, H, W, 0.1, 1.0, flags=_capi.F_NO_GRAPH, row0=r0, rows=n) for r0, n in parts]
    for s, (r0, n) in zip(sh, parts):
        for v in s.var_names:
            s.set_state(v, np.full([n, W], -80.0 if v == 'V' else 0.5, np.float32))
        s.set_phase(np.ones([H, W], np.float32), 0)
    _capi.step_group(sh, 0, 3)
    for s in sh:
        s.sync()
        s.close()



if __name__ == '__main__':
    test_every_flavour_on_degenerate_grids(0)
    print('small grids OK')
