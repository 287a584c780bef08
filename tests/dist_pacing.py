"""torchrun --nproc-per-node N tests/dist_pacing.py : NCCL row-sharded pacing (IonicModel.pace) must leave every
plane BIT-IDENTICAL to the unsharded run that rank 0 performs on its own GPU with fire_op at the same iterations --
4v (one and two time steps per launch), Beeler-Reuter and Courtemanche, with a phase field and a rectangle whose
rows cross every seam, fired inside one multi-iteration fib_step call."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    from cuda_adapter import CLASSES
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank, world = dist.get_rank(), dist.get_world_size()
    base = {'width': 200, 'height': 40 * world + 11, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.1, 'duration': 1,
            'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False,
            'cheby': False, 'ultra_slow': False}
    ok = True
    for kind, extra, iters in (('fenton4v', {}, 40), ('fenton4v', {'steps_per_launch': 2}, 40),
                               ('br', {'cheby': True, 'skip': True}, 40), ('court_ultra', {}, 60)):
        cfg = dict(base, **extra)
        models = [CLASSES[kind](dict(cfg, distributed=True, device=local))]
        if rank == 0:
            models.append(CLASSES[kind](dict(cfg, device=local, persist=False)))
        beats = [5, 12, 19, 26]
        for m in models:
            m.add_hole_to_phase_field(90, 60, 17)
            m.define()
            m._ops['band'] = ('pace', (3, cfg['height'] - 3, 60, 120), float(m.max_v))
        models[0].pace('band', beats[0], 7, len(beats))
        for start in range(0, iters, 10):              # the beats fall inside fib_step(10) calls
            models[0]._ctx.step(models[0].ode_op(start), 10)
            models[0].iterations += 10
            if rank == 0:
                m = models[1]
                for i in range(start, start + 10):
                    m._ctx.step(m.ode_op(i), 1)
                    if i in beats:
                        m.fire_op('band')
        planes = {v: models[0]._State[v].eval() for v in models[0]._ctx.var_names}   # collective
        if rank == 0:
            same = all(np.array_equal(planes[v].view(np.uint32), models[1]._ctx.get_state(v).view(np.uint32))
                       for v in planes)
            ok &= same
            print('%-12s %s, %d ranks: sharded pacing == unsharded fire_op: %s' % (kind, extra, world, same), flush=True)
        for m in models:
            m.close()
    flag = torch.tensor([1 if ok else 0], device='cuda')
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    if not flag.item():
        sys.exit(1)
    if rank == 0:
        print('DIST PACING OK')


if __name__ == '__main__':
    main()
