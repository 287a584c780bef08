"""torchrun --nproc-per-node N tests/dist_frames.py : NCCL row-sharded frames, gathered by IonicModel.frames(), must
be BIT-IDENTICAL to the frames of the unsharded run that rank 0 performs on its own GPU -- 4v (one and two time
steps per launch), Beeler-Reuter and Courtemanche, with a phase field, a stimulus between iterations and a
stride that does not divide the shard heights."""
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
    for kind, extra, iters, stride in (('fenton4v', {}, 40, 3), ('fenton4v', {'steps_per_launch': 2}, 40, 1),
                                       ('br', {'cheby': True, 'skip': True}, 40, 7), ('court_ultra', {}, 60, 3)):
        cfg = dict(base, **extra)
        models = [CLASSES[kind](dict(cfg, distributed=True, device=local))]
        if rank == 0:
            models.append(CLASSES[kind](dict(cfg, device=local, persist=False)))
        for m in models:
            m.add_hole_to_phase_field(90, 60, 17)
            m.define()
            m.add_pace_op('s2', 'luq', float(m.max_v))
            m.record_frames(4, stride=stride, first=0)
        for i in range(iters):
            for m in models:
                m._ctx.step(m.ode_op(i), 1)
                if i == iters // 2:
                    m.fire_op('s2')
        got_k, got = models[0].frames()                    # gathered over the ranks (collective)
        if rank == 0:
            want_k, want = models[1].frames()
            same = list(got_k) == list(want_k) and got.shape == want.shape and \
                np.array_equal(got.view(np.uint32), want.view(np.uint32))
            ok &= same
            print('%-12s %s stride %d, %d ranks: sharded frames == unsharded: %s' % (kind, extra, stride, world, same),
                  flush=True)
        for m in models:
            m.close()
    flag = torch.tensor([1 if ok else 0], device='cuda')
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    if not flag.item():
        sys.exit(1)
    if rank == 0:
        print('DIST FRAMES OK')


if __name__ == '__main__':
    main()
