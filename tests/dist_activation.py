"""torchrun --nproc-per-node N tests/dist_activation.py : NCCL row-sharded activation maps, gathered by
IonicModel.activation_maps(), must be BIT-IDENTICAL to the maps of the unsharded run that rank 0 performs on
its own GPU -- 4v (one and two time steps per launch), Beeler-Reuter and Courtemanche, with a phase field, a
perturbed band of the potential crossing the seams and a stimulus between iterations."""
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
        rng = np.random.default_rng(99)                     # the same band on every rank
        for m in models:
            m.add_hole_to_phase_field(90, 60, 17)
            m.define()
            m.add_pace_op('s2', 'luq', float(m.max_v))
        H, W = cfg['height'], cfg['width']
        lv = float(models[0].min_v) + 0.5 * (float(models[0].max_v) - float(models[0].min_v))
        band = (lv + 0.3 * (float(models[0].max_v) - float(models[0].min_v)) *
                rng.uniform(-1.0, 1.0, (H // 2, W))).astype(np.float32)
        for m in models:
            full = m._State[m._pot_name].eval()            # (collective for the sharded model)
            full[H // 4:H // 4 + H // 2] = band
            m._State[m._pot_name].assign(full)
            m.watch_activation()
        for i in range(iters):
            for m in models:
                m._ctx.step(m.ode_op(i), 1)
                if i == iters // 2:
                    m.fire_op('s2')
        got = models[0].activation_maps()                  # gathered over the ranks (collective)
        if rank == 0:
            want = models[1].activation_maps()
            for key in got:
                same = np.array_equal(got[key], want[key], equal_nan=True)
                ok &= same
                if not same:
                    print('MISMATCH %s %s %s' % (kind, extra, key))
            ok &= bool(np.nansum(want['count']) > 0)
            print('%-12s %s %d ranks: sharded maps == unsharded: %s' % (kind, extra, world, ok), flush=True)
        for m in models:
            m.close()
    flag = torch.tensor([1 if ok else 0], device='cuda')
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    if not flag.item():
        sys.exit(1)
    if rank == 0:
        print('DIST ACTIVATION OK')


if __name__ == '__main__':
    main()
