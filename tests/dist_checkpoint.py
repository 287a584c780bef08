"""torchrun --nproc-per-node N tests/dist_checkpoint.py : checkpoints across rank counts.  A checkpoint saved on N NCCL
shards (IonicModel.checkpoint / wait, collective) is restored by rank 0 alone, and one saved by rank 0 alone is
restored on N NCCL shards (their first iterations behind the pipelined upload, odd ranks uploading bottom to
top); both must continue BIT-IDENTICALLY to the uninterrupted unsharded run rank 0 performs on its own GPU."""
import os
import shutil
import sys
import tempfile

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def drive(m, n, slow):
    i0 = m.iterations
    m.duration = n * m.dt_per_step * m.dt * (1 + 1e-9)
    for i in m.run(None, block=False):
        if slow and (i0 + i) % 10 == 0:
            m.fire_op('slow')
        if i0 + i == 7:
            m.fire_op('s2')


def main():
    os.environ.setdefault('FIB_PIPELINE_MIN_CELLS', '0')
    os.environ.setdefault('FIB_PIPELINE_BLOCK_ROWS', '40')
    from cuda_adapter import CLASSES
    from fib_tf_b200 import checkpoint as ck
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    rank, world = dist.get_rank(), dist.get_world_size()
    box = [tempfile.mkdtemp(prefix='fib_ck_') if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    root = box[0]
    base = {'width': 200, 'height': 160 * world + 11, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.1, 'duration': 1,
            'timeline': False, 'timeline_name': 'x', 'save_graph': False, 'skip': False, 'cheby': False,
            'ultra_slow': False, 'upload_window': 5}
    ok = True
    for kind, extra, n, slow in (('fenton4v', {}, 12, False), ('fenton4v', {'steps_per_launch': 2}, 12, False),
                                 ('br', {'cheby': True, 'skip': True}, 12, False), ('court', {}, 25, True)):
        cfg = dict(base, **extra)

        def make(sharded):
            m = CLASSES[kind](dict(cfg, distributed=True, device=local) if sharded else dict(cfg, device=local))
            m.add_hole_to_phase_field(90, 60, 17)
            return m

        def start(m):
            m.define()
            m.add_pace_op('s2', 'luq', float(m.max_v))
            return m

        ref = None
        if rank == 0:
            ref = start(make(False))
            drive(ref, 2 * n, slow)
        # N shards save, rank 0 restores alone
        path = os.path.join(root, '%s_%d_sharded' % (kind, len(extra)))
        m = start(make(True))
        drive(m, n, slow)
        h = m.checkpoint(path)
        drive(m, n, slow)
        h.wait()
        m.close()
        # rank 0 saves alone, N shards restore
        path1 = os.path.join(root, '%s_%d_single' % (kind, len(extra)))
        if rank == 0:
            s = start(make(False))
            drive(s, n, slow)
            s.checkpoint(path1).wait()
            s.close()
        dist.barrier()
        r = make(True)
        r.restore(path1)
        r.add_pace_op('s2', 'luq', float(r.max_v))
        drive(r, n, slow)
        behind = r._upload_window_used
        got = {v: r._State[v].eval() for v in r._ctx.var_names}          # gathered (collective)
        r.close()
        if rank == 0:
            one = make(False)
            one.restore(path)
            one.add_pace_op('s2', 'luq', float(one.max_v))
            drive(one, n, slow)
            for v in ref._ctx.var_names:
                want = ref._ctx.get_state(v).view(np.uint32)
                a = np.array_equal(one._ctx.get_state(v).view(np.uint32), want)
                b = np.array_equal(got[v].view(np.uint32), want)
                ok &= a and b
                if not (a and b):
                    print('MISMATCH %s %s: %d shards -> 1: %s, 1 -> %d shards: %s' % (kind, v, world, a, world, b))
            print('%-12s %s: %d shards -> 1 and 1 -> %d shards (%d iterations behind the upload) == uninterrupted: %s'
                  % (kind, extra, world, world, behind, ok), flush=True)
            one.close()
            ref.close()
    flag = torch.tensor([1 if ok else 0], device='cuda')
    dist.broadcast(flag, 0)
    dist.barrier()
    if rank == 0:
        shutil.rmtree(root, ignore_errors=True)
    dist.destroy_process_group()
    if not flag.item():
        sys.exit(1)
    if rank == 0:
        print('DIST CHECKPOINT OK')


if __name__ == '__main__':
    main()
