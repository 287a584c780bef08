"""CPU: the host side of checkpoint / restart (fib_tf_b200/checkpoint.py, IonicModel.checkpoint / restore) against a
fake context that stages and reads its shard the way include/fib_b200.h fib_checkpoint_begin / _read / _end do,
and the new entry points' argument checks without a GPU."""
import ctypes as C
import json
import os

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from fib_tf_b200 import _capi
from fib_tf_b200 import checkpoint as ck
from fib_tf_b200.br import BeelerReuter
from fib_tf_b200.fenton import Fenton4v
from fib_tf_b200.sharding import partition_rows
from test_sharded_gloo import free_port

NAMES = {_capi.FENTON4V: ['U', 'V', 'W', 'S'], _capi.BR: ['V', 'C', 'M', 'H', 'J', 'D', 'F', 'XI']}
CFG = {'width': 24, 'height': 37, 'dt': 0.1, 'dt_per_plot': 10, 'diff': 1.5, 'duration': 3, 'timeline': False,
       'timeline_name': 'unused', 'save_graph': False, 'skip': False, 'cheby': False}


def full_plane(name, k, H, W):
    """The global plane `name` after k iterations: distinct per variable, row, column and iteration."""
    seed = sum(ord(ch) for ch in name)
    r, c = np.meshgrid(np.arange(H), np.arange(W), indexing='ij')
    return (seed + 1000.0 * r + c + 0.25 * k).astype(np.float32)


class CheckpointContext:
    """Shard of a fake model: stepping adds 0.25 to every cell; checkpoint_begin stages a copy, checkpoint_read
    reads rows of it (and raises after `fail_after` reads); set_rect_async writes at once and records its order."""
    fail_after = None

    def __init__(self, model, height, width, dt, diff, flags=0, device=0, row0=0, rows=0, steps_per_launch=0):
        self.model, self.height, self.width, self.dt, self.diff, self.flags = model, height, width, dt, diff, flags
        self.row0, self.rows = (row0, rows) if rows else (0, height)
        self.var_names = list(NAMES[model])
        self.nvars, self.dt_per_step = len(self.var_names), 10 if model == _capi.FENTON4V else 5
        self.state = {v: np.zeros((self.rows, width), np.float32) for v in self.var_names}
        self.iters, self.calls, self.staged, self.reads = 0, [], None, 0
        self.act, self.fr = None, None

    def set_state(self, var, host):
        self.state[var][...] = host

    def get_state(self, var, out=None):
        return self.state[var].copy()

    def set_phase(self, rows, first_row=0):
        pass

    def set_table(self, table, data):
        pass

    def comm_init(self, nranks, rank, uid):
        pass

    def step(self, op=0, n_iter=1):
        for v in self.var_names:
            self.state[v] += np.float32(0.25) * n_iter
        self.iters += n_iter
        if self.act is not None:
            self.act['k'] += n_iter
        if self.fr is not None:
            self.fr['k'] += n_iter

    def checkpoint_begin(self):
        if self.staged is not None:
            raise _capi.FibError('a checkpoint is already in flight')
        self.calls.append('checkpoint_begin')
        self.staged = [self.state[v].copy() for v in self.var_names]
        info = dict(nparts=self.nvars, iterations=self.iters, act_armed=0, act_up=0.0, act_down=0.0, act_k=0,
                    fr_armed=0, fr_var=0, fr_first=0, fr_every=0, fr_stride=0, fr_capacity=0, fr_k=0)
        if self.act is not None:
            self.staged += [m.copy() for m in self.act['maps']]
            info.update(nparts=self.nvars + 6, act_armed=1, act_up=self.act['up'], act_down=self.act['down'],
                        act_k=self.act['k'])
        if self.fr is not None:
            info.update(fr_armed=1, fr_var=self.fr['var'], fr_first=self.fr['first'], fr_every=self.fr['every'],
                        fr_stride=self.fr['stride'], fr_capacity=self.fr['capacity'], fr_k=self.fr['k'])
        return info

    def checkpoint_read(self, part, r0, out):
        self.reads += 1
        if self.fail_after is not None and self.reads > self.fail_after:
            raise OSError('disk full')
        out[...] = self.staged[part][r0 - self.row0:r0 - self.row0 + len(out)]

    def checkpoint_end(self):
        self.staged = None

    def set_rect_async(self, var, r0, c0, block):
        self.calls.append(('rect', var, r0, len(block)))
        self.state[var][r0 - self.row0:r0 - self.row0 + len(block), c0:c0 + block.shape[1]] = block

    def activation_watch(self, up, down):
        self.act = {'up': up, 'down': down, 'k': 0, 'maps': [np.full((self.rows, self.width), np.nan, np.float32)
                                                             for _ in range(6)]}

    def activation_resume(self, up, down, k):
        self.activation_watch(up, down)
        self.act['k'] = k

    def activation_set(self, which, plane):
        self.act['maps'][ck._ACT_MAPS.index(which)][...] = plane

    def frames_watch(self, var, first, every, stride, capacity):
        self.fr = {'var': self.var_names.index(var), 'first': first, 'every': every, 'stride': stride,
                   'capacity': capacity, 'k': 0}

    def frames_resume(self, var, first, every, stride, capacity, k):
        self.frames_watch(var, first, every, stride, capacity)
        self.fr['k'] = k

    def frames_shape(self):
        s = self.fr['stride']
        return -(-self.rows // s), -(-self.width // s)

    def frames_fetch(self, max_frames):
        self.calls.append('frames_fetch')
        rows, cols = self.frames_shape()
        return np.empty(0, np.uint64), np.empty((0, rows, cols), np.float32)

    def probe_watch(self, *a):
        pass

    def sync(self):
        self.calls.append('sync')

    def close(self):
        pass


@pytest.fixture
def fake(monkeypatch):
    monkeypatch.setattr(_capi, 'Context', CheckpointContext)
    monkeypatch.setattr(_capi, 'pinned_empty', lambda shape, dtype=np.float32: np.empty(shape, dtype))
    monkeypatch.setattr(_capi, 'pinned_free', lambda a: None)
    monkeypatch.setattr(_capi, 'comm_unique_id', lambda: bytes(128))
    monkeypatch.setattr(CheckpointContext, 'fail_after', None)
    monkeypatch.setattr(ck, 'STRIP_BYTES', 5 * 4 * CFG['width'])       # 5-row strips: several per shard
    monkeypatch.setattr(ck, 'RESTORE_BLOCK_ROWS', 4)


def shard_contexts(H, W, n, k, model=_capi.FENTON4V):
    out = []
    for row0, rows in partition_rows(H, n):
        c = CheckpointContext(model, H, W, 0.1, 1.5, row0=row0, rows=rows if n > 1 else 0)
        for v in c.var_names:
            c.state[v][...] = full_plane(v, k, H, W)[row0:row0 + rows]
        c.iters = k
        out.append(c)
    return out


def save_group(ctxs, path):
    os.makedirs(path)
    writers = [ck.save_shard(c, path) for c in ctxs]
    assert all(w.join() for w in writers)
    ck.write_manifest(path, ck.manifest(ctxs[0], writers[0].info, [w.record for w in writers]))


@pytest.mark.parametrize('H', [37, 31])
@pytest.mark.parametrize('n_save,n_load', [(1, 3), (3, 2), (2, 1)])
def test_read_rows_and_restore_across_partitions(fake, tmp_path, H, n_save, n_load):
    W, k = 24, 7
    path = str(tmp_path / 'ck')
    save_group(shard_contexts(H, W, n_save, k), path)
    man = ck.load_manifest(path)
    assert [s['rows'] for s in man['shards']] == [[r0, r0 + n] for r0, n in partition_rows(H, n_save)]
    for v in NAMES[_capi.FENTON4V]:
        assert np.array_equal(ck.read_rows(path, v, 0, H), full_plane(v, k, H, W))
        for r0, r1 in ((0, 1), (H - 1, H), (H // 3 - 1, H // 3 + 2), (5, H - 4)):      # across the seams
            assert np.array_equal(ck.read_rows(path, v, r0, r1), full_plane(v, k, H, W)[r0:r1])
    for rank, c in enumerate(shard_contexts(H, W, n_load, 0)):
        for v in c.var_names:
            c.state[v][...] = 0
        ck.check_compatible(man, c)
        pinned = ck.restore_context(c, path, bottom_up=rank % 2 == 1)
        for v in c.var_names:
            assert np.array_equal(c.state[v], full_plane(v, k, H, W)[c.row0:c.row0 + c.rows])
        # block-major, every plane of a block before the next block; odd ranks bottom to top
        rects = [x for x in c.calls if x[0] == 'rect']
        starts = [x[2] for x in rects[::c.nvars]]
        assert all(x[1] == v for blk in range(len(starts)) for x, v in zip(rects[blk * c.nvars:], c.var_names))
        assert starts == sorted(starts, reverse=rank % 2 == 1)
        assert len(pinned) == c.nvars


def test_manifest_round_trips(fake, tmp_path):
    path = str(tmp_path / 'ck')
    ctxs = shard_contexts(37, 24, 2, 3, model=_capi.BR)
    ctxs[0].flags = ctxs[1].flags = _capi.F_CHEBY | _capi.F_SKIP
    save_group(ctxs, path)
    man = ck.load_manifest(path)
    with open(os.path.join(path, ck.MANIFEST)) as f:
        assert json.load(f) == man
    assert man['version'] == ck.VERSION and man['iterations'] == 3
    assert man['config'] == {'model': 'br', 'height': 37, 'width': 24, 'dt': 0.1, 'diff': 1.5, 'cheby': True,
                             'skip': True, 'cheby_strict': False, 'lut': False, 'ultra_slow': False,
                             'no_chronic': False, 'no_clip': False}
    assert man['parts'] == NAMES[_capi.BR] and man['phase'] is False
    assert man['activation'] == {'armed': False} and man['frames'] == {'armed': False}
    for sh in man['shards']:
        for part, fn in sh['files'].items():
            a = np.load(os.path.join(path, fn), mmap_mode='r')
            assert a.dtype == np.float32 and a.shape == (sh['rows'][1] - sh['rows'][0], 24)


def test_mismatches_and_unknown_versions_are_refused(fake, tmp_path):
    path = str(tmp_path / 'ck')
    m = Fenton4v(dict(CFG))
    m.add_hole_to_phase_field(10, 12, 4)
    m.define()
    m.checkpoint(path).wait()
    for change, key in ((dict(diff=1.4), 'diff'), (dict(width=28), 'width')):
        with pytest.raises(ValueError, match=key):
            r = Fenton4v(dict(CFG, **change))
            r.add_hole_to_phase_field(10, 12, 4)
            r.restore(path)
    with pytest.raises(ValueError, match='model'):
        BeelerReuter(dict(CFG)).restore(path)
    with pytest.raises(ValueError, match='phase'):
        Fenton4v(dict(CFG)).restore(path)                      # no phase field
    r = Fenton4v(dict(CFG))
    r.add_hole_to_phase_field(10, 13, 4)                       # another phase field
    with pytest.raises(ValueError, match='phase'):
        r.restore(path)
    assert not r.defined
    r = Fenton4v(dict(CFG))
    r.add_hole_to_phase_field(10, 12, 4)
    r.restore(path)
    fn = os.path.join(path, ck.MANIFEST)
    man = json.load(open(fn))
    man['version'] = ck.VERSION + 1
    json.dump(man, open(fn, 'w'))
    with pytest.raises(ck.CheckpointError, match='version'):
        Fenton4v(dict(CFG)).restore(path)
    os.remove(fn)
    with pytest.raises(ck.CheckpointError, match='no manifest.json'):
        Fenton4v(dict(CFG)).restore(path)


def test_a_failing_writer_leaves_the_previous_checkpoint(fake, tmp_path):
    path = str(tmp_path / 'ck')
    m = Fenton4v(dict(CFG))
    m.define()
    m._ctx.step(0, 2)
    m.iterations = 2
    m.checkpoint(path).wait()
    m._ctx.step(0, 3)
    m.iterations = 5
    m._ctx.fail_after = 3                                      # half-way through the second plane
    h = m.checkpoint(path)
    with pytest.raises(RuntimeError, match='disk full'):
        h.wait()
    assert not os.path.exists(os.path.join(path + '.partial', ck.MANIFEST))
    man = ck.load_manifest(path)
    assert man['iterations'] == 2
    r = Fenton4v(dict(CFG))
    r.restore(path)
    assert r.iterations == 2
    assert np.array_equal(r._ctx.state['U'], np.full((37, 24), 0.5, np.float32) + np.pad(
        np.ones((37, 1), np.float32), ((0, 0), (1, 22))))
    m._ctx.fail_after = None
    m.checkpoint(path).wait()                                  # and the next save replaces it
    assert ck.load_manifest(path)['iterations'] == 5


def test_checkpoint_drains_frames_first_and_restore_resumes_the_observers(fake, tmp_path):
    path = str(tmp_path / 'ck')
    m = Fenton4v(dict(CFG))
    m.define()
    m.record_frames(every=3, stride=2)
    m.watch_activation()
    m._ctx.step(0, 7)
    m.iterations = 7
    m._ctx.act['maps'][2][...] = 42.0
    m._ctx.calls.clear()
    ck_ = m.checkpoint(path)
    assert m._ctx.calls.index('frames_fetch') < m._ctx.calls.index('checkpoint_begin')
    m.close()                                                   # waits for the save
    assert ck_.done
    r = Fenton4v(dict(CFG))
    man = r.restore(path)
    assert man['frames'] == {'armed': True, 'var': 'U', 'first': 1, 'every': 3, 'stride': 2,
                             'capacity': Fenton4v.default_frame_capacity(3), 'k': 7}
    assert man['activation']['armed'] and man['activation']['k'] == 7
    assert r._ctx.act['k'] == 7 and r._ctx.fr['k'] == 7
    assert np.all(r._ctx.act['maps'][2] == 42.0)
    assert r._frames['k'] == 7 and r._frames['upto'] == 3       # frames at k = 1, 4, 7 stay with the saver


def test_a_second_checkpoint_waits_for_the_first(fake, tmp_path):
    m = Fenton4v(dict(CFG))
    m.define()
    first = m.checkpoint(str(tmp_path / 'a'))
    second = m.checkpoint(str(tmp_path / 'b'))
    assert first.done and not second.done
    second.wait()
    assert ck.load_manifest(str(tmp_path / 'a'))['iterations'] == 0
    assert ck.load_manifest(str(tmp_path / 'b'))['iterations'] == 0


def test_checkpoint_entry_points_validate_without_a_gpu():
    L = _capi.lib()
    assert C.sizeof(_capi.CheckpointInfo) == 96
    assert _capi.CheckpointInfo.act_k.offset == 32 and _capi.CheckpointInfo.fr_k.offset == 64
    info = _capi.CheckpointInfo()
    info.struct_size = C.sizeof(info)
    buf = np.zeros(4, np.float32)
    p = buf.ctypes.data_as(C.c_void_p)
    for rc in (L.fib_checkpoint_begin(None, C.byref(info)), L.fib_checkpoint_begin(None, None),
               L.fib_checkpoint_read(None, 0, 0, 1, p), L.fib_checkpoint_end(None),
               L.fib_activation_resume(None, 0.5, 0.5, 3), L.fib_activation_set(None, _capi.ACT_SAMPLE, p, 4),
               L.fib_frames_resume(None, 0, 1, 10, 1, 4, 7)):
        assert rc == -1
        assert b'NULL' in L.fib_last_error()


# ---- two ranks over gloo: the same collectives on every rank, also when one rank's writer fails -------------
def worker(rank, world, port, path, fail_rank, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        _capi.Context = CheckpointContext
        _capi.pinned_empty = lambda shape, dtype=np.float32: np.empty(shape, dtype)
        _capi.pinned_free = lambda a: None
        _capi.comm_unique_id = lambda: bytes(128)
        log = []
        for name in ('barrier', 'all_gather_object', 'broadcast_object_list', 'all_reduce', 'broadcast'):
            def wrap(fn, name=name):
                def f(*a, **kw):
                    log.append(name)
                    return fn(*a, **kw)
                return f
            setattr(dist, name, wrap(getattr(dist, name)))
        m = Fenton4v(dict(CFG, distributed=True))
        m.define()
        m._ctx.step(0, 4)
        m.iterations = 4
        log.clear()
        if rank == fail_rank:
            m._ctx.fail_after = 1
        h = m.checkpoint(path)
        try:
            h.wait()
            result = 'ok'
        except RuntimeError as e:
            result = str(e)
        out[rank] = (log, result)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize('fail_rank', [None, 1])
def test_two_ranks_issue_the_same_collectives(tmp_path, monkeypatch, fail_rank):
    path = str(tmp_path / 'ck')
    out = mp.Manager().dict()
    mp.spawn(worker, args=(2, free_port(), path, fail_rank, out), nprocs=2, join=True)
    assert out[0][0] == out[1][0] and out[0][0]
    if fail_rank is None:
        assert out[0][1] == out[1][1] == 'ok'
        monkeypatch.setattr(_capi, 'Context', CheckpointContext)
        monkeypatch.setattr(_capi, 'pinned_empty', lambda shape, dtype=np.float32: np.empty(shape, dtype))
        monkeypatch.setattr(_capi, 'pinned_free', lambda a: None)
        r = Fenton4v(dict(CFG))
        r.restore(path)
        assert r.iterations == 4
        assert np.array_equal(r._ctx.state['V'], np.full((37, 24), 2.0, np.float32))
    else:
        assert 'rank 1' in out[0][1] and 'rank 1' in out[1][1] and 'disk full' in out[0][1]
        assert not os.path.exists(path) and not os.path.exists(os.path.join(path + '.partial', ck.MANIFEST))
