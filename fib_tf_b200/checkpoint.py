"""
fib_tf_b200.checkpoint -- checkpoint and restart: a run's state and observers saved while stepping continues,
restored bit for bit into a context on any number of GPUs.

Format: a directory.
    manifest.json                written last (a directory without it is not a checkpoint): the format version,
                                 the model and the config that changes arithmetic, `iterations`, the observers'
                                 info, the pacing entries still to fire and the shard files with their global row
                                 ranges
    <part>.rows<r0>-<r1>.npy     one [r1 - r0, width] float32 array per (shard, part); parts are the state
                                 planes by their reference names, the activation map's last sample and five maps
                                 (act_*) when one was armed, and `phase` when the model has a phase field

The device side is include/fib_b200.h fib_checkpoint_begin / _read / _end: begin stages a copy of the shard
behind everything stepped so far and returns, a writer thread reads it out strip by strip through a small
page-locked bounce buffer while the caller keeps stepping.  These functions work on _capi.Context objects (one
process may save from, and restore into, shard groups); IonicModel.checkpoint() / restore() use them.
"""
import ctypes as C
import errno
import json
import os
import shutil
import threading

import numpy as np

from . import _capi

FORMAT = 'fib_tf_b200 checkpoint'
VERSION = 1
MANIFEST = 'manifest.json'
ACT_PARTS = ('act_sample', 'act_first', 'act_last', 'act_prev', 'act_repol', 'act_count')
_ACT_MAPS = (_capi.ACT_SAMPLE, _capi.ACT_FIRST, _capi.ACT_LAST, _capi.ACT_PREV, _capi.ACT_REPOL, _capi.ACT_COUNT)
MODEL_NAMES = {_capi.FENTON4V: 'fenton4v', _capi.BR: 'br', _capi.COURT: 'court', _capi.COURT_ULTRA: 'court_ultra'}
# the fib_config flags that change arithmetic (graph / persistent / steps per launch do not: every route is
# bit-identical)
ARITH_FLAGS = (('cheby', _capi.F_CHEBY), ('skip', _capi.F_SKIP), ('cheby_strict', _capi.F_CHEBY_STRICT),
               ('lut', _capi.F_LUT), ('ultra_slow', _capi.F_ULTRA_SLOW), ('no_chronic', _capi.F_NO_CHRONIC),
               ('no_clip', _capi.F_NO_CLIP))
STRIP_BYTES = 32 << 20          # the writer's bounce buffer
RESTORE_BLOCK_ROWS = 1024       # rows per block of the restore upload (the library's pipelined block, at least)


class CheckpointError(RuntimeError):
    pass


def arithmetic_config(ctx):
    """The model and the config keys of a context that change what it computes."""
    cfg = {'model': MODEL_NAMES[ctx.model], 'height': int(ctx.height), 'width': int(ctx.width),
           'dt': float(ctx.dt), 'diff': float(ctx.diff)}
    replicas = getattr(ctx, 'replicas', 1)
    if replicas > 1:        # the parts are then [replicas * height, width]: replica b is rows b * height ..
        cfg.update(replicas=int(replicas), diff=[float(d) for d in ctx.replica_diff])
    for key, bit in ARITH_FLAGS:
        cfg[key] = bool(ctx.flags & bit)
    return cfg


def part_names(ctx, info):
    return list(ctx.var_names) + (list(ACT_PARTS) if info['act_armed'] else [])


def shard_file(part, r0, r1):
    return '%s.rows%d-%d.npy' % (part, r0, r1)


# page-locked bounce buffers, kept for the next checkpoint: freeing page-locked memory synchronises the device
_bounce_lock = threading.Lock()
_bounce_free = []


def _bounce(width):
    rows = max(1, STRIP_BYTES // (4 * width))
    with _bounce_lock:
        for k, b in enumerate(_bounce_free):
            if b.shape[1] == width:
                return _bounce_free.pop(k)
    return _capi.pinned_empty((rows, width))


def _write_npy(path, rows, width, fill, buf):
    """[rows, width] float32 .npy at `path`, filled strip by strip: fill(r, out) writes rows [r, r + len(out))
    of the array into `out`.  Durable (fsync) when it returns."""
    with open(path, 'wb') as f:
        np.lib.format.write_array_header_1_0(f, {'descr': '<f4', 'fortran_order': False, 'shape': (rows, width)})
        for r in range(0, rows, buf.shape[0]):
            out = buf[:min(buf.shape[0], rows - r)]
            fill(r, out)
            f.write(memoryview(out).cast('B'))
        f.flush()
        os.fsync(f.fileno())


class ShardWriter:
    """One shard's save: fib_checkpoint_begin on the caller's thread (the copy is ordered after everything
    stepped so far), then a thread that reads the staged parts out into `directory` while the caller steps on."""

    def __init__(self, ctx, directory, phase_rows=None):
        self.ctx, self.directory = ctx, directory
        self.info = ctx.checkpoint_begin()
        r0, r1 = ctx.row0, ctx.row0 + ctx.rows
        parts = part_names(ctx, self.info)
        names = parts + (['phase'] if phase_rows is not None else [])
        self.record = {'rows': [r0, r1], 'files': {p: shard_file(p, r0, r1) for p in names}}
        self.error = None
        self._thread = threading.Thread(target=self._run, args=(parts, phase_rows), daemon=True,
                                        name='fib-checkpoint-writer')
        self._thread.start()

    def _run(self, parts, phase_rows):
        ctx, buf = self.ctx, None
        try:
            buf = _bounce(ctx.width)
            r0 = ctx.row0
            for k, name in enumerate(parts):
                _write_npy(os.path.join(self.directory, self.record['files'][name]), ctx.rows, ctx.width,
                           lambda r, out, k=k: ctx.checkpoint_read(k, r0 + r, out), buf)
            if phase_rows is not None:
                ph = np.asarray(phase_rows, dtype=np.float32)
                _write_npy(os.path.join(self.directory, self.record['files']['phase']), ctx.rows, ctx.width,
                           lambda r, out: out.__setitem__(Ellipsis, ph[r:r + len(out)]), buf)
        except BaseException as e:          # reported by join(); the caller decides, collectively
            self.error = e
        finally:
            if buf is not None:
                with _bounce_lock:
                    _bounce_free.append(buf)

    def join(self):
        """Waits for the writer and releases the staging copy; True if the shard was saved."""
        self._thread.join()
        try:
            self.ctx.checkpoint_end()
        except Exception as e:
            self.error = self.error or e
        return self.error is None


def save_shard(ctx, directory, phase_rows=None):
    """Starts saving one shard (a _capi.Context) into `directory` and returns its ShardWriter at once.
    `phase_rows`: the phase field's rows of this shard, saved as part `phase`, or None."""
    return ShardWriter(ctx, directory, phase_rows)


def pacing_state(entries, iterations):
    """The pacing entries (IonicModel.pace) that still fire after absolute ODE iteration `iterations`, as manifest
    records: name, rect [r0, r1, c0, c1], value, floor, `next` (the absolute iteration its next beat follows),
    `every` and `count` (the beats left; 0: until removed).  An entry fires after iterations next + j * every."""
    out = []
    for e in entries:
        step = max(int(e['every']), 1)
        done = 0 if iterations < e['next'] else (iterations - e['next']) // step + 1
        if e['count'] and done >= e['count']:
            continue
        out.append({'name': e['name'], 'rect': [int(x) for x in e['rect']], 'value': float(e['value']),
                    'floor': float(e['floor']), 'next': int(e['next'] + done * step), 'every': int(e['every']),
                    'count': int(e['count'] - done) if e['count'] else 0})
        if e.get('replica') is not None:                # a batched model's entry of one replica
            out[-1]['replica'] = int(e['replica'])
    return out


def resume_pacing(ctx, entries, iterations):
    """Adds the manifest's pacing records `entries` to `ctx`, a context that continues absolute ODE iteration
    `iterations`, so that every beat follows the same absolute iteration as in the saved run; returns the records
    with their entry ids (key `id`)."""
    out = []
    for e in entries:
        if e['next'] <= iterations:
            raise CheckpointError('pacing entry %r: next beat after iteration %d, but the run continues from %d'
                                  % (e['name'], e['next'], iterations))
        where = {'replica': e['replica']} if e.get('replica') is not None else {}
        pid = ctx.pace_add(*e['rect'], e['value'], e['floor'], e['next'] - iterations, e['every'], e['count'], **where)
        out.append(dict(e, id=pid))
    return out


def manifest(ctx, info, shards, iterations=None, pacing=()):
    """The manifest dict of a checkpoint of `ctx`'s model: `shards` = the ShardWriter records of every shard,
    `pacing` = pacing_state() of the run at the checkpoint."""
    act = {'armed': bool(info['act_armed'])}
    if act['armed']:
        act.update(up=float(info['act_up']), down=float(info['act_down']), k=int(info['act_k']))
    frames = {'armed': bool(info['fr_armed'])}
    if frames['armed']:
        frames.update(var=ctx.var_names[info['fr_var']], first=int(info['fr_first']), every=int(info['fr_every']),
                      stride=int(info['fr_stride']), capacity=int(info['fr_capacity']), k=int(info['fr_k']))
    shards = sorted(shards, key=lambda s: s['rows'][0])
    return {'format': FORMAT, 'version': VERSION, 'config': arithmetic_config(ctx),
            'iterations': int(info['iterations'] if iterations is None else iterations),
            'parts': part_names(ctx, info), 'phase': 'phase' in shards[0]['files'],
            'activation': act, 'frames': frames, 'pacing': list(pacing), 'shards': shards}


def write_manifest(directory, man):
    """Writes manifest.json durably: to a temporary name, fsync, then renamed into place."""
    tmp = os.path.join(directory, MANIFEST + '.tmp')
    with open(tmp, 'w') as f:
        json.dump(man, f, indent=1)
        f.flush()
        os.fsync(f.fileno())
    os.replace(tmp, os.path.join(directory, MANIFEST))
    _fsync_dir(directory)


def _fsync_dir(path):
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def _exchange(a, b):
    """Swaps two directory entries atomically (renameat2 RENAME_EXCHANGE); False where that is unsupported."""
    try:
        libc = C.CDLL(None, use_errno=True)
        fn = libc.renameat2
    except (OSError, AttributeError):
        return False
    fn.argtypes = [C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_uint]
    AT_FDCWD, RENAME_EXCHANGE = -100, 2
    if fn(AT_FDCWD, os.fsencode(a), AT_FDCWD, os.fsencode(b), RENAME_EXCHANGE) == 0:
        return True
    if C.get_errno() in (errno.ENOSYS, errno.EINVAL, errno.ENOTSUP):
        return False
    raise OSError(C.get_errno(), 'renameat2(%s, %s): %s' % (a, b, os.strerror(C.get_errno())))


def publish(partial, path):
    """Makes the complete checkpoint in `partial` the one at `path`, replacing a previous one atomically where
    the file system can swap two directories; the previous one is then deleted."""
    parent = os.path.dirname(os.path.abspath(path))
    if os.path.isdir(path) and _exchange(partial, path):
        _fsync_dir(parent)
        shutil.rmtree(partial)
        return
    if os.path.isdir(path):             # no atomic swap here: move the old one aside first
        old = path + '.old'
        shutil.rmtree(old, ignore_errors=True)
        os.rename(path, old)
        os.rename(partial, path)
        _fsync_dir(parent)
        shutil.rmtree(old)
        return
    os.rename(partial, path)
    _fsync_dir(parent)


def load_manifest(path):
    """The manifest of the checkpoint at `path`; CheckpointError if it is not a complete checkpoint of this
    format and version."""
    fn = os.path.join(path, MANIFEST)
    if not os.path.isfile(fn):
        raise CheckpointError('%s is not a complete checkpoint: it has no %s (a save that did not finish, or not '
                              'a checkpoint at all)' % (path, MANIFEST))
    with open(fn) as f:
        man = json.load(f)
    if man.get('format') != FORMAT:
        raise CheckpointError('%s: not a %s' % (fn, FORMAT))
    if man.get('version') != VERSION:
        raise CheckpointError('%s: checkpoint format version %r, this library reads version %d'
                              % (fn, man.get('version'), VERSION))
    return man


def read_rows(path, part, r0, r1, man=None):
    """Global rows [r0, r1) of part `part` (a state variable, act_*, or phase) as a [r1 - r0, width] float32
    array, assembled from whichever shard files cover them (memory-mapped: only these rows are read)."""
    man = load_manifest(path) if man is None else man
    width = man['config']['width']
    height = man['config']['height'] * man['config'].get('replicas', 1)
    if not 0 <= r0 < r1 <= height:
        raise ValueError('rows [%d, %d) outside the grid of height %d' % (r0, r1, height))
    out = np.empty((r1 - r0, width), np.float32)
    covered = 0
    for sh in man['shards']:
        s0, s1 = sh['rows']
        a, b = max(r0, s0), min(r1, s1)
        if a >= b:
            continue
        if part not in sh['files']:
            raise KeyError('checkpoint %s has no part %r' % (path, part))
        arr = np.load(os.path.join(path, sh['files'][part]), mmap_mode='r')
        if arr.shape != (s1 - s0, width) or arr.dtype != np.float32:
            raise CheckpointError('%s: shape %r / dtype %s, expected (%d, %d) float32'
                                  % (sh['files'][part], arr.shape, arr.dtype, s1 - s0, width))
        out[a - r0:b - r0] = arr[a - s0:b - s0]
        covered += b - a
    if covered != r1 - r0:
        raise CheckpointError('checkpoint %s: its shards cover %d of rows [%d, %d)' % (path, covered, r0, r1))
    return out


def check_compatible(man, ctx, phase_rows=None):
    """ValueError naming the first key in which `ctx` (and `phase_rows`, its shard's rows of the phase field or
    None) would compute differently from the run that was saved."""
    mine = arithmetic_config(ctx)
    saved_cfg = dict({'replicas': 1}, **man['config'])
    mine.setdefault('replicas', 1)
    for key, saved in saved_cfg.items():
        if mine.get(key) != saved:
            raise ValueError('checkpoint was saved with %s=%r, this model has %s=%r' % (key, saved, key, mine.get(key)))
    if man['phase'] != (phase_rows is not None):
        raise ValueError('phase: the checkpoint was saved %s a phase field, this model has %s'
                         % ('with' if man['phase'] else 'without', 'one' if phase_rows is not None else 'none'))


def check_phase(path, man, ctx, phase_rows):
    if phase_rows is None:
        return
    saved = read_rows(path, 'phase', ctx.row0, ctx.row0 + ctx.rows, man)
    if not np.array_equal(saved, np.asarray(phase_rows, dtype=np.float32)):
        raise ValueError('phase: the phase field differs from the one the checkpoint was saved with')


def restore_context(ctx, path, bottom_up=False, man=None):
    """Loads the checkpoint at `path` into a fresh context `ctx` of any partition: its rows of every state plane,
    and the activation map and frame recorder if they were armed (resumed with their counters, so the next
    iteration continues them).  The planes go up as full-width blocks of RESTORE_BLOCK_ROWS rows with
    fib_set_rect_async, every plane of a block before the next block, top to bottom (bottom to top with
    `bottom_up`: odd ranks of NCCL shards), so that a large grid steps behind its own upload when no observer
    is armed.  Returns the page-locked host copies, which must stay untouched until the context's next
    synchronous call; pass them to release() then.  The caller checks compatibility first (check_compatible)."""
    man = load_manifest(path) if man is None else man
    r0, rows = ctx.row0, ctx.rows
    act, fr = man['activation'], man['frames']
    if act['armed']:
        ctx.activation_resume(act['up'], act['down'], act['k'])
        for name, which in zip(ACT_PARTS, _ACT_MAPS):
            ctx.activation_set(which, read_rows(path, name, r0, r0 + rows, man))
    if fr['armed']:
        ctx.frames_resume(fr['var'], fr['first'], fr['every'], fr['stride'], fr['capacity'], fr['k'])
    pinned = []
    try:
        for v in ctx.var_names:
            pinned.append(_capi.pinned_empty((rows, ctx.width)))
            pinned[-1][...] = read_rows(path, v, r0, r0 + rows, man)
        starts = list(range(0, rows, RESTORE_BLOCK_ROWS))
        for s in (reversed(starts) if bottom_up else starts):
            for v, host in zip(ctx.var_names, pinned):
                ctx.set_rect_async(v, r0 + s, 0, host[s:s + RESTORE_BLOCK_ROWS])
    except BaseException:
        ctx.sync()
        release(pinned)
        raise
    return pinned


def release(pinned):
    """Frees the host copies restore_context() returned (after the context's next synchronous call)."""
    for a in pinned:
        _capi.pinned_free(a)
    del pinned[:]
