"""Host column emitter: BAM records -> int32 columns for libecb200.

Does what alntools/bam_utils.process_convert_bam does up to (not including) the key build: decode,
the unmapped/paired-end filters (bam_utils.py:264-270), read-name trimming (:301-304) and the
name-change test (:306).  Per VALID alignment it emits
    read_group  (changes whenever the reference would start a new read)
    target_idx, hap_idx  (header lookup of the alignment's reference id)
    [cell_idx]  multisample only: dense id of field 14 of the '|||'-split group name
                (bam_utils_multisample.py:270-280)
Everything after that - grouping, de-duplication, counting, ordering, matrix build - runs on the GPU.
"""
import collections

import numpy as np

from . import bam_io, bamcols, utils


def _trim(name):
    i = name.find(" ")
    return name[:i] if i > 0 else name


def _valid(flag, tid, ntid, npos):
    if flag & 0x4:
        return False
    if flag & 0x1 and ((flag & 0x80) or not (flag & 0x2) or tid != ntid or npos < 0):
        return False
    return True


class Columns(object):
    __slots__ = ("read_group", "target_idx", "hap_idx", "cell_idx", "all_alignments", "valid_alignments",
                 "n_groups")

    def __init__(self, rg, tg, hp, cell, all_alignments, n_groups):
        self.read_group = np.asarray(rg, dtype=np.int32)
        self.target_idx = np.asarray(tg, dtype=np.int32)
        self.hap_idx = np.asarray(hp, dtype=np.int32)
        self.cell_idx = None if cell is None else np.asarray(cell, dtype=np.int32)
        self.all_alignments = all_alignments
        self.valid_alignments = len(self.read_group)
        self.n_groups = n_groups


def emit_single(records, tables):
    """records: iterable of (qname, flag, tid, pos, next_tid, next_pos); bam_utils.py:258-328."""
    rg, tids = [], []
    current = None
    group = -1
    total = 0
    for qname, flag, tid, _pos, ntid, npos in records:
        total += 1
        if not _valid(flag, tid, ntid, npos):
            continue
        name = _trim(qname)
        if name != current or group < 0:
            current = name
            group += 1
        rg.append(group)
        tids.append(tid)
    tids = np.asarray(tids, dtype=np.int64)
    return Columns(rg, tables.tid_target[tids] if len(tids) else [], tables.tid_hap[tids] if len(tids) else [],
                   None, total, group + 1)


def emit_multisample(records, tables, cell_ids):
    """One BAM file of the per-cell path (bam_utils_multisample.py:209-300).

    cell_ids: dict cell name -> dense int, shared by all files of the job and extended here.
    Quirks kept: the remembered group name is trimmed only for the first group of a file (:258-262 vs
    :292), the cell comes from the remembered name, and a name with fewer than 15 '|||' fields raises
    IndexError exactly where the reference does.  The last read is NOT dropped here; the caller pushes
    the file with drop_last_group=1 (:306-308).
    """
    rg, tids, cells = [], [], []
    current = None
    group = -1
    cell = 0
    pending = False   # the current group's cell is resolved when the reference would: at the next valid alignment
    total = 0
    for qname, flag, tid, _pos, ntid, npos in records:
        total += 1
        if not _valid(flag, tid, ntid, npos):
            continue
        if current is None:
            current = _trim(qname)
            group = 0
            cell = cell_ids.setdefault(current.split("|||")[14], len(cell_ids))
        elif pending:
            cell = cell_ids.setdefault(current.split("|||")[14], len(cell_ids))   # :270-280
            cells[-1] = cell
            pending = False
        if current != _trim(qname):                                              # :288
            current = qname                                                      # :292 (untrimmed)
            group += 1
            pending = True
            cell = 0
        rg.append(group)
        tids.append(tid)
        cells.append(cell)
    tids = np.asarray(tids, dtype=np.int64)
    return Columns(rg, tables.tid_target[tids] if len(tids) else [], tables.tid_hap[tids] if len(tids) else [],
                   cells, total, group + 1)


def use_python_emitter():
    """ALNTOOLS_B200_EMITTER=python selects the record-level Python emitter above (slow; kept as the
    readable statement of the rules and as a cross-check); the default is the native one (bamcols)."""
    import os
    return os.environ.get("ALNTOOLS_B200_EMITTER", "native").lower() == "python"


def decode_mode(decode=None):
    """Where a single-sample convert() decodes the BAM file: `decode`, else the environment variable
    ALNTOOLS_B200_DECODE (the CLI keeps the reference's options, so the environment is its only way to say it):
    "host" (default: libbamcols on the CPU threads) or "device" (BGZF inflate and the record pass on the GPU)."""
    import os
    mode = decode if decode is not None else os.environ.get("ALNTOOLS_B200_DECODE", "host")
    if str(mode).lower() not in ("host", "device"):
        raise ValueError("the BAM decode must be 'host' or 'device' (decode= / ALNTOOLS_B200_DECODE), not %r" % (mode,))
    return str(mode).lower()


def collate_mode(collate=None):
    """Whether a single-sample convert() collates alignments by read name: `collate`, else the environment variable
    ALNTOOLS_B200_COLLATE ("0", the default, or "1"; the CLI keeps the reference's options, so the environment is
    its only way to say it)."""
    import os
    if collate is not None:
        return bool(collate)
    value = os.environ.get("ALNTOOLS_B200_COLLATE", "0").strip()
    if value not in ("0", "1"):
        raise ValueError("ALNTOOLS_B200_COLLATE must be 0 or 1, not %r" % (value,))
    return value == "1"


def collate_budget():
    """Device bytes a collator may hold, from the environment variable ALNTOOLS_B200_COLLATE_BUDGET (a non-negative
    integer; unset or 0: automatic, half of the GPU's free memory).  A collation whose rows do not fit spills them to
    host memory and works in passes; the outputs do not depend on it.  On a shared GPU it caps what a job takes."""
    import os
    value = os.environ.get("ALNTOOLS_B200_COLLATE_BUDGET", "").strip()
    if not value:
        return 0
    if not (value.isascii() and value.isdigit()):
        raise ValueError("ALNTOOLS_B200_COLLATE_BUDGET must be a non-negative integer (bytes), not %r" % (value,))
    return int(value)


def max_read():
    """Longest read (alignments with one name) a conversion accepts, from the environment variable
    ALNTOOLS_B200_MAX_READ (a non-negative integer; unset: 16384, the library's default; 0: no limit below the push
    limit of 2^31 - 8192).  Reads longer than 16384 alignments then go through a sort-based pass on the GPU.  The
    default is kept because in a file grouped by name a read that long more often means a broken input; values from 1
    to 16383 are refused by the library.  The CLI keeps the reference's options, so the environment is its only way to
    say it."""
    import os
    value = os.environ.get("ALNTOOLS_B200_MAX_READ", "").strip()
    if not value:
        return 16384
    if not (value.isascii() and value.isdigit()):
        raise ValueError("ALNTOOLS_B200_MAX_READ must be a non-negative integer (alignments), not %r" % (value,))
    return int(value)


Mode = collections.namedtuple("Mode", ["python", "decode", "collate", "launcher", "gpus"])


def resolve_mode(cells, devices=None, decode=None, collate=None, range_file=False):
    """The settings of one conversion, read once from the arguments and the environment: the emitter
    (use_python_emitter), the decode (decode_mode), collation (collate_mode), whether this process is one rank of a
    one-process-per-GPU job (utils.under_launcher) and otherwise how many GPUs to spread the job over
    (utils.requested_gpus; 1 under a launcher, which has started the ranks).  cells: the per-cell converter, whose
    decode and collation come from the environment only.  Refuses what no converter runs - ValueError for a value it
    does not know, NotImplementedError for a combination - before any file is opened or any GPU is touched."""
    python = use_python_emitter()
    decode = decode_mode(decode)
    if cells and decode == "device":
        raise NotImplementedError("the per-cell (--multisample) conversion has no device BAM decode yet: it needs a GPU "
                                  "cell-name dictionary (unset ALNTOOLS_B200_DECODE)")
    collate = collate_mode(collate)
    if cells and collate:
        raise NotImplementedError("the per-cell (--multisample) conversion has no collation by read name: its rules "
                                  "depend on consecutive records (unset ALNTOOLS_B200_COLLATE)")
    launcher = utils.under_launcher()
    gpus = 1 if launcher else utils.requested_gpus(devices)
    multi = launcher or gpus > 1
    if decode == "device":
        if multi:
            raise NotImplementedError("device BAM decode runs on one GPU; the multi-GPU convert has no device decode yet "
                                      "(use decode='host' / unset ALNTOOLS_B200_DECODE)")
        if python:
            raise NotImplementedError("device BAM decode replaces the native emitter; it does not combine with "
                                      "ALNTOOLS_B200_EMITTER=python")
    if collate:
        if multi:
            raise NotImplementedError("collation by read name runs on one GPU: reads span the shards of a multi-GPU "
                                      "convert (unset ALNTOOLS_B200_COLLATE or use one GPU)")
        if decode == "device":
            raise NotImplementedError("collation by read name takes the host decode (use decode='host' / unset "
                                      "ALNTOOLS_B200_DECODE)")
    if python and multi:
        raise NotImplementedError("the multi-GPU path needs the native emitter (unset ALNTOOLS_B200_EMITTER)")
    if python and range_file:
        raise NotImplementedError("--rangefile needs the native emitter (unset ALNTOOLS_B200_EMITTER)")
    return Mode(python, decode, collate, launcher, gpus)


def emit_collated(records, tables):
    """The rows convert(collate=True) builds from: a read is every valid alignment whose trimmed name (as emit_single
    trims it) is the same, wherever it lies in the file; reads are ordered by their first valid alignment, and each
    read's alignments follow in file order.  So the result is emit_single of the file regrouped that way."""
    reads = {}                                            # trimmed name -> tids; dicts keep insertion order
    total = 0
    for qname, flag, tid, _pos, ntid, npos in records:
        total += 1
        if _valid(flag, tid, ntid, npos):
            reads.setdefault(_trim(qname), []).append(tid)
    rg = np.repeat(np.arange(len(reads), dtype=np.int32), [len(t) for t in reads.values()])
    tids = np.asarray([t for ts in reads.values() for t in ts], dtype=np.int64)
    return Columns(rg, tables.tid_target[tids] if len(tids) else [], tables.tid_hap[tids] if len(tids) else [],
                   None, total, len(reads))


_PINNED = []      # pinned buffer sets of finished streams, reused by later streams of this process


def _buffers(rows, dtypes, pinned):
    """A set of host buffers of `rows` elements, one per dtype name in `dtypes`; pinned: page-locked torch tensors.
    Pinning host memory costs about as much as decoding into it, so a pinned set of the same dtypes that an earlier
    stream of this process left in the pool is taken again when it is large enough."""
    if not pinned:
        return [np.empty(rows, dtype=d) for d in dtypes]
    import torch
    dtypes = [getattr(torch, d) for d in dtypes]
    for i, bufs in enumerate(_PINNED):
        if [b.dtype for b in bufs] == dtypes and int(bufs[0].shape[0]) >= rows:
            return _PINNED.pop(i)
    return [torch.empty(rows, dtype=d, pin_memory=True) for d in dtypes]


def _release(sets):
    """Pinned buffer sets of a finished stream go back to the pool (at most 8 sets of the same dtypes are kept)."""
    for bufs in sets:
        kind = [b.dtype for b in bufs]
        if sum([b.dtype for b in held] == kind for held in _PINNED) < 8:
            _PINNED.append(bufs)


def _feed(fill, consume, depth):
    """Run `fill` on a worker thread up to `depth` buffers ahead of `consume`, which runs in the calling thread.

    fill(buf) fills a buffer and returns (buf, item, done): the buffer it was given (None until the ring holds `depth`
    buffers: fill makes one then) or one it made in its place, and what consume(buf, item) needs to use it.  Buffers
    reach consume in the order they were filled and go back to fill once consumed; nothing is filled after the item
    with done=True.  An exception raised in fill is raised here.  However this returns, the thread has stopped
    first, so the caller may free what fill works on (bamcols_close frees what bamcols_emit works on)."""
    import queue
    import threading
    free, full = queue.Queue(), queue.Queue()
    for _ in range(depth):
        free.put(None)
    stop = threading.Event()

    def produce():
        try:
            done = False
            while not done and not stop.is_set():
                try:
                    buf = free.get(timeout=0.05)
                except queue.Empty:
                    continue
                buf, item, done = fill(buf)
                full.put((buf, item, done, None))
        except BaseException as exc:                      # re-raised by the consumer
            full.put((None, None, True, exc))

    worker = threading.Thread(target=produce, daemon=True)
    worker.start()
    try:
        done = False
        while not done:
            buf, item, done, exc = full.get()
            if exc is not None:
                raise exc
            consume(buf, item)
            item = None                                   # not kept alive while the next one is waited for
            free.put(buf)
    finally:
        stop.set()
        worker.join()


def stream_single(reader, builder, chunk_rows=1 << 21, pinned=True, depth=3):
    """Decode `reader` (bamcols.BamColumnReader, tables set) on a worker thread into a small ring of
    pinned buffers and push every filled buffer to the GPU while the next one is being decoded.
    Chunks end on read boundaries (bamcols_emit never splits a read), order_base = rows pushed so far,
    so the result equals one push of the whole file.  Returns the number of valid alignments."""
    rows, sets, pushed = int(chunk_rows), [], 0

    def fill(bufs):
        nonlocal rows
        while True:
            if bufs is None or int(bufs[0].shape[0]) < rows:   # none yet, or one from before the buffers grew
                bufs = _buffers(rows, ("int32",) * 3, pinned)
                sets.append(bufs)
            try:
                n, done = reader.emit(bufs[0], bufs[1], bufs[2])
                return bufs, n, done
            except ValueError as exc:                     # a read longer than the buffers hold: grow and retry
                if "buffers hold" in str(exc) and rows < (1 << 28):   # (as BamColumnReader.read_all does)
                    rows *= 4
                    continue
                raise

    def consume(bufs, n):
        nonlocal pushed
        if n:
            builder.push(bufs[0], bufs[1], bufs[2], order_base=pushed, n=n)
            pushed += n

    try:
        _feed(fill, consume, depth)
    finally:
        if pinned:
            _release(sets)
    return pushed


def stream_collated(reader, builder, chunk_rows=1 << 21, pinned=True, depth=3):
    """Collate the valid alignments of `reader` (bamcols.BamColumnReader, tables set) by read name on the GPU and
    push them into `builder` as name-grouped reads (_native.Collator).  A worker thread fills a small ring of pinned
    buffers from emit_keys while the previous buffer is added.  Returns (valid alignments, reads, collator stats)."""
    from ._native import Collator
    sets, added = [], 0

    def fill(bufs):
        if bufs is None:
            bufs = _buffers(chunk_rows, ("int64", "int64", "int32", "int32"), pinned)
            sets.append(bufs)
        n, done = reader.emit_keys(*bufs)
        return bufs, n, done

    with Collator(builder) as col:
        def consume(bufs, n):
            nonlocal added
            if n:
                col.add(*bufs, n=n)
                added += n

        try:
            _feed(fill, consume, depth)
        finally:
            if pinned:
                _release(sets)
        reads = col.push()
        return added, reads, col.stats()


def stream_single_device(path, reader, builder, tables, track_ranges, max_bytes=128 << 20, depth=3):
    """Decode the single-sample BAM file `path` on the GPU (_native.BamDecoder on `builder`'s context) and push
    its columns.  `reader` (bamcols.BamColumnReader of the same file) lists the BGZF blocks; a worker thread reads
    runs of whole blocks (up to max_bytes) into a small ring of pinned buffers while the previous run is decoded.
    order_base = rows pushed so far, so the result equals stream_single's.  A call's blocks are inflated one thread
    per block, so runs are large: a 128 MiB run holds a few thousand blocks.
    Returns (valid alignments, (all_alignments, n_groups), (range_min, range_max) or None, decoder stats)."""
    from ._native import BamDecoder
    first = reader.plan_shards(1)[0]                      # virtual offset of the first record
    cap = int(max_bytes) + (1 << 17)                      # a run holds at least one block (< 64 KiB + header)
    c, skip, pushed, sets = first >> 16, first & 0xFFFF, 0, []
    with BamDecoder(builder, tables.tid_target, tables.tid_hap, track_ranges) as dec, open(path, "rb") as fh:
        def fill(buf):
            nonlocal c
            off, length, isize, c_end = reader.blocks(c, max_bytes)
            if len(off) == 0:
                return buf, None, True
            if buf is None:
                buf = _buffers(cap, ("uint8",), True)
                sets.append(buf)
            n = c_end - c
            fh.seek(c)
            if fh.readinto(memoryview(buf[0].numpy())[:n]) != n:
                raise IOError("%s changed while it was read" % path)
            c = c_end
            return buf, (n, (off, length, isize)), False

        def consume(buf, run):
            nonlocal skip, pushed
            if run is None:                               # the end of the file
                rg, tg, hp = dec.decode(np.zeros(0, np.uint8), [], [], [], last=True)
            else:
                rg, tg, hp = dec.decode(buf[0], *run[1], skip=skip, n_bytes=run[0])
                skip = 0
            rows = int(rg.shape[0])
            if rows:
                builder.push(rg, tg, hp, order_base=pushed, n=rows)
                pushed += rows

        try:
            _feed(fill, consume, depth)
        finally:
            _release(sets)
        return pushed, dec.counters(), dec.ranges() if track_ranges else None, dec.stats()


def stream_files(bam_files, tables, cells, builder, order_base=0, n_threads=0, track_ranges=False):
    """Decode the per-cell BAM files in order on a worker thread, one file ahead of the push, so that at most two
    decoded files are in host memory, and push every file whole into `builder` (with cells) at order keys from
    `order_base` on.  One push per file: the file is part of the (file, EC, cell) key and its last read is dropped
    (drop_last_group; bam_utils_multisample.py:306-308).  tables: the job's target tables; cells: the
    bamcols.CellDictionary that gives the cell ids.
    Returns (alignments pushed, (range_min, range_max) over the files or None without track_ranges or files)."""
    todo = collections.deque(bam_files)
    pushed, lo, hi = 0, None, None

    def fill(_):
        with bamcols.BamColumnReader(todo.popleft(), n_threads=n_threads) as reader:
            reader.set_tables(tables)
            if track_ranges:
                reader.track_ranges(True)
            cols = reader.read_all(cells=cells, chunk=1 << 23)
            ranges = reader.ranges() if track_ranges else None
        return None, (cols, ranges), not todo

    def consume(_, item):
        nonlocal pushed, lo, hi
        cols, ranges = item
        builder.push(cols["read_group"], cols["target_idx"], cols["hap_idx"], cols["cell_idx"],
                     order_base=order_base + pushed, drop_last_group=True)
        pushed += len(cols["read_group"])
        if ranges is not None:                            # merged over the files (bam_utils_multisample.py:568-576)
            lo = ranges[0] if lo is None else np.minimum(lo, ranges[0])
            hi = ranges[1] if hi is None else np.maximum(hi, ranges[1])

    if todo:
        _feed(fill, consume, 2)
    return pushed, None if lo is None else (lo, hi)


def read_bam(filename):
    """(BamHeader, record iterator) using the built-in reader."""
    raw = bam_io.inflate_file(filename)
    header = bam_io.parse_header(raw)
    return header, bam_io.iter_records(raw, header.records_offset)
