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
import numpy as np

from . import bam_io


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


_PINNED_POOL = []      # pinned buffer sets of finished conversions, reused by the next one in this process


def _column_buffers(rows, with_cells, pinned):
    n = 4 if with_cells else 3
    if pinned:
        import torch
        # pinning host memory costs about as much as decoding it: a set that an earlier convert() of this
        # process has pinned is taken again when it is large enough
        for i, bufs in enumerate(_PINNED_POOL):
            if len(bufs) == n and int(bufs[0].shape[0]) >= rows:
                return _PINNED_POOL.pop(i)
        return [torch.empty(rows, dtype=torch.int32, pin_memory=True) for _ in range(n)]
    return [np.empty(rows, dtype=np.int32) for _ in range(n)]


def _release_buffers(sets, pinned):
    """Buffer sets of a finished stream go back to the pool (at most 8 sets are kept)."""
    if pinned:
        for bufs in sets:
            if len(_PINNED_POOL) < 8:
                _PINNED_POOL.append(bufs)


def stream_single(reader, builder, chunk_rows=1 << 21, pinned=True, depth=3):
    """Decode `reader` (bamcols.BamColumnReader, tables set) on a worker thread into a small ring of
    pinned buffers and push every filled buffer to the GPU while the next one is being decoded.
    Chunks end on read boundaries (bamcols_emit never splits a read), order_base = rows pushed so far,
    so the result equals one push of the whole file.  Returns the number of valid alignments."""
    import queue
    import threading
    free, full = queue.Queue(), queue.Queue()
    allocated = [0]
    all_sets = []
    stop = threading.Event()
    rows = [int(chunk_rows)]

    def next_buffers():
        """A free buffer set; a new one is pinned only when all existing ones are in flight."""
        while not stop.is_set():
            try:
                bufs = free.get_nowait()
            except queue.Empty:
                if allocated[0] < depth:
                    allocated[0] += 1
                    bufs = _column_buffers(rows[0], False, pinned)
                    all_sets.append(bufs)
                    return bufs
                try:
                    bufs = free.get(timeout=0.05)
                except queue.Empty:
                    continue
            if int(bufs[0].shape[0]) >= rows[0]:
                return bufs
            allocated[0] -= 1                             # a set from before the buffers grew: let it go
        return None

    def produce():
        try:
            while not stop.is_set():
                bufs = next_buffers()
                if bufs is None:
                    return
                try:
                    n, done = reader.emit(bufs[0], bufs[1], bufs[2])
                except ValueError as exc:                 # a read longer than the buffers hold: grow and retry
                    if "buffers hold" in str(exc) and rows[0] < (1 << 28):   # (as BamColumnReader.read_all does)
                        rows[0] *= 4
                        allocated[0] -= 1
                        continue
                    raise
                full.put((bufs, n, done, None))
                if done:
                    return
        except BaseException as exc:                      # re-raised by the consumer
            full.put((None, 0, True, exc))

    worker = threading.Thread(target=produce, daemon=True)
    worker.start()
    pushed = 0
    try:
        while True:
            bufs, n, done, exc = full.get()
            if exc is not None:
                raise exc
            if n:
                builder.push(bufs[0], bufs[1], bufs[2], order_base=pushed, n=n)
                pushed += n
            free.put(bufs)
            if done:
                break
    finally:
        # whatever happened, the producer has left native code before the caller may close the reader:
        # bamcols_close frees what bamcols_emit is working on
        stop.set()
        worker.join()
        _release_buffers(all_sets, pinned)
    return pushed


_PINNED_KEYS = []      # pinned key buffer sets of finished collations, reused by the next one in this process


def stream_collated(reader, builder, chunk_rows=1 << 21, pinned=True, depth=3):
    """Collate the valid alignments of `reader` (bamcols.BamColumnReader, tables set) by read name on the GPU and
    push them into `builder` as name-grouped reads (_native.Collator).  A worker thread fills a small ring of pinned
    buffers from emit_keys while the previous buffer is added.  Returns (valid alignments, reads, collator stats)."""
    import queue
    import threading
    from ._native import Collator
    free, full = queue.Queue(), queue.Queue()
    sets = []
    for _ in range(depth):
        bufs = None
        if pinned:
            import torch
            while _PINNED_KEYS and bufs is None:
                b = _PINNED_KEYS.pop()
                if int(b[0].shape[0]) >= chunk_rows:
                    bufs = b
            if bufs is None:
                bufs = [torch.empty(chunk_rows, dtype=torch.int64, pin_memory=True) for _ in range(2)] + \
                       [torch.empty(chunk_rows, dtype=torch.int32, pin_memory=True) for _ in range(2)]
        else:
            bufs = [np.empty(chunk_rows, np.uint64), np.empty(chunk_rows, np.uint64), np.empty(chunk_rows, np.int32),
                    np.empty(chunk_rows, np.int32)]
        sets.append(bufs)
        free.put(bufs)
    stop = threading.Event()

    def produce():
        try:
            while not stop.is_set():
                try:
                    bufs = free.get(timeout=0.05)
                except queue.Empty:
                    continue
                n, done = reader.emit_keys(*bufs)
                full.put((bufs, n, done, None))
                if done:
                    return
        except BaseException as exc:                      # re-raised by the consumer
            full.put((None, 0, True, exc))

    added = 0
    with Collator(builder) as col:
        worker = threading.Thread(target=produce, daemon=True)
        worker.start()
        try:
            while True:
                bufs, n, done, exc = full.get()
                if exc is not None:
                    raise exc
                if n:
                    col.add(*bufs, n=n)
                    added += n
                free.put(bufs)
                if done:
                    break
        finally:
            # the producer leaves native code before the caller may close the reader (as in stream_single)
            stop.set()
            worker.join()
            if pinned:
                _PINNED_KEYS.extend(sets)
        reads = col.push()
        return added, reads, col.stats()


_PINNED_BYTES = []     # pinned read buffers of finished device decodes, reused by the next one in this process


def stream_single_device(path, reader, builder, tables, track_ranges, max_bytes=128 << 20, depth=3):
    """Decode the single-sample BAM file `path` on the GPU (_native.BamDecoder on `builder`'s context) and push
    its columns.  `reader` (bamcols.BamColumnReader of the same file) lists the BGZF blocks; a worker thread reads
    runs of whole blocks (up to max_bytes) into a small ring of pinned buffers while the previous run is decoded.
    order_base = rows pushed so far, so the result equals stream_single's.  A call's blocks are inflated one thread
    per block, so runs are large: a 128 MiB run holds a few thousand blocks.
    Returns (valid alignments, (all_alignments, n_groups), (range_min, range_max) or None, decoder stats)."""
    import queue
    import threading
    import torch
    from ._native import BamDecoder
    first = reader.plan_shards(1)[0]                      # virtual offset of the first record
    free, full = queue.Queue(), queue.Queue()
    cap = int(max_bytes) + (1 << 17)                      # a run holds at least one block (< 64 KiB + header)
    bufs = []
    while _PINNED_BYTES and len(bufs) < depth:           # pinning costs about as much as reading the bytes
        b = _PINNED_BYTES.pop()
        if int(b.shape[0]) >= cap:
            bufs.append(b)
    bufs += [torch.empty(cap, dtype=torch.uint8, pin_memory=True) for _ in range(depth - len(bufs))]
    for b in bufs:
        free.put(b)
    stop = threading.Event()

    def produce():
        try:
            c = first >> 16
            with open(path, "rb") as fh:
                while not stop.is_set():
                    off, length, isize, c_end = reader.blocks(c, max_bytes)
                    if len(off) == 0:
                        full.put((None, 0, None, None))
                        return
                    buf = None
                    while buf is None and not stop.is_set():
                        try:
                            buf = free.get(timeout=0.05)
                        except queue.Empty:
                            pass
                    if buf is None:
                        return
                    n = c_end - c
                    fh.seek(c)
                    if fh.readinto(memoryview(buf.numpy())[:n]) != n:
                        raise IOError("%s changed while it was read" % path)
                    full.put((buf, n, (off, length, isize), None))
                    c = c_end
        except BaseException as exc:                      # re-raised by the consumer
            full.put((None, 0, None, exc))

    pushed = 0
    with BamDecoder(builder, tables.tid_target, tables.tid_hap, track_ranges) as dec:
        worker = threading.Thread(target=produce, daemon=True)
        worker.start()
        try:
            skip = first & 0xFFFF
            while True:
                buf, n, table, exc = full.get()
                if exc is not None:
                    raise exc
                if buf is None:
                    rg, tg, hp = dec.decode(np.zeros(0, np.uint8), [], [], [], last=True)
                else:
                    rg, tg, hp = dec.decode(buf, *table, skip=skip, n_bytes=n)
                    skip = 0
                rows = int(rg.shape[0])
                if rows:
                    builder.push(rg, tg, hp, order_base=pushed, n=rows)
                    pushed += rows
                if buf is None:
                    break
                free.put(buf)
        finally:
            stop.set()
            worker.join()
            _PINNED_BYTES.extend(bufs)
        return pushed, dec.counters(), dec.ranges() if track_ranges else None, dec.stats()


def read_bam(filename):
    """(BamHeader, record iterator) using the built-in reader."""
    raw = bam_io.inflate_file(filename)
    header = bam_io.parse_header(raw)
    return header, bam_io.iter_records(raw, header.records_offset)
