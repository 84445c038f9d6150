"""EC binary file (format 2) writer/reader fed by device-built arrays.

Byte layout = alntools/bin_utils.ecsave2 (bin_utils.py:105-277): every integer a little-endian int32,
strings raw UTF-8 with an int32 length prefix, no padding:
    2 | H | H x [len, bytes] | T | T x [len, bytes, H x length] | S | S x [len, bytes]
    | A (CSR, E x T): len(indptr)=E+1, nnz, indptr, indices, data (haplotype bitmask)
    | N (CSC, E x S): len(indptr)=S+1, nnz, indptr, indices (EC ids), data (counts)
The reference packs every array with struct.pack('<{n}i', *arr) (one Python int per element);
ndarray.astype('<i4').tobytes() yields the same bytes.
"""
import os
import struct

import numpy as np


def _i32(arr):
    """Little-endian int32 bytes of `arr` without a copy when it already is a contiguous int32 array
    (the library's result buffers are written to the file directly)."""
    a = np.ascontiguousarray(arr, dtype="<i4")
    return a.data if a.size else b""


def _name_bytes(name):
    """The bytes ecsave2 writes for a name: pack('<{len(name)}s', name.encode()) keeps len(name) BYTES, so a
    non-ASCII name is cut inside its UTF-8 encoding (bin_utils.py:131-135,153-159,177-180).  Same here, so the
    file stays byte-identical and the length prefix always matches what follows."""
    if isinstance(name, bytes):                      # a name as read from an EC file: written as it was
        return name
    return name.encode("utf-8")[:len(name)]


def _target_section(target_names, lengths, n_haps):
    """T x [len(name), name bytes, H x length] (bin_utils.py:153-159).  ASCII names (every aligner
    index) are laid out with numpy scatters; anything else takes the per-name loop."""
    joined = "".join(target_names)
    n = len(target_names)
    if n == 0:
        return b""
    if not joined.isascii():
        parts = []
        for idx, name in enumerate(target_names):
            parts.append(struct.pack("<i", len(name)))
            parts.append(_name_bytes(name))
            parts.append(_i32(lengths[idx, :n_haps]))
        return b"".join(parts)
    nb = np.fromiter(map(len, target_names), dtype=np.int64, count=n)
    rec = 4 + nb + 4 * n_haps
    start = np.cumsum(rec) - rec
    out = np.empty(int(rec.sum()), dtype=np.uint8)
    out[start[:, None] + np.arange(4)] = nb.astype("<i4").view(np.uint8).reshape(n, 4)
    name_first = np.cumsum(nb) - nb
    out[np.repeat(start + 4 - name_first, nb) + np.arange(int(nb.sum()))] = np.frombuffer(joined.encode("ascii"),
                                                                                         dtype=np.uint8)
    if n_haps:
        lens = np.ascontiguousarray(lengths[:, :n_haps], dtype="<i4").view(np.uint8).reshape(n, 4 * n_haps)
        out[(start + 4 + nb)[:, None] + np.arange(4 * n_haps)] = lens
    return out.tobytes()


def ecsave2_arrays(ec_filename, haplotypes, target_names, lengths, sample_names, a_csr, n_csc, target_section=None,
                   n_targets=None):
    """a_csr / n_csc: (indptr, indices, data) int32 arrays.  target_section (with n_targets): the bytes of the
    targets section when the caller already has them (the native header tables build them without creating
    a Python string per target); then target_names / lengths are not looked at."""
    with open(ec_filename, "wb") as fh:
        fh.write(struct.pack("<i", 2))
        fh.write(struct.pack("<i", len(haplotypes)))
        for hap in haplotypes:
            fh.write(struct.pack("<i", len(hap)))
            fh.write(_name_bytes(hap))
        if target_section is not None:
            fh.write(struct.pack("<i", int(n_targets)))
            fh.write(target_section)
        else:
            lengths = np.asarray(lengths).astype(int)
            fh.write(struct.pack("<i", len(target_names)))
            fh.write(_target_section(target_names, lengths, len(haplotypes)))
        fh.write(struct.pack("<i", len(sample_names)))
        parts = []
        for sample in sample_names:
            parts.append(struct.pack("<i", len(sample)))
            parts.append(_name_bytes(sample))
        fh.write(b"".join(parts))
        for indptr, indices, data in (a_csr, n_csc):
            fh.write(struct.pack("<i", len(indptr)))
            fh.write(struct.pack("<i", len(indices)))
            fh.write(_i32(indptr))
            fh.write(_i32(indices))
            fh.write(_i32(data))


def ec_header_bytes(haplotypes, target_names, lengths, sample_names, target_section=None, n_targets=None):
    """The sections of an EC file in front of the matrices (format tag, haplotypes, targets, samples), as
    ecsave2_arrays writes them."""
    parts = [struct.pack("<i", 2), struct.pack("<i", len(haplotypes))]
    for hap in haplotypes:
        parts.append(struct.pack("<i", len(hap)))
        parts.append(_name_bytes(hap))
    if target_section is not None:
        parts.append(struct.pack("<i", int(n_targets)))
        parts.append(bytes(target_section))
    else:
        parts.append(struct.pack("<i", len(target_names)))
        parts.append(_target_section(target_names, np.asarray(lengths).astype(int), len(haplotypes)))
    parts.append(struct.pack("<i", len(sample_names)))
    for sample in sample_names:
        parts.append(struct.pack("<i", len(sample)))
        parts.append(_name_bytes(sample))
    return b"".join(parts)


def _a_layout(header_bytes, n_ec_total, nnz_total):
    """Byte offsets of the A (CSR) section behind the header: len(indptr), nnz, indptr[E + 1], indices[Z],
    data[Z].  -> (a_at, a_indptr_at, a_indices_at, a_data_at, end)."""
    E, Z = int(n_ec_total), int(nnz_total)
    a_at = header_bytes
    a_indptr_at = a_at + 8
    a_indices_at = a_indptr_at + 4 * (E + 1)
    a_data_at = a_indices_at + 4 * Z
    return a_at, a_indptr_at, a_indices_at, a_data_at, a_data_at + 4 * Z


def _create_a(fh, header, n_ec_total, nnz_total):
    """Header sections, the A sizes and indptr[0] (the part of the file only its creator writes)."""
    fh.write(header)
    fh.write(struct.pack("<ii", int(n_ec_total) + 1, int(nnz_total)))
    fh.write(struct.pack("<i", 0))


def _write_a_slice(fd, layout, id_base, nnz_base, a_indptr_local, a_indices, a_data):
    """A slice's byte ranges of the A section: indptr[id_base + 1 ..], indices and data at nnz_base."""
    _, a_indptr_at, a_indices_at, a_data_at, _ = layout
    if len(a_indptr_local) > 1:
        indptr = (np.asarray(a_indptr_local[1:], dtype=np.int64) + int(nnz_base)).astype("<i4")
        os.pwrite(fd, _i32(indptr), a_indptr_at + 4 * (int(id_base) + 1))
    if len(a_indices):
        os.pwrite(fd, _i32(a_indices), a_indices_at + 4 * int(nnz_base))
        os.pwrite(fd, _i32(a_data), a_data_at + 4 * int(nnz_base))


def ecsave2_slice(ec_filename, header, n_ec_total, nnz_total, id_base, nnz_base, a_indptr_local, a_indices, a_data,
                  counts, create):
    """Single-sample EC file written by several processes, each holding the ECs [id_base, id_base + n) of the
    final matrices (the multi-GPU build leaves them partitioned by EC-id range): every process writes its
    own byte ranges of the A (CSR) and N (CSC, one sample) sections; the one with create=True also lays the
    file out (header sections, the four size fields, indptr[0], N's indptr) and must run first.
    a_indptr_local: [n + 1] offsets local to the slice (a_indptr_local[0] == 0); nnz_base = non-zeros of the
    slices in front.  Same bytes as ecsave2_arrays on the assembled matrices (alntools/bin_utils.py:105-277)."""
    E = int(n_ec_total)
    n = len(counts)
    layout = _a_layout(len(header), n_ec_total, nnz_total)
    n_at = layout[4]                             # N: 2, E, [0, E], indices[E] = 0..E-1, data[E] = counts
    n_indices_at = n_at + 16
    n_data_at = n_indices_at + 4 * E
    total = n_data_at + 4 * E
    if create:
        with open(ec_filename, "wb") as fh:
            _create_a(fh, header, n_ec_total, nnz_total)
            fh.truncate(total)
            fh.seek(n_at)
            fh.write(struct.pack("<iiii", 2, E, 0, E))
    fd = os.open(ec_filename, os.O_WRONLY)
    try:
        _write_a_slice(fd, layout, id_base, nnz_base, a_indptr_local, a_indices, a_data)
        if n:
            os.pwrite(fd, _i32(np.arange(int(id_base), int(id_base) + n, dtype=np.int32)), n_indices_at + 4 * int(id_base))
            os.pwrite(fd, _i32(counts), n_data_at + 4 * int(id_base))
    finally:
        os.close(fd)


def ecsave2_cells_slice(ec_filename, header, n_ec_total, nnz_total, id_base, nnz_base, a_indptr_local, a_indices, a_data,
                        n_indptr, n_col_counts, n_col_offset, n_indices_local, n_data, create):
    """Per-cell EC file written by several processes, each holding the ECs [id_base, id_base + n) (as
    ecsave2_slice; `header` names the cells in column order).  The A part is written as by ecsave2_slice.  N
    (CSC, E x S): this process holds, for every column c, n_col_counts[c] entries (n_indices_local: EC ids local
    to the slice, ascending inside a column; n_data: counts; both in column-major order); they go to
    n_indptr[c] + n_col_offset[c] on, where n_col_offset[c] = entries of column c held by the slices in front in
    id order, in one vectorised scatter.  The process with create=True lays the file out (header, sizes, the
    global n_indptr [S + 1]) and must run first.  Same bytes as ecsave2_arrays on the assembled matrices."""
    n_indptr = np.asarray(n_indptr, dtype=np.int64)
    S, nnz_n = len(n_indptr) - 1, int(n_indptr[-1])
    layout = _a_layout(len(header), n_ec_total, nnz_total)
    n_at = layout[4]                             # N: S + 1, nnz, indptr[S + 1], indices[nnz], data[nnz]
    n_indices_at = n_at + 8 + 4 * (S + 1)
    n_data_at = n_indices_at + 4 * nnz_n
    if create:
        with open(ec_filename, "wb") as fh:
            _create_a(fh, header, n_ec_total, nnz_total)
            fh.truncate(n_data_at + 4 * nnz_n)
            fh.seek(n_at)
            fh.write(struct.pack("<ii", S + 1, nnz_n))
            fh.write(_i32(n_indptr.astype("<i4")))
    fd = os.open(ec_filename, os.O_WRONLY)
    try:
        _write_a_slice(fd, layout, id_base, nnz_base, a_indptr_local, a_indices, a_data)
    finally:
        os.close(fd)
    counts = np.asarray(n_col_counts, dtype=np.int64)
    m = int(counts.sum())
    if m:
        if len(n_indices_local) != m or len(n_data) != m:
            raise ValueError("%d N entries given, the column counts say %d" % (len(n_indices_local), m))
        starts = np.cumsum(counts) - counts
        col = np.repeat(np.arange(S), counts)
        dest = n_indptr[col] + np.asarray(n_col_offset, dtype=np.int64)[col] + (np.arange(m) - starts[col])
        section = np.memmap(ec_filename, dtype="<i4", mode="r+", offset=n_indices_at, shape=(2, nnz_n))
        section[0, dest] = np.asarray(n_indices_local, dtype=np.int64) + int(id_base)
        section[1, dest] = n_data
        section.flush()
        del section


def ecload_arrays(ec_filename):
    """Inverse of ecsave2_arrays (what bin_utils.ecload :32-102 / bin_file.ECFile :99-402 parse)."""
    with open(ec_filename, "rb") as fh:
        buf = fh.read()
    pos = [0]

    def i32():
        v = struct.unpack_from("<i", buf, pos[0])[0]
        pos[0] += 4
        return v

    def text():
        n = i32()
        s = buf[pos[0]:pos[0] + n].decode("utf-8", errors="replace")   # (a cut non-ASCII name: see _name_bytes)
        pos[0] += n
        return s

    def arr(n):
        a = np.frombuffer(buf, dtype="<i4", count=n, offset=pos[0]).copy()
        pos[0] += 4 * n
        return a

    fmt = i32()
    if fmt != 2:
        raise ValueError("only EC format 2 is supported, found %d" % fmt)
    haplotypes = [text() for _ in range(i32())]
    n_targets = i32()
    targets = []
    lengths = np.zeros((n_targets, len(haplotypes)), dtype=np.int32)
    for t in range(n_targets):
        targets.append(text())
        lengths[t] = arr(len(haplotypes))
    samples = [text() for _ in range(i32())]
    mats = []
    for _ in range(2):
        n_ptr, nnz = i32(), i32()
        mats.append((arr(n_ptr), arr(nnz), arr(nnz)))
    if pos[0] != len(buf):
        raise ValueError("trailing bytes in EC file")
    return {"haplotypes": haplotypes, "targets": targets, "lengths": lengths, "samples": samples,
            "a": mats[0], "n": mats[1]}


def save_outputs(tables, section, sample_names, a_csr, n_csc, cells, ec_filename=None, emase_filename=None,
                 range_filename=None, references=None, ranges=None):
    """Write the outputs of a conversion that were asked for, each in place of an old file of that name: the EMASE
    and EC files from the final host matrices a_csr / n_csc (as alntools/bam_utils.py:726-876 does), and the
    --rangefile report from the header's reference names and the (range_min, range_max) arrays per reference.
    section: the targets section the native header tables built (TargetTables.target_section(), read while their
    reader is open), or None; without an EMASE file, which needs the name list anyway, it saves building the names.
    cells: the per-cell converter, whose EMASE file is titled "Multisample APM" and keeps the counts; the
    single-sample one is titled "bam2ec" and is incidence only."""
    from . import emase, utils
    target_names = list(tables.main_targets.keys()) if (emase_filename or section is None) else None
    if emase_filename:
        utils.delete_file(emase_filename)
        emase.save_emase(emase_filename, "Multisample APM" if cells else "bam2ec",
                         (tables.num_targets, tables.num_haplotypes, len(a_csr[0]) - 1), tables.haplotypes,
                         target_names, tables.lengths, sample_names, a_csr, n_csc, incidence_only=not cells)
    if ec_filename:
        utils.delete_file(ec_filename)
        ecsave2_arrays(ec_filename, tables.haplotypes, target_names, tables.lengths, sample_names, a_csr, n_csc,
                       target_section=section, n_targets=tables.num_targets)
    if range_filename is not None:
        utils.write_range_file(range_filename, list(tables.main_targets.keys()), tables.haplotypes, references,
                               ranges[0], ranges[1])


def ec2emase(ec_filename, emase_filename):
    """EC binary file -> EMASE (.h5) file (alntools/bin_utils.py:979-995: ecload, then APM.save with the title
    'Converted from <ec file>' and the data arrays included).  Needs PyTables like every EMASE output."""
    import os
    from . import emase
    ec = ecload_arrays(ec_filename)
    try:
        os.remove(emase_filename)
    except OSError:
        pass
    shape = (len(ec["targets"]), len(ec["haplotypes"]), len(ec["a"][0]) - 1)
    emase.save_emase(emase_filename, "Converted from {}".format(ec_filename), shape, ec["haplotypes"], ec["targets"],
                     ec["lengths"], ec["samples"], ec["a"], ec["n"], incidence_only=False, as_ecload=True)


def _ec_sections(path, first=None):
    """Where the sections of EC file `path` (format 2) lie, read without its matrices: -> dict(header: the bytes from
    the format word to the end of the targets section, haplotypes: their names as bytes, n_targets, section: the bytes
    of the targets after their count, samples: names as bytes, matrices_at, n_ec, nnz_a, n_cols, nnz_n, size).
    `first`: the sections of the first file of a merge, whose header this file must repeat byte for byte.  Raises
    ValueError naming the file when it is not a well-formed file of format 2 or has no sample."""
    import mmap
    size = os.path.getsize(path)
    with open(path, "rb") as fh:
        if size < 4:
            raise ValueError("%s: truncated EC file" % path)
        with mmap.mmap(fh.fileno(), 0, access=mmap.ACCESS_READ) as mm:
            pos = [0]

            def i32():
                if pos[0] + 4 > size:
                    raise ValueError("%s: truncated EC file" % path)
                v = struct.unpack_from("<i", mm, pos[0])[0]
                pos[0] += 4
                return v

            def skip(n, what):
                if n < 0 or pos[0] + n > size:
                    raise ValueError("%s: truncated EC file (%s)" % (path, what))
                start = pos[0]
                pos[0] += n
                return start

            def name(what):
                n = i32()
                return bytes(mm[skip(n, what):pos[0]])

            fmt = i32()
            if fmt != 2:
                raise ValueError("%s: not an EC file of format 2 (format %d)" % (path, fmt))
            if first is not None:
                h = first["header"]
                if size < len(h):
                    raise ValueError("%s: truncated EC file (header)" % path)
                if mm[:len(h)] != h:
                    raise ValueError("%s: its haplotype or target section differs from that of %s" % (path, first["path"]))
                pos[0] = len(h)
                out = dict(first)
            else:
                n_haps = i32()
                if n_haps < 0:
                    raise ValueError("%s: negative number of haplotypes" % path)
                haplotypes = [name("haplotype names") for _ in range(n_haps)]
                n_targets = i32()
                if n_targets < 0:
                    raise ValueError("%s: negative number of targets" % path)
                section_at = pos[0]
                for _ in range(n_targets):
                    skip(i32(), "target names")
                    skip(4 * n_haps, "target lengths")
                out = {"header": bytes(mm[:pos[0]]), "haplotypes": haplotypes, "n_targets": n_targets,
                       "section": bytes(mm[section_at:pos[0]])}
            n_samples = i32()
            if n_samples <= 0:
                raise ValueError("%s: an EC file needs at least one sample, found %d" % (path, n_samples))
            samples = [name("sample names") for _ in range(n_samples)]
            matrices_at = pos[0]
            a_ptr, nnz_a = i32(), i32()
            if a_ptr < 1 or nnz_a < 0:
                raise ValueError("%s: inconsistent A sizes (%d offsets, %d entries)" % (path, a_ptr, nnz_a))
            skip(4 * (a_ptr + 2 * nnz_a), "A matrix")
            n_ptr, nnz_n = i32(), i32()
            if n_ptr != n_samples + 1 or nnz_n < 0:
                raise ValueError("%s: inconsistent N sizes (%d offsets for %d samples, %d entries)"
                                 % (path, n_ptr, n_samples, nnz_n))
            skip(4 * (n_ptr + 2 * nnz_n), "N matrix")
            if pos[0] != size:
                raise ValueError("%s: trailing bytes in EC file (%d)" % (path, size - pos[0]))
    out.update(path=path, samples=samples, matrices_at=matrices_at, n_ec=a_ptr - 1, nnz_a=nnz_a, n_cols=n_samples,
               nnz_n=nnz_n, size=size)
    return out


def _ec_matrices(sec):
    """The A and N arrays of a file described by _ec_sections, read at once: int32 views of one buffer."""
    buf = np.fromfile(sec["path"], dtype="<i4", count=(sec["size"] - sec["matrices_at"]) // 4, offset=sec["matrices_at"])
    e, za, s, zn = sec["n_ec"], sec["nnz_a"], sec["n_cols"], sec["nnz_n"]
    at = [2]

    def take(n):
        v = buf[at[0]:at[0] + n]
        at[0] += n
        return v

    a = (take(e + 1), take(za), take(za))
    at[0] += 2
    return a, (take(s + 1), take(zn), take(zn))


def merge_ec_files(ec_files, ec_filename, sample_names=None, device=0):
    """Merge EC files (format 2) into one EC file with one shared EC index, on one GPU.

    Every file must have the first file's haplotype and target sections, byte for byte; the output takes them.  An EC
    is a distinct A row (a set of (target, haplotype) elements): the output holds every distinct row of the inputs,
    and its EC ids follow the row's first appearance as (file index, id in that file).  N has the columns of every
    file in order, each entry moved to the merged id of its row; zeros are not stored and ids ascend in a column.
    Columns are never joined by name.  The samples are the inputs' sample lists back to back, or sample_names (one per
    output column).  EC ids being ranks of first occurrence, the merge of convert() outputs of several BAM files is the
    file convert_samples() writes for those files, and merging is associative.

    Every file is checked (format, sizes, samples, header) before a GPU is touched or the output is written; values
    the GPU finds malformed (a target out of range, unsorted or empty rows, bad masks, repeated rows, N indices out of
    range, negative counts) raise ValueError naming the file.  The next file is read on a worker thread while the
    current one is pushed, so at most two files are in host memory.  One GPU: inside a multi-GPU launcher or with
    ALNTOOLS_GPUS > 1 it raises NotImplementedError, as it does for an EMASE (.h5) output (ec2emase converts the
    merged file).  -> dict(n_ec, nnz_a, nnz_n, n_samples, ecs_added (per file), seconds (read, push, finalize, write))."""
    import time
    from . import utils
    from .emitter import _feed
    ec_files = [str(f) for f in ec_files]
    if not ec_files:
        raise ValueError("merge_ec_files needs at least one EC file")
    if str(ec_filename).lower().endswith(".h5"):
        raise NotImplementedError("merge_ec_files writes EC files only; convert the merged file with ec2emase")
    if utils.under_launcher() or utils.requested_gpus(None) > 1:
        raise NotImplementedError("merge_ec_files runs on one GPU (unset ALNTOOLS_GPUS, or run it outside a multi-GPU "
                                  "launcher)")
    secs = [_ec_sections(ec_files[0])]
    secs += [_ec_sections(f, secs[0]) for f in ec_files[1:]]
    names = [n for s in secs for n in s["samples"]]
    if sample_names is not None:
        sample_names = list(sample_names)
        if len(sample_names) != len(names):
            raise ValueError("%d sample names for %d columns" % (len(sample_names), len(names)))
        names = sample_names
    first = secs[0]
    from ._native import ECB_ERR_FORMAT, ECB_ERR_LIMIT, EcBuilder, EcbError
    seconds = {"read": 0.0, "push": 0.0, "finalize": 0.0, "write": 0.0}
    added = []
    todo = list(range(len(secs)))

    def fill(_):
        t0 = time.perf_counter()
        k = todo.pop(0)
        mats = _ec_matrices(secs[k])
        seconds["read"] += time.perf_counter() - t0
        return None, (k, mats), not todo

    with EcBuilder(max(first["n_targets"], 1), max(len(first["haplotypes"]), 1), device=device,
                   pageable_results=1) as builder:
        def consume(_, item):
            k, (a, n) = item
            t0 = time.perf_counter()
            before = builder.stats()["ec_claimed"]
            try:
                builder.push_ecs(*a)
                builder.append_samples(*n)
            except EcbError as exc:
                if exc.code in (ECB_ERR_FORMAT, ECB_ERR_LIMIT):
                    raise ValueError("%s: %s" % (ec_files[k], str(exc).split(": ", 1)[-1])) from None
                raise
            added.append(builder.stats()["ec_claimed"] - before)
            seconds["push"] += time.perf_counter() - t0

        _feed(fill, consume, 2)
        t0 = time.perf_counter()
        res = builder.finalize_samples(copy=False)
        seconds["finalize"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        utils.delete_file(ec_filename)
        ecsave2_arrays(ec_filename, first["haplotypes"], None, None, names,
                       (res["a_indptr"], res["a_indices"], res["a_data"]),
                       (res["n_indptr"], res["n_indices"], res["n_data"]), target_section=first["section"],
                       n_targets=first["n_targets"])
        seconds["write"] = time.perf_counter() - t0
        return {"n_ec": int(res["n_ec"]), "nnz_a": int(res["nnz_a"]), "nnz_n": int(res["nnz_n"]),
                "n_samples": int(res["n_samples"]), "ecs_added": added, "seconds": seconds}
