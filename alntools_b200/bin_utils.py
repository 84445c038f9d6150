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
