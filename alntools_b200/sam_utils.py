"""Single-sample conversion of SAM text (a file or standard input) into an EC file, parsed on the GPU.

The rule: SAM text S converts to the EC file (and --rangefile report) that bam_utils.convert() writes for the BAM file
B holding S's @SQ list as its references and, per alignment line, a record with refID = the @SQ index of RNAME ('*':
-1), pos = POS - 1, next_refID from RNEXT ('=': refID, '*': -1, else its @SQ index), next_pos = PNEXT - 1, and FLAG and
QNAME as written.  read_header and iter_records below state it in Python; convert_sam runs it on the GPU
(_native.SamDecoder), or through emitter.emit_single with ALNTOOLS_B200_EMITTER=python.

Call stack: convert_sam -> read_header (host) -> TargetTables -> a worker thread fills pinned buffers with whole lines
-> SamDecoder.parse (H2D + sm_100a kernels: lines, fields, rules) -> EcBuilder.push (device rows) -> finalize -> EC file.
"""
import os
import sys
import time

import numpy as np

from . import bin_utils, emitter, utils
from ._native import EcBuilder
from .header import TargetTables

LOG = utils.get_logger()

# What is wrong with a bad alignment line, by kind, in the order one line is checked.  The library (ecb_sam.cuh,
# sam_bad_line in ecb_api.cu) checks in the same order and words its messages the same way.
_BAD = {
    1: "a header line (starting with '@') after the first alignment line",
    2: "fewer than 11 tab-separated fields",
    3: "QNAME empty or longer than 254 bytes",
    4: "FLAG not a decimal integer in [0, 65535]",
    5: "RNAME not '*' and not an @SQ name",
    6: "POS not a decimal integer in [0, 2147483647]",
    7: "RNEXT not '*', '=' or an @SQ name",
    8: "PNEXT not a decimal integer in [0, 2147483647]",
}
_INT31 = (1 << 31) - 1


def _decimal(field, limit):
    """int(field) for a non-empty run of ASCII digits at most `limit`, else None."""
    if not field.isdigit():
        return None
    value = int(field)
    return value if value <= limit else None


def read_header(stream, name="SAM input"):
    """The header of a SAM stream (a binary buffered reader, positioned at its start): the run of lines at the start
    that begin with '@'.  Only @SQ lines are used, in order, through their SN: and LN: tags.  The stream is left at the
    first alignment line.  -> (references, lengths, header line count)."""
    if stream.peek(2)[:2] == b"\x1f\x8b":
        raise ValueError("%s is gzip-compressed (BGZF or gzip), not SAM text; convert BAM files with bam2ec" % name)
    references, lengths, n = [], [], 0
    while stream.peek(1)[:1] == b"@":
        line = stream.readline()
        n += 1
        fields = line.rstrip(b"\n").split(b"\t")
        if fields[0] != b"@SQ":
            continue
        sn = ln = None
        for tag in fields[1:]:
            if sn is None and tag.startswith(b"SN:"):
                sn = tag[3:]
            elif ln is None and tag.startswith(b"LN:"):
                ln = tag[3:]
        length = None if ln is None else _decimal(ln, _INT31)
        if sn is None or length is None:
            raise ValueError("%s: line %d: @SQ line without SN: or without a decimal LN: in [0, 2147483647]" % (name, n))
        references.append(sn.decode())                    # as bam_io.parse_header decodes @SQ names
        lengths.append(length)
    return tuple(references), tuple(lengths), n


def iter_records(stream, references, first_line, name="SAM input"):
    """Yield (qname, flag, tid, pos, next_tid, next_pos) per alignment line of `stream` (positioned after the header;
    its first line has number first_line), the tuples emitter.emit_single takes.  A bad line raises ValueError naming
    `name` and the line number; the checks run in the order of _BAD, then a valid alignment whose RNAME is '*' is the
    BAM path's refID error."""
    tid_of = {}
    for tid, ref in enumerate(references):
        tid_of.setdefault(ref.encode(), tid)
    for i, line in enumerate(stream):
        number = first_line + i
        if line.endswith(b"\n"):
            line = line[:-1]
        kind = 0
        if line[:1] == b"@":
            kind = 1
        elif line.count(b"\t") < 10:
            kind = 2
        else:
            qname, flag, rname, pos, _mapq, _cigar, rnext, pnext = line.split(b"\t", 8)[:8]
            flag, pos, pnext = _decimal(flag, 65535), _decimal(pos, _INT31), _decimal(pnext, _INT31)
            tid = -1 if rname == b"*" else tid_of.get(rname, -2)
            ntid = -1 if rnext == b"*" else tid if rnext == b"=" else tid_of.get(rnext, -2)
            if not qname or len(qname) > 254:
                kind = 3
            elif flag is None:
                kind = 4
            elif tid == -2:
                kind = 5
            elif pos is None:
                kind = 6
            elif ntid == -2:
                kind = 7
            elif pnext is None:
                kind = 8
            elif tid < 0 and emitter._valid(flag, tid, ntid, pnext - 1):
                raise ValueError("%s: line %d: alignment with reference id -1 outside the header's %d references"
                                 % (name, number, len(references)))
        if kind:
            raise ValueError("%s: line %d: %s" % (name, number, _BAD[kind]))
        yield qname.decode(), flag, tid, pos - 1, ntid, pnext - 1


def _last_newline(arr, n):
    """Offset of the last b'\\n' in arr[:n] (a uint8 array), or -1."""
    hi = n
    while hi > 0:
        lo = max(0, hi - (1 << 20))
        at = arr[lo:hi].tobytes().rfind(b"\n")
        if at >= 0:
            return lo + at
        hi = lo
    return -1


def stream_sam_device(stream, name, builder, tables, references, first_line, track_ranges, max_bytes=128 << 20, depth=3):
    """Parse the alignment lines of `stream` on the GPU (_native.SamDecoder on `builder`'s context) and push their rows.
    A worker thread fills a ring of pinned buffers of max_bytes: it reads until a buffer is full or the input ends (so a
    pipe that delivers small writes still gives large calls), cuts the buffer after its last '\\n' and carries the tail
    to the front of the next buffer; a line longer than a buffer makes the buffers grow.  order_base = rows pushed so
    far, so the result equals one push of the whole input.
    Returns (valid alignments, (all_alignments, n_groups), (range_min, range_max) or None, decoder stats)."""
    from ._native import SamDecoder
    size, tail, pushed, sets = max(1, int(max_bytes)), b"", 0, []

    def new_buffer(n):
        buf = emitter._buffers(n, ("uint8",), True)
        sets.append(buf)
        return buf

    with SamDecoder(builder, references, tables.tid_target, tables.tid_hap, first_line, track_ranges) as dec:
        def fill(buf):
            nonlocal size, tail
            if buf is None or int(buf[0].shape[0]) < size:
                buf = new_buffer(size)
            arr = buf[0].numpy()
            filled = len(tail)
            arr[:filled] = np.frombuffer(tail, dtype=np.uint8)
            while True:
                eof = False
                while filled < len(arr):
                    got = stream.readinto(memoryview(arr)[filled:])
                    if not got:
                        eof = True
                        break
                    filled += got
                if eof:
                    n, tail = filled, b""
                    break
                cut = _last_newline(arr, filled)
                if cut >= 0:
                    n, tail = cut + 1, arr[cut + 1:filled].tobytes()
                    break
                size = 2 * len(arr)                       # a line longer than the buffer
                grown = new_buffer(size)
                grown[0].numpy()[:filled] = arr[:filled]
                buf, arr = grown, grown[0].numpy()
            return buf, (n, eof), eof

        def consume(buf, item):
            nonlocal pushed
            n, last = item
            try:
                rg, tg, hp = dec.parse(buf[0], n, last=last)
            except ValueError as exc:
                raise ValueError("%s: %s" % (name, exc)) from None
            rows = int(rg.shape[0])
            if rows:
                builder.push(rg, tg, hp, order_base=pushed, n=rows)
                pushed += rows

        try:
            emitter._feed(fill, consume, depth)
        finally:
            emitter._release(sets)
        return pushed, dec.counters(), dec.ranges() if track_ranges else None, dec.stats()


def convert_sam(sam_filename, ec_filename, range_filename=None, sample=None, target_filename=None, device=0,
                max_bytes=128 << 20):
    """Convert single-sample SAM text into an EC file (and, with range_filename, the --rangefile report): the bytes
    bam_utils.convert() writes for the BAM file that holds the same alignments (see the module's rule).

    sam_filename: a path, or "-" for standard input (a pipe from the aligner works: the header is read first and the
    rest is streamed once).  sample: the sample name (default: the file's base name, "stdin" for "-").  target_filename,
    ALNTOOLS_B200_MAX_READ and ALNTOOLS_B200_EMITTER=python work as for convert(); ALNTOOLS_B200_DECODE concerns BAM
    files and is not read.  max_bytes: the size of one pinned text buffer (one library call).  A bad line raises
    ValueError naming the input and the line number, and nothing is written.  An EMASE (.h5) output, more than one GPU
    (ALNTOOLS_GPUS or a launcher), ALNTOOLS_B200_COLLATE=1 and --rangefile with the Python emitter are refused before
    the input is read."""
    start_time = time.time()
    if str(ec_filename).lower().endswith(".h5"):
        raise NotImplementedError("convert_sam writes EC files only; make the EMASE (.h5) file from the EC file with "
                                  "ec2emase")
    mode = emitter.resolve_mode(False, None, "host", None, range_filename is not None)
    if mode.launcher or mode.gpus > 1:
        raise NotImplementedError("SAM conversion runs on one GPU (unset ALNTOOLS_GPUS, or run it outside a multi-GPU "
                                  "launcher)")
    if mode.collate:
        raise NotImplementedError("SAM conversion has no collation by read name (unset ALNTOOLS_B200_COLLATE)")
    limit = emitter.max_read()
    stdin = sam_filename == "-"
    name = "stdin" if stdin else sam_filename
    if sample is None:
        sample = "stdin" if stdin else os.path.basename(sam_filename)
        LOG.info("Sample not supplied, using: {}".format(sample))
    stream = sys.stdin.buffer if stdin else open(sam_filename, "rb")
    try:
        references, lengths, n_header = read_header(stream, name)
        tables = TargetTables(references, lengths, target_filename)
        track = range_filename is not None

        def save(res, valid, ranges):
            LOG.info("# Valid Alignments: {:,}".format(valid))
            LOG.info("# Main Targets: {:,}".format(tables.num_targets))
            LOG.info("# Haplotypes: {:,}".format(tables.num_haplotypes))
            LOG.info("# Equivalence Classes: {:,}".format(res["n_ec"]))
            LOG.info("# Unique Reads: {:,}".format(res["n_reads"]))
            bin_utils.save_outputs(tables, tables.target_section(), [sample],
                                   (res["a_indptr"], res["a_indices"], res["a_data"]),
                                   (res["n_indptr"], res["n_indices"], res["n_data"]), False, ec_filename, None,
                                   range_filename, references if track else None, ranges)
            LOG.info("{} created, total time: {}".format(ec_filename, utils.format_time(start_time, time.time())))
            return {k: v for k, v in res.items() if not hasattr(v, "shape")}

        if mode.python:
            cols = emitter.emit_single(iter_records(stream, references, n_header + 1, name), tables)
            if cols.valid_alignments == 0:
                raise RuntimeError("The shape must be a tuple of three positive integers.")   # as convert()
            with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=False,
                           alignments_hint=cols.valid_alignments, device=device, max_read=limit) as builder:
                builder.push(cols.read_group, cols.target_idx, cols.hap_idx, order_base=0)
                return save(builder.finalize(), cols.valid_alignments, None)
        with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=False, alignments_hint=0, device=device,
                       pageable_results=1, max_read=limit) as builder:
            valid, _, ranges, _ = stream_sam_device(stream, name, builder, tables, references, n_header + 1, track,
                                                    max_bytes)
            if valid == 0:
                raise RuntimeError("The shape must be a tuple of three positive integers.")   # as convert()
            return save(builder.finalize(copy=False), valid, ranges)
    finally:
        if not stdin:
            stream.close()
