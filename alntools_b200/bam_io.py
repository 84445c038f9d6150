"""Host-side BGZF/BAM container I/O (SAM spec sections 4.1/4.2).

The reference leaves BAM decode to pysam/htslib (bam_utils.py:253-304); neither is installed in
this image, so the host side carries its own small reader. Only the fixed-offset fields the
EC-construction path looks at are decoded: refID, pos, l_read_name, flag, next_refID, next_pos and
the read name. A writer is included so that tests and benchmarks can mint synthetic name-grouped
BAM files.
"""
import struct
import zlib

import numpy as np

BGZF_EOF = (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00"
            b"\x1b\x00\x03\x00\x00\x00\x00\x00\x00\x00\x00\x00")
_BGZF_HEAD = b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00"
_CORE = struct.Struct("<iiBBHHHiiii")


def bgzf_block(payload, level=6):
    comp = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = comp.compress(payload) + comp.flush()
    return (_BGZF_HEAD + struct.pack("<H", len(body) + 25) + body
            + struct.pack("<II", zlib.crc32(payload) & 0xFFFFFFFF, len(payload)))


def bam_header_bytes(references):
    """references: iterable of (name, length)."""
    text = b"@HD\tVN:1.0\tSO:queryname\n" + b"".join(
        b"@SQ\tSN:%s\tLN:%d\n" % (n.encode(), l) for n, l in references)
    out = [b"BAM\x01", struct.pack("<i", len(text)), text, struct.pack("<i", len(references))]
    for n, l in references:
        nb = n.encode() + b"\x00"
        out.append(struct.pack("<i", len(nb)) + nb + struct.pack("<i", l))
    return b"".join(out)


def bam_record_bytes(qname, flag, tid, pos=0, next_tid=-1, next_pos=-1):
    qn = qname.encode() + b"\x00"
    core = _CORE.pack(tid, pos, len(qn), 255, 4680, 0, flag, 0, next_tid, next_pos, 0) + qn
    return struct.pack("<i", len(core)) + core


def _write_blocks(fh, payload, block_payload, level):
    """BGZF blocks hold at most 64 KiB: split long payloads (e.g. a 200k-reference header)."""
    for off in range(0, len(payload), block_payload):
        fh.write(bgzf_block(payload[off:off + block_payload], level))


def write_bam(filename, references, alignments, block_payload=60000, level=6):
    """Write a BAM file.

    references: [(name, length)]; alignments: iterable of tuples
    (qname, flag, tid[, pos[, next_tid[, next_pos]]]) with no sequence/cigar.
    The header is placed in its own BGZF block so alignments start on a block boundary.
    """
    with open(filename, "wb") as fh:
        _write_blocks(fh, bam_header_bytes(references), min(block_payload, 60000), level)
        buf = []
        size = 0
        for aln in alignments:
            rec = bam_record_bytes(*aln)
            buf.append(rec)
            size += len(rec)
            if size >= block_payload:
                fh.write(bgzf_block(b"".join(buf), level))
                buf, size = [], 0
        if buf:
            fh.write(bgzf_block(b"".join(buf), level))
        fh.write(BGZF_EOF)


_CID_FIELDS = b"|||CR|||x|||CY|||x|||UR|||x|||UY|||x|||BC|||x|||QT|||x|||CID|||cell"
_CID_DIGITS = 7


def write_bam_columns(filename, references, qname_ids, flags, tids, name_fmt="read%09d",
                      block_payload=60000, level=1, cell_ids=None):
    """Vectorised writer for large synthetic BAMs: record i is (name_fmt % qname_ids[i], flags[i],
    tids[i]); all names must have the same byte length.  cell_ids: per-record cell ids (< 10^7) put in field 14
    of a 10x-style '|||'-separated name as 'cell%07d' (what the per-cell path reads)."""
    n = len(tids)
    tail = 0 if cell_ids is None else len(_CID_FIELDS) + _CID_DIGITS
    name_len = len(name_fmt % 0) + tail + 1
    rec_len = 4 + 32 + name_len
    raw = np.zeros((n, rec_len), dtype=np.uint8)
    raw[:, 0:4] = np.frombuffer(struct.pack("<i", 32 + name_len), dtype=np.uint8)
    core = np.zeros(n, dtype=np.dtype([("tid", "<i4"), ("pos", "<i4"), ("l_name", "u1"), ("mapq", "u1"),
                                       ("bin", "<u2"), ("ncig", "<u2"), ("flag", "<u2"), ("lseq", "<i4"),
                                       ("ntid", "<i4"), ("npos", "<i4"), ("tlen", "<i4")]))
    core["tid"] = tids
    core["pos"] = 10
    core["l_name"] = name_len
    core["mapq"] = 255
    core["bin"] = 4680
    core["flag"] = flags
    core["ntid"] = -1
    core["npos"] = -1
    raw[:, 4:36] = core.view(np.uint8).reshape(n, 32)
    ids = np.asarray(qname_ids, dtype=np.int64)
    prefix = name_fmt.split("%")[0].encode()
    ndig = name_len - 1 - tail - len(prefix)
    raw[:, 36:36 + len(prefix)] = np.frombuffer(prefix, dtype=np.uint8)
    rem = ids.copy()
    for d in range(ndig - 1, -1, -1):
        raw[:, 36 + len(prefix) + d] = (rem % 10 + 48).astype(np.uint8)
        rem //= 10
    if cell_ids is not None:
        at = 36 + len(prefix) + ndig
        raw[:, at:at + len(_CID_FIELDS)] = np.frombuffer(_CID_FIELDS, dtype=np.uint8)
        rem = np.asarray(cell_ids, dtype=np.int64).copy()
        for d in range(_CID_DIGITS - 1, -1, -1):
            raw[:, at + len(_CID_FIELDS) + d] = (rem % 10 + 48).astype(np.uint8)
            rem //= 10
    flat = raw.reshape(-1)
    per_block = max(1, block_payload // rec_len) * rec_len
    with open(filename, "wb") as fh:
        _write_blocks(fh, bam_header_bytes(references), 60000, level)
        for off in range(0, flat.size, per_block):
            fh.write(bgzf_block(flat[off:off + per_block].tobytes(), level))
        fh.write(BGZF_EOF)


def iter_bgzf_blocks(fh):
    """Yield (file_offset, block_size, payload_size) for every BGZF block without inflating
    (same information as reference bam_utils.py:1320-1367)."""
    offset = 0
    while True:
        head = fh.read(18)
        if len(head) < 18:
            return
        if head[:4] != b"\x1f\x8b\x08\x04":
            raise ValueError("not a BGZF block at offset %d" % offset)
        xlen = struct.unpack_from("<H", head, 10)[0]
        if xlen == 6 and head[12:14] == b"BC":
            bsize = struct.unpack_from("<H", head, 16)[0] + 1
            fh.seek(offset + bsize - 4)
        else:  # generic extra-field walk
            fh.seek(offset + 12)
            extra = fh.read(xlen)
            bsize, p = None, 0
            while p < xlen:
                slen = struct.unpack_from("<H", extra, p + 2)[0]
                if extra[p:p + 2] == b"BC":
                    bsize = struct.unpack_from("<H", extra, p + 4)[0] + 1
                p += 4 + slen
            if bsize is None:
                raise ValueError("BGZF block without BC field")
            fh.seek(offset + bsize - 4)
        isize = struct.unpack("<I", fh.read(4))[0]
        yield offset, bsize, isize
        offset += bsize


def inflate_file(filename):
    """Inflate every BGZF block of `filename`; returns one bytes object."""
    parts = []
    with open(filename, "rb") as fh:
        data = fh.read()
    off, n = 0, len(data)
    while off + 18 <= n:
        if data[off:off + 4] != b"\x1f\x8b\x08\x04":
            raise ValueError("not a BGZF block at offset %d" % off)
        xlen = struct.unpack_from("<H", data, off + 10)[0]
        p, bsize = off + 12, None
        while p < off + 12 + xlen:
            slen = struct.unpack_from("<H", data, p + 2)[0]
            if data[p:p + 2] == b"BC":
                bsize = struct.unpack_from("<H", data, p + 4)[0] + 1
            p += 4 + slen
        if bsize is None:
            raise ValueError("BGZF block without BC field")
        parts.append(zlib.decompress(data[off + 12 + xlen:off + bsize - 8], -15))
        off += bsize
    return b"".join(parts)


class BamHeader(object):
    __slots__ = ("references", "lengths", "records_offset")

    def __init__(self, references, lengths, records_offset):
        self.references = references
        self.lengths = lengths
        self.records_offset = records_offset

    def get_tid(self, name):
        try:
            return self.references.index(name)
        except ValueError:
            return -1


def parse_header(raw):
    """raw: inflated BAM bytes. Returns BamHeader (references in header order = tid order)."""
    if raw[:4] != b"BAM\x01":
        raise ValueError("not a BAM stream")
    l_text = struct.unpack_from("<i", raw, 4)[0]
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", raw, p)[0]
    p += 4
    names, lengths = [], []
    for _ in range(n_ref):
        l_name = struct.unpack_from("<i", raw, p)[0]
        names.append(raw[p + 4:p + 4 + l_name - 1].decode())
        lengths.append(struct.unpack_from("<i", raw, p + 4 + l_name)[0])
        p += 8 + l_name
    return BamHeader(tuple(names), tuple(lengths), p)


def read_header(filename):
    """Parse only as many leading BGZF blocks as the header needs."""
    raw = b""
    with open(filename, "rb") as fh:
        if fh.read(4) != b"\x1f\x8b\x08\x04":
            raise ValueError("File {} is not a BAM file".format(filename))
        fh.seek(0)
        blocks = iter_bgzf_blocks(fh)
        with open(filename, "rb") as fh2:
            for off, bsize, _ in blocks:
                fh2.seek(off)
                blk = fh2.read(bsize)
                xlen = struct.unpack_from("<H", blk, 10)[0]
                raw += zlib.decompress(blk[12 + xlen:-8], -15)
                try:
                    return parse_header(raw)
                except (struct.error, IndexError):
                    continue
    raise ValueError("truncated BAM header in {}".format(filename))


def iter_records(raw, offset):
    """Yield (qname:str, flag, tid, pos, next_tid, next_pos) from inflated BAM bytes."""
    n = len(raw)
    unpack = _CORE.unpack_from
    while offset + 4 <= n:
        bs = struct.unpack_from("<i", raw, offset)[0]
        tid, pos, l_name, _mq, _bin, _nc, flag, _ls, ntid, npos, _tl = unpack(raw, offset + 4)
        yield raw[offset + 36:offset + 36 + l_name - 1].decode(), flag, tid, pos, ntid, npos
        offset += 4 + bs


def read_virtual(filename, virtual_offset, nbytes):
    """`nbytes` inflated bytes starting at a BGZF virtual offset (compressed block start << 16 | offset inside
    the inflated block), continuing over as many blocks as it takes - what the reference does with
    Bio.bgzf.BgzfReader.seek() + read() when it cuts a chunk (bam_utils.py:173-179, 185-191)."""
    out, need = [], int(nbytes)
    block, within = int(virtual_offset) >> 16, int(virtual_offset) & 0xFFFF
    with open(filename, "rb") as fh:
        while need > 0:
            fh.seek(block)
            head = fh.read(18)
            if len(head) < 18 or head[:4] != b"\x1f\x8b\x08\x04":
                break
            xlen = struct.unpack_from("<H", head, 10)[0]
            fh.seek(block + 12)
            extra = fh.read(xlen)
            bsize, p = None, 0
            while p < xlen:
                slen = struct.unpack_from("<H", extra, p + 2)[0]
                if extra[p:p + 2] == b"BC":
                    bsize = struct.unpack_from("<H", extra, p + 4)[0] + 1
                p += 4 + slen
            if bsize is None:
                raise ValueError("BGZF block without BC field")
            data = zlib.decompress(fh.read(bsize - 12 - xlen - 8), -15)
            take = data[within:within + need]
            out.append(take)
            need -= len(take)
            block += bsize
            within = 0
    return b"".join(out)
