"""Render BAM alignments as SAM text: the S of the SAM rule for a BAM file B (alntools_b200/sam_utils.py).  SEQ and
QUAL are '*' or synthetic read_len-base strings, so that lines are long; names holding a tab or a newline cannot be
rendered and are refused."""
import numpy as np

from alntools_b200 import bam_io


def sam_text(references, lengths, records, read_len=0, header_extra=True, seed=0):
    """references / lengths: the @SQ list; records: (qname, flag, tid, pos, next_tid, next_pos) tuples."""
    rng = np.random.default_rng(seed)
    out = [b"@HD\tVN:1.6\tSO:queryname\n"] if header_extra else []
    out += [b"@SQ\tSN:%s\tLN:%d\n" % (name.encode(), length) for name, length in zip(references, lengths)]
    if header_extra:
        out.append(b"@PG\tID:render\tPN:sam_render\n")
    refs = [r.encode() for r in references]
    for qname, flag, tid, pos, ntid, npos in records:
        if "\t" in qname or "\n" in qname:
            raise ValueError("read name %r holds a tab or a newline: no SAM line can hold it" % qname)
        if pos < -1 or npos < -1:
            raise ValueError("pos %d / next_pos %d below -1: no SAM line can hold it" % (pos, npos))
        rname = refs[tid] if tid >= 0 else b"*"
        rnext = b"*" if ntid < 0 else b"=" if ntid == tid else refs[ntid]
        if read_len:
            seq = bytes(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, read_len)])
            qual = bytes(rng.integers(35, 74, read_len, dtype=np.uint8))
            cigar = b"%dM" % read_len
        else:
            seq = qual = cigar = b"*"
        out.append(b"\t".join([qname.encode(), b"%d" % flag, rname, b"%d" % (pos + 1), b"255", cigar, rnext,
                               b"%d" % (npos + 1), b"0", seq, qual]) + b"\n")
    return b"".join(out)


def bam_to_sam(bam_path, sam_path, read_len=0):
    raw = bam_io.inflate_file(bam_path)
    header = bam_io.parse_header(raw)
    with open(sam_path, "wb") as fh:
        fh.write(sam_text(header.references, header.lengths, bam_io.iter_records(raw, header.records_offset), read_len))
    return header
