"""Seeded synthetic workloads for the bam2ec path (SURVEY.md section 8d).

Columns are what the host emitter hands to the device: per valid alignment an int32 read-group id
(non-decreasing), main-target index and haplotype index, optionally a cell index.  Transcript
popularity is Zipf(1.3) mod T; a read hits k transcripts, each on a uniformly random non-empty
subset of the H haplotypes.
"""
import numpy as np


def _reads_per_k(rng, n_reads, mode):
    """Number of transcripts per read."""
    if isinstance(mode, int):                       # fixed multimapping degree
        return np.full(n_reads, mode, dtype=np.int64)
    if mode == "light":                              # P(k>1) = 1/8, k in 2..4 then
        multi = rng.integers(0, 8, n_reads) == 0
        return np.where(multi, rng.integers(2, 5, n_reads), 1).astype(np.int64)
    if mode == "diploid":                            # cfg2: about 1.5 transcripts per read
        k = rng.geometric(0.65, n_reads)
        return np.minimum(k, 16).astype(np.int64)
    if mode == "heavy":                              # cfg3: geometric, mean about 8 transcripts, cap 256
        k = rng.geometric(0.12, n_reads)
        return np.minimum(k, 256).astype(np.int64)
    raise ValueError(mode)


def make_columns_fixed_degree(n_reads, n_targets, n_haps, seed, degree):
    """The multimapping-degree sweep (BASELINE.json configs[4]): every read has exactly `degree` alignments,
    each on a Zipf(1.3) transcript and a uniformly random haplotype (duplicates inside a read are possible
    and collapse, as in the reference)."""
    rng = np.random.default_rng(seed)
    n = int(n_reads) * int(degree)
    return {
        "read_group": np.repeat(np.arange(n_reads, dtype=np.int32), degree),
        "target_idx": (rng.zipf(1.3, n) % n_targets).astype(np.int32),
        "hap_idx": rng.integers(0, n_haps, n, dtype=np.int32),
        "n_reads": int(n_reads),
    }


def make_columns(n_reads, n_targets, n_haps, seed, mode="light", n_cells=0, dup_rate=0.0):
    """Return dict(read_group, target_idx, hap_idx[, cell_idx]) int32 arrays plus n_reads.

    dup_rate: fraction of alignments duplicated verbatim inside their read (same transcript hit at a
    second position), which the reference collapses (bam_utils.py:322-325).
    """
    if isinstance(mode, str) and mode.startswith("aln"):           # "aln<k>": exactly k alignments per read
        return make_columns_fixed_degree(n_reads, n_targets, n_haps, seed, int(mode[3:]))
    rng = np.random.default_rng(seed)
    k = _reads_per_k(rng, n_reads, mode)
    n_hits = int(k.sum())
    hit_read = np.repeat(np.arange(n_reads, dtype=np.int64), k)
    hit_target = (rng.zipf(1.3, n_hits) % n_targets).astype(np.int64)
    mask = rng.integers(1, 1 << n_haps, n_hits, dtype=np.int64)
    nbits = np.zeros(n_hits, dtype=np.int64)
    for h in range(n_haps):
        nbits += (mask >> h) & 1
    aln_hit = np.repeat(np.arange(n_hits, dtype=np.int64), nbits)
    # haplotype of each alignment: the j-th set bit of its hit's mask
    first = np.cumsum(nbits) - nbits
    j = np.arange(len(aln_hit), dtype=np.int64) - first[aln_hit]
    hap = np.zeros(len(aln_hit), dtype=np.int64)
    m = mask[aln_hit]
    seen = np.zeros(len(aln_hit), dtype=np.int64)
    for h in range(n_haps):
        bit = (m >> h) & 1
        sel = (bit == 1) & (seen == j)
        hap[sel] = h
        seen += bit
    rg = hit_read[aln_hit]
    tg = hit_target[aln_hit]
    if dup_rate > 0:
        dup = rng.random(len(rg)) < dup_rate
        reps = np.where(dup, 2, 1)
        rg, tg, hap = np.repeat(rg, reps), np.repeat(tg, reps), np.repeat(hap, reps)
    out = {
        "read_group": rg.astype(np.int32),
        "target_idx": tg.astype(np.int32),
        "hap_idx": hap.astype(np.int32),
        "n_reads": int(n_reads),
    }
    if n_cells:
        read_cell = (rng.zipf(1.2, n_reads) % n_cells).astype(np.int32)
        out["cell_idx"] = read_cell[rg]
    return out


def reference_names(n_targets, n_haps, hap_letters="ABCDEFGH"):
    """@SQ names 'ENSMUST%011d_<hap>' with tid = target * H + hap, lengths 1000 + target."""
    return [("ENSMUST%011d_%s" % (t, hap_letters[h]), 1000 + t)
            for t in range(n_targets) for h in range(n_haps)]


def columns_to_bam_cells(filename, cols, n_targets, n_haps, level=1):
    """Materialise per-cell columns as one name-grouped BAM file of the per-cell path: the cell of every read is
    field 14 of its '|||'-separated name ('cell%07d' % cell_idx)."""
    from . import bam_io
    tids = cols["target_idx"].astype(np.int64) * n_haps + cols["hap_idx"]
    bam_io.write_bam_columns(filename, reference_names(n_targets, n_haps), cols["read_group"],
                             np.zeros(len(tids), dtype=np.uint16), tids, level=level, cell_ids=cols["cell_idx"])


def columns_to_bam(filename, cols, n_targets, n_haps, level=1):
    """Materialise single-sample columns as a name-grouped BAM (read names 'read%09d')."""
    from . import bam_io
    tids = cols["target_idx"].astype(np.int64) * n_haps + cols["hap_idx"]
    bam_io.write_bam_columns(filename, reference_names(n_targets, n_haps), cols["read_group"],
                             np.zeros(len(tids), dtype=np.uint16), tids, level=level)


def columns_to_bam_seq(filename, cols, n_targets, n_haps, read_len=100, level=1, seed=0):
    """columns_to_bam with the record shape of a real aligner's output: every record carries a CIGAR of one
    read_len-M operation, the packed sequence and the base qualities (seeded random bases and qualities)."""
    from . import bam_io
    import struct
    tids = cols["target_idx"].astype(np.int64) * n_haps + cols["hap_idx"]
    ids = np.asarray(cols["read_group"], dtype=np.int64)
    n = len(tids)
    name_len = len("read%09d" % 0) + 1
    seq_len = (read_len + 1) // 2
    body = 32 + name_len + 4 + seq_len + read_len
    rec_len = 4 + body
    raw = np.zeros((n, rec_len), dtype=np.uint8)
    raw[:, 0:4] = np.frombuffer(struct.pack("<i", body), dtype=np.uint8)
    core = np.zeros(n, dtype=np.dtype([("tid", "<i4"), ("pos", "<i4"), ("l_name", "u1"), ("mapq", "u1"),
                                       ("bin", "<u2"), ("ncig", "<u2"), ("flag", "<u2"), ("lseq", "<i4"),
                                       ("ntid", "<i4"), ("npos", "<i4"), ("tlen", "<i4")]))
    core["tid"] = tids
    core["pos"] = 10
    core["l_name"] = name_len
    core["mapq"] = 255
    core["bin"] = 4680
    core["ncig"] = 1
    core["lseq"] = read_len
    core["ntid"] = -1
    core["npos"] = -1
    raw[:, 4:36] = core.view(np.uint8).reshape(n, 32)
    raw[:, 36:40] = np.frombuffer(b"read", dtype=np.uint8)
    rem = ids.copy()
    for d in range(8, -1, -1):
        raw[:, 40 + d] = (rem % 10 + 48).astype(np.uint8)
        rem //= 10
    at = 36 + name_len
    raw[:, at:at + 4] = np.frombuffer(struct.pack("<I", read_len << 4), dtype=np.uint8)
    rng = np.random.default_rng(seed)
    bases = np.array([1, 2, 4, 8], dtype=np.uint8)                 # A C G T in BAM's 4-bit code
    seq = bases[rng.integers(0, 4, (n, 2 * seq_len))]
    raw[:, at + 4:at + 4 + seq_len] = (seq[:, 0::2] << 4) | seq[:, 1::2]
    raw[:, at + 4 + seq_len:] = rng.integers(2, 41, (n, read_len), dtype=np.uint8)
    flat = raw.reshape(-1)
    per_block = max(1, 60000 // rec_len) * rec_len
    with open(filename, "wb") as fh:
        header = bam_io.bam_header_bytes(reference_names(n_targets, n_haps))
        for off in range(0, len(header), 60000):
            fh.write(bam_io.bgzf_block(header[off:off + 60000], level))
        for off in range(0, flat.size, per_block):
            fh.write(bam_io.bgzf_block(flat[off:off + per_block].tobytes(), level))
        fh.write(bam_io.BGZF_EOF)


def columns_to_sam(filename, cols, n_targets, n_haps, read_len=0, seed=0, chunk=1 << 20):
    """The alignments of columns_to_bam (read_len=0: CIGAR, SEQ and QUAL '*') or columns_to_bam_seq (read_len > 0: a
    CIGAR of one read_len-M operation and seeded random bases and qualities) as SAM text, with the same @SQ list, names
    ('read%09d'), flags (0), POS (11) and mates ('*', 0); written in fixed-width rows with numpy."""
    tids = cols["target_idx"].astype(np.int64) * n_haps + cols["hap_idx"]
    ids = np.asarray(cols["read_group"], dtype=np.int64)
    refs = reference_names(n_targets, n_haps)
    if read_len == 0:
        tail = b"*\t*\t0\t0\t*\t*\n"
    else:
        tail = b"%dM\t*\t0\t0\t" % read_len
    head = b"read000000000\t0\tENSMUST00000000000_A\t11\t255\t"
    width = len(head) + len(tail) + (2 * read_len + 2 if read_len else 0)
    rng = np.random.default_rng(seed)
    letters = np.frombuffer(b"ABCDEFGH", dtype=np.uint8)
    bases = np.frombuffer(b"ACGT", dtype=np.uint8)
    with open(filename, "wb") as fh:
        fh.write(b"@HD\tVN:1.0\tSO:queryname\n")
        fh.write(b"".join(b"@SQ\tSN:%s\tLN:%d\n" % (name.encode(), length) for name, length in refs))
        for lo in range(0, len(tids), chunk):
            t, r = tids[lo:lo + chunk], ids[lo:lo + chunk].copy()
            n = len(t)
            rows = np.empty((n, width), dtype=np.uint8)
            rows[:, :len(head)] = np.frombuffer(head, dtype=np.uint8)
            rows[:, len(head):len(head) + len(tail)] = np.frombuffer(tail, dtype=np.uint8)
            for d in range(8, -1, -1):                       # read%09d
                rows[:, 4 + d] = (r % 10 + 48).astype(np.uint8)
                r //= 10
            target, hap = t // n_haps, t % n_haps
            for d in range(10, -1, -1):                      # ENSMUST%011d_<hap>
                rows[:, 23 + d] = (target % 10 + 48).astype(np.uint8)
                target //= 10
            rows[:, 35] = letters[hap]
            if read_len:
                at = len(head) + len(tail)
                rows[:, at:at + read_len] = bases[rng.integers(0, 4, (n, read_len))]
                rows[:, at + read_len] = ord("\t")
                rows[:, at + read_len + 1:at + 2 * read_len + 1] = rng.integers(35, 74, (n, read_len), dtype=np.uint8)
                rows[:, -1] = ord("\n")
            fh.write(rows.tobytes())
