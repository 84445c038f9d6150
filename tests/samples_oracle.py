"""What convert_samples / ecb_finalize_samples must produce, built from the oracles, for the sample tests.

Files: oracle/ec_oracle.py groups every file on its own (a read never spans two files), merges the files in order (EC
id = rank of the first occurrence over the files in order), builds A from the keys, and N takes each file's counts
as its column.  Columns: oracle/c_oracle.py builds A and the counts of the concatenated columns, and the per-file
counts come from numpy, by matching every read's set of (target, haplotype) elements with an A row."""
import numpy as np

from alntools_b200 import bam_io, emitter
from oracle import c_oracle, ec_oracle


def load(path):
    raw = bam_io.inflate_file(path)
    header = bam_io.parse_header(raw)
    return header, list(bam_io.iter_records(raw, header.records_offset))


def regrouped(records):
    """The valid records of a file, each read (trimmed name) contiguous, reads in order of their first alignment."""
    reads = {}
    for rec in records:
        if emitter._valid(rec[1], rec[2], rec[4], rec[5]):
            reads.setdefault(emitter._trim(rec[0]), []).append(rec)
    return [r for rs in reads.values() for r in rs]


def n_csc(columns):
    """columns: per sample, a dict EC id -> reads, or an array of reads per EC id.  -> (indptr, indices, data) int32,
    ids ascending in a column, zeros not stored."""
    cols = []
    for c in columns:
        if isinstance(c, dict):
            c = sorted(c.items())
            cols.append((np.asarray([e for e, _ in c], np.int64), np.asarray([n for _, n in c], np.int64)))
        else:
            nz = np.flatnonzero(c)
            cols.append((nz, np.asarray(c)[nz]))
    indptr = np.cumsum([0] + [len(e) for e, _ in cols]).astype(np.int32)
    return (indptr, np.concatenate([e for e, _ in cols] + [np.zeros(0, np.int64)]).astype(np.int32),
            np.concatenate([n for _, n in cols] + [np.zeros(0, np.int64)]).astype(np.int32))


def ec_file_bytes(paths, names, target_filename=None, collate=False):
    """The EC file of convert_samples(paths, sample_names=names)."""
    header, results = None, []
    for path in paths:
        h, records = load(path)
        header = header or h
        results.append(ec_oracle.group_chunk_single(regrouped(records) if collate else records))
    tables = ec_oracle.HeaderTables(header.references, header.lengths, target_filename)
    keys = list(ec_oracle.merge_single(results).keys())
    ids = {k: i for i, k in enumerate(keys)}
    a = ec_oracle.a_matrix_from_keys(keys, tables)
    n = n_csc([{ids[k]: v for k, v in r.ec.items()} for r in results])
    return ec_oracle.ecsave2_bytes(tables.haplotypes, list(tables.main_targets.keys()), tables.lengths, names, a, n)


def union_goldens(paths, out_dir):
    """The records of several BAM files rewritten onto one header: the references of every file, in file order, with
    'g<i>' put in front of file i's reference names and read names (so no two files share a target or a read name).
    -> the new paths."""
    refs, offsets, files = [], [], []
    for i, path in enumerate(paths):
        header, records = load(path)
        offsets.append(len(refs))
        refs += [("g%d%s" % (i, n), length) for n, length in zip(header.references, header.lengths)]
        files.append(records)
    out = []
    for i, records in enumerate(files):
        moved = [("g%d%s" % (i, q), flag, tid + offsets[i] if tid >= 0 else tid, pos,
                  ntid + offsets[i] if ntid >= 0 else ntid, npos) for q, flag, tid, pos, ntid, npos in records]
        p = "%s/u%d.bam" % (out_dir, i)
        bam_io.write_bam(p, refs, moved, block_payload=5000)
        out.append(p)
    return out


# ---- columns ---------------------------------------------------------------------------------------------------
def _mix(x):
    """splitmix64 of uint64 codes (a set's hash is the sum of its distinct elements' mixes)."""
    with np.errstate(over="ignore"):
        z = x.astype(np.uint64) + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def _sum_by(groups, values):
    """Sum (mod 2^64) of values per group; groups ascending and dense from 0."""
    if len(groups) == 0:
        return np.zeros(0, np.uint64)
    starts = np.flatnonzero(np.r_[True, groups[1:] != groups[:-1]])
    return np.add.reduceat(values, starts)


def _read_hashes(cols):
    rg, tg, hp = (np.asarray(cols[k], dtype=np.int64) for k in ("read_group", "target_idx", "hap_idx"))
    read = np.cumsum(np.r_[0, rg[1:] != rg[:-1]]) if len(rg) else rg
    key = np.unique((read << 32) | (tg << 5) | hp)
    return _sum_by(key >> 32, _mix(key & 0xFFFFFFFF))


def columns_result(samples):
    """samples: per sample, a list of column dicts (read_group, target_idx, hap_idx), one per push.  -> (a_indptr,
    a_indices, a_data, n_indptr, n_indices, n_data, n_reads) of ecb_finalize_samples."""
    pushes = [p for s in samples for p in s if len(p["read_group"])]
    rg = np.concatenate([np.asarray(p["read_group"], np.int64) + (i << 32) for i, p in enumerate(pushes)])
    read = np.cumsum(np.r_[0, rg[1:] != rg[:-1]]).astype(np.int32)     # reads never merge across pushes
    tg = np.concatenate([p["target_idx"] for p in pushes]).astype(np.int32)
    hp = np.concatenate([p["hap_idx"] for p in pushes]).astype(np.int32)
    indptr, indices, data, _counts, n_reads = c_oracle.ec_from_columns(read, tg, hp)
    # A rows -> hashes of their element sets
    rows = np.repeat(np.arange(len(indptr) - 1, dtype=np.int64), np.diff(indptr))
    parts = []
    for h in range(31):
        sel = ((np.asarray(data, np.int64) >> h) & 1).astype(bool)
        parts.append((rows[sel] << 32) | (np.asarray(indices, np.int64)[sel] << 5) | h)
    key = np.sort(np.concatenate(parts))
    row_hash = _sum_by(key >> 32, _mix(key & 0xFFFFFFFF))
    order = np.argsort(row_hash)
    assert len(np.unique(row_hash)) == len(row_hash)
    columns = []
    for sample in samples:
        counts = np.zeros(len(indptr) - 1, np.int64)
        for p in sample:
            if not len(p["read_group"]):
                continue
            h = _read_hashes(p)
            ids = order[np.searchsorted(row_hash, h, sorter=order)]
            assert np.array_equal(row_hash[ids], h)
            counts += np.bincount(ids, minlength=len(counts))
        columns.append(counts)
    return (indptr, indices, data) + n_csc(columns) + (n_reads,)
