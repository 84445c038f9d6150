"""Collation by read name on the GPU (ecb_collate_* in include/ecb200.h, _native.Collator, convert(collate=True)).

The rule: for a file F, convert(collate=True) writes what the default convert() writes for F', the valid alignments of
F regrouped - a read is every alignment with one trimmed name, reads in order of their first alignment.  F' is written
here by Python from emitter.emit_collated (or the records themselves) and converted on the default path."""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_records
from alntools_b200 import bam_io, bam_utils, bamcols, emitter, synth

pytestmark = pytest.mark.gpu

N_TARGETS, N_HAPS = 100_000, 2


@pytest.fixture(scope="module", autouse=True)
def _built(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")


def _read(path):
    with open(path, "rb") as fh:
        return fh.read()


def _convert(bam, out_dir, tag, collate=None, targets=None, ranges=False, **kw):
    ec = os.path.join(str(out_dir), tag + ".bin")
    rng = os.path.join(str(out_dir), tag + ".range.txt") if ranges else None
    summary = bam_utils.convert(bam, ec, None, range_filename=rng, target_filename=targets, sample="s",
                                collate=collate, **kw)
    return _read(ec), (_read(rng) if ranges else None), summary


def _split_name(records):
    """Does some trimmed name have two separate runs of valid alignments?"""
    seen, prev = set(), None
    for q, flag, tid, _p, ntid, npos in records:
        if not emitter._valid(flag, tid, ntid, npos):
            continue
        name = emitter._trim(q)
        if name != prev:
            if name in seen:
                return True
            seen.add(name)
            prev = name
    return False


def _regrouped(records):
    """F' as records: the valid ones, each read contiguous, reads in order of their first alignment."""
    reads = {}
    for rec in records:
        if emitter._valid(rec[1], rec[2], rec[4], rec[5]):
            reads.setdefault(emitter._trim(rec[0]), []).append(rec)
    return [r for rs in reads.values() for r in rs]


# ---- goldens ---------------------------------------------------------------------------------------------------
SPLIT = {"toy_single": False, "mixed_single": False, "mixed_single_targets": False, "synth_h2": False,
         "synth_h8_heavy": False, "range_single": False, "range_single_targets": False}


@pytest.mark.parametrize("case", golden_cases("single"), ids=lambda c: c["name"])
def test_goldens(case, tmp_path):
    bam = os.path.join(GOLDEN, case["bam"])
    header, records = load_records(bam)
    assert _split_name(records) == SPLIT[case["name"]]
    targets = os.path.join(GOLDEN, case["targets"]) if case.get("targets") else None
    has_range = bool(case.get("range"))
    # the EC file names the sample after the BAM file: the golden itself, with the default sample
    ec_path, rng_path = str(tmp_path / "c.bin"), (str(tmp_path / "c.range.txt") if has_range else None)
    bam_utils.convert(bam, ec_path, None, range_filename=rng_path, target_filename=targets, collate=True)
    assert not SPLIT[case["name"]]
    assert hashlib.sha256(_read(ec_path)).hexdigest() == case["sha256"]
    if has_range:
        assert _read(rng_path) == _read(os.path.join(GOLDEN, case["range"]))

    # the same records shuffled: some names now have several runs; the result is the default convert() of F'
    rng_gen = np.random.default_rng(len(records))
    shuffled = [records[i] for i in rng_gen.permutation(len(records))]
    assert _split_name(shuffled)
    refs = list(zip(header.references, header.lengths))
    f, fp = str(tmp_path / "f.bam"), str(tmp_path / "fp.bam")
    bam_io.write_bam(f, refs, shuffled, block_payload=3000)
    bam_io.write_bam(fp, refs, _regrouped(shuffled))
    got = _convert(f, tmp_path, "got", collate=True, targets=targets, ranges=True)
    want = _convert(fp, tmp_path, "want", targets=targets, ranges=True)
    assert got[0] == want[0] and got[1] == want[1]
    assert got[2]["n_reads"] == want[2]["n_reads"] and got[2]["n_alignments"] == want[2]["n_alignments"]


# ---- synthetic files: grouped, shuffled, coordinate-like -------------------------------------------------------
def _write_columns(path, rg, tg, hp):
    tids = np.asarray(tg, dtype=np.int64) * N_HAPS + np.asarray(hp, dtype=np.int64)
    bam_io.write_bam_columns(path, synth.reference_names(N_TARGETS, N_HAPS), rg, np.zeros(len(tids), np.uint16), tids)


def _layouts(cols, seed):
    rg, tg, hp = cols["read_group"], cols["target_idx"], cols["hap_idx"]
    perm = np.random.default_rng(seed).permutation(len(rg))
    by_target = np.argsort(tg, kind="stable")
    return {"grouped": (rg, tg, hp), "shuffled": (rg[perm], tg[perm], hp[perm]),
            "by_target": (rg[by_target], tg[by_target], hp[by_target])}


def _regrouped_columns(rg):
    """Order of F' for a file whose read names are the ids rg: alignments of a read together, reads in order of their
    first alignment, file order inside a read (what emitter.emit_collated does, in numpy)."""
    first = np.full(int(rg.max()) + 1, len(rg), dtype=np.int64)
    np.minimum.at(first, rg, np.arange(len(rg)))
    return np.argsort(first[rg], kind="stable")


@pytest.fixture(scope="module")
def synthetic(tmp_path_factory):
    d = tmp_path_factory.mktemp("collate_synth")
    cols = synth.make_columns(1_000_000, N_TARGETS, N_HAPS, 1002, mode="diploid")
    out = {}
    for name, (rg, tg, hp) in _layouts(cols, 3).items():
        path = str(d / (name + ".bam"))
        _write_columns(path, rg, tg, hp)
        out[name] = path
    return d, out


@pytest.mark.parametrize("layout", ["grouped", "shuffled", "by_target"])
def test_synthetic_layouts(layout, synthetic, tmp_path, monkeypatch):
    d, paths = synthetic
    f = paths[layout]
    header, records = emitter.read_bam(f)
    with bamcols.BamColumnReader(f) as r:
        tables = r.build_tables(None)
    cols = emitter.emit_collated(records, tables)
    fp = str(tmp_path / "fp.bam")
    _write_columns(fp, cols.read_group, cols.target_idx, cols.hap_idx)
    got = _convert(f, tmp_path, "got", collate=True, ranges=True)
    want = _convert(fp, tmp_path, "want", ranges=True)
    assert got[0] == want[0] and got[1] == want[1]
    assert got[2]["n_reads"] == want[2]["n_reads"] == cols.n_groups
    with monkeypatch.context() as m:
        m.setenv("ALNTOOLS_B200_EMITTER", "python")
        py = _convert(f, tmp_path, "py", collate=True)
    assert py[0] == got[0]
    if layout == "grouped":
        assert _convert(f, tmp_path, "default", ranges=True)[:2] == got[:2]
    else:
        assert _convert(f, tmp_path, "default")[0] != got[0]    # the default path splits the reads of this file


# ---- the collator on its own -----------------------------------------------------------------------------------
def _key_columns(n_reads, seed, long_read=0):
    """Alignments of n_reads names (keys from a seeded generator) in random order; one name may have long_read
    alignments scattered through the file.  -> (key_lo, key_hi, target_idx, hap_idx, name id of every row)."""
    rng = np.random.default_rng(seed)
    per = rng.integers(1, 6, n_reads)
    if long_read:
        per[n_reads // 2] = long_read
    ids = np.repeat(np.arange(n_reads), per)[rng.permutation(int(per.sum()))]
    lo = rng.integers(0, 1 << 63, n_reads, dtype=np.int64).astype(np.uint64)
    hi = rng.integers(0, 1 << 63, n_reads, dtype=np.int64).astype(np.uint64)
    tg = rng.integers(0, 500, len(ids)).astype(np.int32)
    hp = rng.integers(0, 2, len(ids)).astype(np.int32)
    return lo[ids], hi[ids], tg, hp, ids


def _want(cols):
    """The default build of the regrouped columns."""
    from alntools_b200._native import EcBuilder
    lo, hi, tg, hp, ids = cols
    order = _regrouped_columns(ids)
    rg = ids[order]
    rg = np.concatenate([[0], np.cumsum(rg[1:] != rg[:-1])]).astype(np.int32)
    with EcBuilder(500, 2) as b:
        b.push(rg, np.ascontiguousarray(tg[order]), np.ascontiguousarray(hp[order]))
        return b.finalize()


def _collate(cols, chunk=None, device=False, **options):
    import torch
    from alntools_b200._native import Collator, EcBuilder
    lo, hi, tg, hp, _ = cols
    n = len(tg)
    chunk = chunk or n
    with EcBuilder(500, 2, **options) as b:
        with Collator(b) as c:
            for a in range(0, n, chunk):
                part = [np.ascontiguousarray(x[a:a + chunk]) for x in (lo, hi, tg, hp)]
                if device:
                    part = [torch.from_numpy(p.view(np.int64) if p.dtype == np.uint64 else p).cuda() for p in part]
                c.add(*part)
            reads = c.push()
            stats = c.stats()
        return b.finalize(), reads, stats


def _same_result(a, b):
    for k in ("n_ec", "nnz_a", "n_reads", "n_alignments"):
        assert a[k] == b[k], k
    for k in ("a_indptr", "a_indices", "a_data", "n_indptr", "n_indices", "n_data"):
        assert np.array_equal(a[k], b[k]), k


def test_results_do_not_depend_on_the_shape_of_the_input():
    small = _key_columns(4000, 21)
    want = _want(small)
    results = [_collate(small, chunk=1), _collate(small, chunk=1000), _collate(small),
               _collate(small, device=True), _collate(small, chunk=1000, device=True), _collate(small, collate_slots=1024)]
    for got, reads, stats in results:
        _same_result(got, want)
        assert reads == 4000 == stats["reads"] and stats["alignments"] == len(small[2])
    assert results[-1][2]["table_grows"] > 0 and results[2][2]["table_grows"] == 0


def test_pieces_end_at_read_ends():
    cols = _key_columns(20000, 22, long_read=5000)
    want = _want(cols)
    one, _, st1 = _collate(cols)
    many, reads, st = _collate(cols, collate_piece=4096)
    assert st1["pieces"] == 1 and st["pieces"] > 3
    _same_result(one, want)
    _same_result(many, want)
    assert reads == 20000


# ---- long reads, empty input -----------------------------------------------------------------------------------
REFS = [("T%d_%s" % (t, h), 100 + t) for t in range(6) for h in "AB"]


def _long_read_file(path, k, grouped):
    rng = np.random.default_rng(k)
    recs = [("long", 0, int(rng.integers(0, 12)), int(rng.integers(0, 90))) for _ in range(k)]
    recs += [("r%05d" % i, 0, int(rng.integers(0, 12)), 5) for i in range(3000)]
    if grouped:
        recs = recs[:k] + recs[k:]
    else:
        recs = [recs[i] for i in rng.permutation(len(recs))]
    bam_io.write_bam(path, REFS, recs, block_payload=20000)
    return path


def test_long_reads(tmp_path):
    from alntools_b200._native import EcbError
    f = _long_read_file(str(tmp_path / "ok.bam"), 16384, grouped=False)
    fp = _long_read_file(str(tmp_path / "ok_grouped.bam"), 16384, grouped=True)
    got = _convert(f, tmp_path, "got", collate=True)
    assert got[2]["n_reads"] == 3001
    header, records = load_records(f)
    bam_io.write_bam(fp, list(zip(header.references, header.lengths)), _regrouped(records))
    assert _convert(fp, tmp_path, "want")[0] == got[0]
    for path, collate in ((_long_read_file(str(tmp_path / "long.bam"), 16385, grouped=False), True),
                          (_long_read_file(str(tmp_path / "long_grouped.bam"), 16385, grouped=True), False)):
        with pytest.raises(EcbError) as info:
            _convert(path, tmp_path, "x", collate=collate)
        assert info.value.code == -4 and "16384" in str(info.value)


def test_no_valid_alignment(tmp_path):
    f = str(tmp_path / "none.bam")
    bam_io.write_bam(f, REFS, [("a", 4, 0), ("b", 1 | 0x80, 1), ("a", 4, 2)])
    for collate in (False, True):
        with pytest.raises(RuntimeError, match="three positive integers"):
            _convert(f, tmp_path, "x", collate=collate)


# ---- scale -----------------------------------------------------------------------------------------------------
def test_eight_million_shuffled_reads(tmp_path):
    cols = synth.make_columns(8_000_000, N_TARGETS, N_HAPS, 1002, mode="diploid")   # bench.py's bam_e2e sample
    rg, tg, hp = _layouts(cols, 5)["shuffled"]
    f, fp = str(tmp_path / "f.bam"), str(tmp_path / "fp.bam")
    _write_columns(f, rg, tg, hp)
    order = _regrouped_columns(rg)
    _write_columns(fp, rg[order], tg[order], hp[order])
    got = _convert(f, tmp_path, "got", collate=True)
    want = _convert(fp, tmp_path, "want")
    assert hashlib.sha256(got[0]).hexdigest() == hashlib.sha256(want[0]).hexdigest()
    assert got[2]["n_reads"] == want[2]["n_reads"] == 8_000_000
    assert got[2]["n_alignments"] == want[2]["n_alignments"] == len(rg)
