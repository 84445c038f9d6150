"""Collation within a device memory budget (ECB_OPT_COLLATE_BUDGET, ALNTOOLS_B200_COLLATE_BUDGET).

A collator whose rows would pass its budget spills them to host memory, partitioned by name key, and collates in passes
(DESIGN.md section 6.2).  The rule does not change: for every budget, convert(collate=True) writes the bytes of the
unbudgeted collation, which are those of the default convert() of F' (the valid alignments regrouped by read, reads in
order of their first alignment).  Every case reads the collator's stats to make sure the intended path ran."""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_records
from alntools_b200 import bam_io, bam_utils, emitter, synth

N_TARGETS, N_HAPS = 100_000, 2
ENV = "ALNTOOLS_B200_COLLATE_BUDGET"
LIMIT = -4


@pytest.fixture
def gpu(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")


@pytest.fixture
def collator_stats(monkeypatch):
    """The collator stats of every emitter.stream_collated call that convert() makes."""
    seen = []
    real = emitter.stream_collated

    def spy(*args, **kwargs):
        out = real(*args, **kwargs)
        seen.append(out[2])
        return out

    monkeypatch.setattr(emitter, "stream_collated", spy)
    return seen


def _read(path):
    with open(path, "rb") as fh:
        return fh.read()


def _convert(bam, out_dir, tag, monkeypatch, budget=None, collate=True, targets=None, ranges=False):
    """convert() with ALNTOOLS_B200_COLLATE_BUDGET = budget (None: unset) -> (EC bytes, range bytes, summary)."""
    ec = os.path.join(str(out_dir), tag + ".bin")
    rng = os.path.join(str(out_dir), tag + ".range.txt") if ranges else None
    with monkeypatch.context() as m:
        if budget is None:
            m.delenv(ENV, raising=False)
        else:
            m.setenv(ENV, str(budget))
        summary = bam_utils.convert(bam, ec, None, range_filename=rng, target_filename=targets, sample="s",
                                    collate=collate)
    return _read(ec), (_read(rng) if ranges else None), summary


def _regrouped(records):
    reads = {}
    for rec in records:
        if emitter._valid(rec[1], rec[2], rec[4], rec[5]):
            reads.setdefault(emitter._trim(rec[0]), []).append(rec)
    return [r for rs in reads.values() for r in rs]


# ---- goldens at every budget from too small to no spill -----------------------------------------------------------
def _budget_scan(bam, tmp_path, monkeypatch, stats, targets, has_range):
    """convert(collate=True) at budgets from 20 kB up by 12 % a step until the collation no longer spills, each
    against the unbudgeted bytes.  -> [(budget, stats)] of the runs that did not hit ECB_ERR_LIMIT."""
    from alntools_b200._native import EcbError
    want = _convert(bam, tmp_path, "want", monkeypatch, targets=targets, ranges=has_range)
    assert stats[-1]["spills"] == 0 and stats[-1]["groups"] == 0
    runs, budget = [], 20_000
    while True:
        try:
            got = _convert(bam, tmp_path, "got", monkeypatch, budget=budget, targets=targets, ranges=has_range)
        except EcbError as err:
            assert err.code == LIMIT and str(budget) in str(err), str(err)
            assert not runs, "a larger budget failed after a smaller one passed (%d)" % budget
        else:
            assert got[0] == want[0] and got[1] == want[1], budget
            assert got[2]["n_reads"] == want[2]["n_reads"] and got[2]["n_alignments"] == want[2]["n_alignments"]
            st = stats[-1]
            runs.append((budget, st))
            if st["spills"] == 0:
                break
            assert st["groups"] >= 1 and st["host_bytes"] >= 28 * st["alignments"]
            assert st["device_bytes"] <= budget + 12 * 16384 * 4, (budget, st["device_bytes"])
        budget = int(budget * 1.12)
    return runs


@pytest.mark.gpu
@pytest.mark.parametrize("case", golden_cases("single"), ids=lambda c: c["name"])
@pytest.mark.parametrize("layout", ["as_is", "shuffled"])
def test_goldens_at_every_budget(gpu, case, layout, tmp_path, monkeypatch, collator_stats):
    bam = os.path.join(GOLDEN, case["bam"])
    targets = os.path.join(GOLDEN, case["targets"]) if case.get("targets") else None
    has_range = bool(case.get("range"))
    header, records = load_records(bam)
    if layout == "shuffled":
        records = [records[i] for i in np.random.default_rng(len(records)).permutation(len(records))]
        bam = str(tmp_path / "f.bam")
        bam_io.write_bam(bam, list(zip(header.references, header.lengths)), records, block_payload=3000)
        # the unbudgeted collation is the default convert() of F'
        fp = str(tmp_path / "fp.bam")
        bam_io.write_bam(fp, list(zip(header.references, header.lengths)), _regrouped(records))
        assert (_convert(fp, tmp_path, "fp", monkeypatch, collate=False, targets=targets, ranges=has_range)[:2] ==
                _convert(bam, tmp_path, "c", monkeypatch, targets=targets, ranges=has_range)[:2])
    runs = _budget_scan(bam, tmp_path, monkeypatch, collator_stats, targets, has_range)
    n = runs[-1][1]["alignments"]
    spilled = [st for _, st in runs if st["spills"] > 0]
    assert runs[-1][1]["spills"] == 0                                  # no spill
    assert any(st["spills"] == 1 and st["groups"] == 1 for st in spilled)   # one spill (at push), one group
    if n >= 100:
        assert any(st["spills"] >= 2 for st in spilled)                # spills in the middle of the one add
    if n >= 10_000:
        assert any(st["groups"] == 2 for st in spilled)
        assert any(st["groups"] >= 8 and st["spills"] >= 8 for st in spilled)


# ---- at scale: 1 M cfg2-shaped reads in three layouts --------------------------------------------------------------
def _write_columns(path, rg, tg, hp):
    tids = np.asarray(tg, dtype=np.int64) * N_HAPS + np.asarray(hp, dtype=np.int64)
    bam_io.write_bam_columns(path, synth.reference_names(N_TARGETS, N_HAPS), rg, np.zeros(len(tids), np.uint16), tids)


def _regrouped_columns(rg):
    first = np.full(int(rg.max()) + 1, len(rg), dtype=np.int64)
    np.minimum.at(first, rg, np.arange(len(rg)))
    return np.argsort(first[rg], kind="stable")


def _layouts(cols, seed):
    rg, tg, hp = cols["read_group"], cols["target_idx"], cols["hap_idx"]
    perm = np.random.default_rng(seed).permutation(len(rg))
    by_target = np.argsort(tg, kind="stable")
    return {"grouped": (rg, tg, hp), "shuffled": (rg[perm], tg[perm], hp[perm]),
            "by_target": (rg[by_target], tg[by_target], hp[by_target])}


@pytest.fixture(scope="module")
def synthetic(tmp_path_factory):
    d = tmp_path_factory.mktemp("spill_synth")
    cols = synth.make_columns(1_000_000, N_TARGETS, N_HAPS, 1002, mode="diploid")
    out = {}
    for name, (rg, tg, hp) in _layouts(cols, 3).items():
        f, fp = str(d / (name + ".bam")), str(d / (name + "_regrouped.bam"))
        _write_columns(f, rg, tg, hp)
        order = _regrouped_columns(rg)
        _write_columns(fp, rg[order], tg[order], hp[order])
        out[name] = (f, fp)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("budget", [24_000_000, 64_000_000])
@pytest.mark.parametrize("layout", ["grouped", "shuffled", "by_target"])
def test_synthetic_layouts_within_budget(gpu, layout, budget, synthetic, tmp_path, monkeypatch, collator_stats):
    f, fp = synthetic[layout]
    want = _convert(fp, tmp_path, "want", monkeypatch, collate=False, ranges=True)
    got = _convert(f, tmp_path, "got", monkeypatch, budget=budget, ranges=True)
    assert got[0] == want[0] and got[1] == want[1]
    assert got[2]["n_reads"] == want[2]["n_reads"] == 1_000_000
    st = collator_stats[-1]
    assert st["spills"] >= 2 and st["groups"] >= 2 and st["reads"] == 1_000_000
    assert st["device_bytes"] <= budget


# ---- the collator on its own ---------------------------------------------------------------------------------------
def _key_columns(n_reads, seed, long_read=0):
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


@pytest.mark.gpu
def test_add_shapes_and_device_input(gpu):
    small = _key_columns(4000, 21)
    want = _want(small)
    budget = 400_000   # a staging area of about 6 800 rows: the 12 000 rows spill twice
    results = [_collate(small, chunk=c, collate_budget=budget) for c in (1, 7, 1000, None)]
    results += [_collate(small, chunk=c, device=True, collate_budget=budget) for c in (1000, None)]
    for got, reads, st in results:
        _same_result(got, want)
        assert reads == 4000 == st["reads"] and st["alignments"] == len(small[2])
        assert st["spills"] >= 2 and st["groups"] >= 1 and st["device_bytes"] <= budget
        assert st["d2h_bytes"] > 28 * st["alignments"]


@pytest.mark.gpu
def test_read_across_spills(gpu):
    cols = _key_columns(20000, 22, long_read=5000)   # one read's 5 000 rows are scattered over the whole input
    want = _want(cols)
    got, reads, st = _collate(cols, chunk=3000, collate_budget=600_000)
    _same_result(got, want)
    assert reads == 20000 and st["spills"] >= 5 and st["groups"] >= 2


@pytest.mark.gpu
def test_budget_too_small_for_the_read_order(gpu):
    from alntools_b200._native import EcbError
    cols = _key_columns(100_000, 23)   # n / 4 + 8 B per read is about 875 kB
    with pytest.raises(EcbError) as info:
        _collate(cols, collate_budget=400_000)
    assert info.value.code == LIMIT and "400000" in str(info.value)
    with pytest.raises(EcbError) as info:
        _collate(cols, collate_budget=10_000)   # not even a staging area
    assert info.value.code == LIMIT and "10000" in str(info.value)


# ---- long reads, empty input ---------------------------------------------------------------------------------------
REFS = [("T%d_%s" % (t, h), 100 + t) for t in range(6) for h in "AB"]


def _long_read_file(path, k, grouped):
    rng = np.random.default_rng(k)
    recs = [("long", 0, int(rng.integers(0, 12)), int(rng.integers(0, 90))) for _ in range(k)]
    recs += [("r%05d" % i, 0, int(rng.integers(0, 12)), 5) for i in range(3000)]
    if not grouped:
        recs = [recs[i] for i in rng.permutation(len(recs))]
    bam_io.write_bam(path, REFS, recs, block_payload=20000)
    return path


@pytest.mark.gpu
def test_long_reads_in_spill_mode(gpu, tmp_path, monkeypatch, collator_stats):
    from alntools_b200._native import EcbError
    budget = 2_000_000   # below the one-pass footprint of 19 384 rows, above the names pass of the long read's bucket
    f = _long_read_file(str(tmp_path / "ok.bam"), 16384, grouped=False)
    got = _convert(f, tmp_path, "got", monkeypatch, budget=budget)
    assert got[2]["n_reads"] == 3001 and collator_stats[-1]["spills"] >= 1
    header, records = load_records(f)
    fp = str(tmp_path / "fp.bam")
    bam_io.write_bam(fp, list(zip(header.references, header.lengths)), _regrouped(records))
    assert _convert(fp, tmp_path, "want", monkeypatch, collate=False)[0] == got[0]
    with pytest.raises(EcbError) as info:
        _convert(_long_read_file(str(tmp_path / "long.bam"), 16385, grouped=False), tmp_path, "x", monkeypatch,
                 budget=budget)
    assert info.value.code == LIMIT and "16384" in str(info.value)
    assert collator_stats == [collator_stats[0]]   # the failing call raised inside stream_collated


@pytest.mark.gpu
def test_no_valid_alignment(gpu, tmp_path, monkeypatch):
    f = str(tmp_path / "none.bam")
    bam_io.write_bam(f, REFS, [("a", 4, 0), ("b", 1 | 0x80, 1), ("a", 4, 2)])
    with pytest.raises(RuntimeError, match="three positive integers"):
        _convert(f, tmp_path, "x", monkeypatch, budget=30_000)


# ---- the environment variable (no GPU) -----------------------------------------------------------------------------
@pytest.mark.parametrize("value", ["-1", "abc", "1e9", "1.5", "12 MB", "０"])
def test_bad_budget_is_refused_before_any_file_is_opened(value, tmp_path, monkeypatch):
    monkeypatch.setenv(ENV, value)
    missing = str(tmp_path / "missing.bam")
    with pytest.raises(ValueError, match=ENV):
        bam_utils.convert(missing, str(tmp_path / "x.bin"), None, collate=True)
    assert not os.path.exists(str(tmp_path / "x.bin"))


def test_budget_values(monkeypatch):
    for value, want in ((None, 0), ("", 0), ("0", 0), (" 123 ", 123), (str(1 << 40), 1 << 40)):
        if value is None:
            monkeypatch.delenv(ENV, raising=False)
        else:
            monkeypatch.setenv(ENV, value)
        assert emitter.collate_budget() == want


# ---- bench.py's bam_e2e sample at 1/8 of the unbudgeted device bytes -----------------------------------------------
@pytest.mark.gpu
def test_eight_million_shuffled_reads_at_an_eighth(gpu, tmp_path, monkeypatch, collator_stats):
    cols = synth.make_columns(8_000_000, N_TARGETS, N_HAPS, 1002, mode="diploid")
    rg, tg, hp = _layouts(cols, 5)["shuffled"]
    f, fp = str(tmp_path / "f.bam"), str(tmp_path / "fp.bam")
    _write_columns(f, rg, tg, hp)
    order = _regrouped_columns(rg)
    _write_columns(fp, rg[order], tg[order], hp[order])
    free = _convert(f, tmp_path, "free", monkeypatch)
    budget = collator_stats[-1]["device_bytes"] // 8
    assert collator_stats[-1]["spills"] == 0
    got = _convert(f, tmp_path, "got", monkeypatch, budget=budget)
    st = collator_stats[-1]
    want = _convert(fp, tmp_path, "want", monkeypatch, collate=False)
    assert hashlib.sha256(got[0]).hexdigest() == hashlib.sha256(want[0]).hexdigest() == hashlib.sha256(free[0]).hexdigest()
    assert got[2]["n_reads"] == want[2]["n_reads"] == 8_000_000
    assert st["spills"] >= 2 and st["groups"] >= 2 and st["device_bytes"] <= budget
