"""The streaming build at the sizes of real inputs: EC-table growth between pushes, probe overflow and the replay
of reads and of parked hot-cache entries, the remap of (file, EC, cell) keys when the EC table grows, pipelined
host pushes, and the per-cell finalisation at its shape and cell-count edges.  Every result is compared bit for
bit with the oracle (the C statement above about 100 k reads), and every test asserts from the builder's stats
that the path it is about has run, so that it fails rather than passes if a change of input or sizing stops it
from getting there."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CELL_KEYS = ("a_indptr", "a_indices", "a_data", "n_indptr", "n_indices", "n_data", "cell_order")


@pytest.fixture(scope="module")
def native(built):
    import torch
    assert torch.cuda.is_available(), "these tests need a B200"
    from alntools_b200 import _native
    _native.load_library()
    return _native


# ---------------------------------------------------------------- helpers
def _read_cuts(rg, every):
    """Read-aligned cut points about `every` alignments apart, as a converter cuts its chunks."""
    cuts = [0]
    while cuts[-1] < len(rg):
        c = min(len(rg), cuts[-1] + every)
        while c < len(rg) and rg[c] == rg[c - 1]:
            c += 1
        cuts.append(c)
    return cuts


def _uniform_pairs(n_reads, n_targets, n_haps, rng, first_read=0):
    """Reads of exactly two alignments, targets and haplotypes uniform: almost every read is an EC of its own."""
    rg = np.repeat(np.arange(first_read, first_read + n_reads, dtype=np.int32), 2)
    tg = rng.integers(0, n_targets, 2 * n_reads, dtype=np.int32)
    hp = rng.integers(0, n_haps, 2 * n_reads, dtype=np.int32)
    return rg, tg, hp


def _read_starts(rg, drop_last):
    """Offsets of the reads a push counts (the last one is not counted when drop_last)."""
    if len(rg) == 0:
        return np.zeros(0, dtype=np.int64)
    starts = np.flatnonzero(np.concatenate(([True], rg[1:] != rg[:-1])))
    return starts[:-1] if drop_last else starts


def _counted_reads(pushes):
    return sum(len(_read_starts(p[0], p[4])) for p in pushes)


def _cell_totals(pushes):
    """(cell ids, reads counted per cell) over all pushes; a read's cell is the one on its first alignment."""
    cells = np.concatenate([np.asarray(p[3])[_read_starts(p[0], p[4])] for p in pushes] + [np.zeros(0, np.int32)])
    return np.unique(cells, return_counts=True)


def _assert_single(got, want):
    indptr, indices, data, counts, n_reads = want
    assert got["n_reads"] == n_reads
    assert got["n_ec"] == len(counts)
    assert np.array_equal(got["a_indptr"], indptr)
    assert np.array_equal(got["a_indices"], indices)
    assert np.array_equal(got["a_data"], data)
    assert np.array_equal(got["n_data"], counts)
    assert got["n_indptr"].tolist() == [0, len(counts)]
    assert np.array_equal(got["n_indices"], np.arange(len(counts), dtype=np.int32))


def _cells_oracle(pushes, min_cell_count):
    """The per-cell result, from the C statement of the merge above about 100 k reads and from the Python one
    below.  Raises ValueError where the reference refuses: when no read is counted at all, and when no cell
    reaches the minimum count (ec_oracle.convert_multisample: the reference cannot shape an empty matrix)."""
    from oracle import c_oracle, ec_oracle
    n_reads = _counted_reads(pushes)
    if n_reads > 100_000:
        want = c_oracle.ec_from_columns_cells(pushes, min_cell_count)
        assert want["n_reads"] == n_reads
    else:
        want = ec_oracle.ec_from_columns_cells(pushes, min_cell_count)
        want["n_reads"] = n_reads
    if len(want["cell_order"]) == 0:
        raise ValueError("no cell reaches the minimum count")
    return want


def _assert_cells(got, want):
    assert got["n_reads"] == want["n_reads"]
    assert got["n_ec"] == len(want["a_indptr"]) - 1
    for k in CELL_KEYS:
        assert np.array_equal(got[k], want[k]), k


def _run_cells(native, pushes, n_targets, n_haps, min_cell_count, **options):
    """Pushes in file order with a running order_base and no alignments hint, as convert_files() makes them."""
    with native.EcBuilder(n_targets, n_haps, with_cells=True, alignments_hint=0, **options) as b:
        base = 0
        for rg, tg, hp, cell, drop in pushes:
            b.push(rg, tg, hp, cell, order_base=base, drop_last_group=drop)
            base += len(rg)
        return b.finalize(min_cell_count), b.stats()


# ---------------------------------------------------------------- single sample: growth, overflow, replay
def test_streamed_single_sample_grows_ahead_of_pushes(native):
    """cfg2's shape at 3 M reads (6.16 M alignments, about 596 k ECs) streamed as bam_utils.convert() streams a
    BAM: no alignments hint, pageable results, read-aligned pushes of about 2^21 alignments with a running
    order_base.  The first push (237 k ECs) sizes the table at 524 288 slots; the projection made before the
    second push grows it, so that no read runs out of probes.  The converter writes its files from the views of
    finalize(copy=False), which are checked as well."""
    from alntools_b200 import synth
    from oracle import c_oracle
    cols = synth.make_columns(3_000_000, 100_000, 2, seed=7, mode="diploid")
    rg, tg, hp = cols["read_group"], cols["target_idx"], cols["hap_idx"]
    cuts = _read_cuts(rg, 1 << 21)
    assert len(cuts) - 1 == 3
    want = c_oracle.ec_from_columns(rg, tg, hp)
    with native.EcBuilder(100_000, 2, alignments_hint=0, pageable_results=1) as b:
        for i, (a, e) in enumerate(zip(cuts[:-1], cuts[1:])):
            b.push(rg[a:e], tg[a:e], hp[a:e], order_base=a)
            if i == 0:
                first = b.stats()
                assert first["table_slots"] == 524_288 and first["table_grows"] == 0
        stats = b.stats()
        assert stats["table_grows"] >= 1 and stats["overflow_reads"] == 0
        views = b.finalize(copy=False)
        assert not views["a_indices"].flags["OWNDATA"]
        assert views["n_alignments"] == len(rg)
        _assert_single(views, want)


@pytest.mark.parametrize("hot_cache", [1, 0])
def test_ec_rich_push_overflows_then_grows_ahead_of_the_next(native, hot_cache):
    """2^20 reads of two alignments uniform over 140 000 targets x 8 haplotypes: 2^21 alignments and about
    1.05 M ECs against the 524 288 slots sized from that first push, so probes run out in the middle of the push
    and the reads that did not fit are replayed into a table grown x4.  A second push of the same kind then
    finds the table too small for its projection and grows it before it starts."""
    from oracle import c_oracle
    rng = np.random.default_rng(11)
    nr = 1 << 20
    p1 = _uniform_pairs(nr, 140_000, 8, rng)
    p2 = _uniform_pairs(nr, 140_000, 8, rng, first_read=nr)
    want = c_oracle.ec_from_columns(*(np.concatenate(c) for c in zip(p1, p2)))
    with native.EcBuilder(140_000, 8, alignments_hint=0, hot_cache=hot_cache) as b:
        b.push(*p1, order_base=0)
        first = b.stats()
        assert first["overflow_reads"] > 0 and first["table_grows"] >= 1
        b.push(*p2, order_base=2 * nr)
        stats = b.stats()
        assert stats["table_grows"] > first["table_grows"] and stats["overflow_reads"] == first["overflow_reads"]
        _assert_single(b.finalize(), want)


@pytest.mark.parametrize("chunk_len", [32, 64, 160])
def test_parked_hot_cache_entries_are_replayed_with_their_counts(native, chunk_len):
    """The spill replay, built on purpose.  One CTA (so one hot-EC cache sees every read) and a table of 1 024
    slots.  16 384 reads with distinct ECs come first; by the time any warp takes a chunk after them, at least
    9 000 of them have been offered to the table (at most 63 wait in each of the 32 warps' queues), so the table
    is full.  Then 8 hot keys follow, 200 reads each, shuffled over many chunks.  A hot key's first read misses
    the cache, is queued, finds no slot and is flagged for the read replay (count 1).  Its next read is admitted
    to the cache (the key has missed once), and the cache counts all later ones.  When the CTA flushes its cache
    the table is still full, so the entry - with the count of all the key's later reads - is parked in the spill
    list and replayed after the table has grown.  A hot key whose cache entry a distinct key took first just overflows read
    by read; with eight of them, some are parked.  The hot counts are right only if the parked entries are
    replayed with their counts."""
    from oracle import ec_oracle
    rng = np.random.default_rng(77)
    n_distinct, n_hot, reps = 16_384, 8, 200
    hot = np.repeat(np.arange(n_hot), reps)
    rng.shuffle(hot)
    tg = np.concatenate([rng.permutation(n_distinct), n_distinct + hot]).astype(np.int32)
    rg = np.arange(len(tg), dtype=np.int32)
    hp = np.zeros(len(tg), dtype=np.int32)
    want = ec_oracle.ec_from_columns(rg, tg, hp) + (len(rg),)
    assert sorted(want[3].tolist())[-n_hot:] == [reps] * n_hot
    with native.EcBuilder(n_distinct + n_hot, 1, alignments_hint=0, grid_ctas=1, table_slots=1024, hot_cache=1,
                          chunk_len=chunk_len) as b:
        b.push(rg, tg, hp)
        stats = b.stats()
        assert stats["overflow_reads"] > n_distinct - 1024 and stats["table_grows"] >= 1
        _assert_single(b.finalize(), want)


# ---------------------------------------------------------------- per cell: growth, remap, replay, pipelining
def test_streamed_cells_remap_triples_when_the_table_grows(native):
    """Three files of cfg2-shaped reads (750 k reads each, 2 000 Zipf-sized cells) pushed as convert_files()
    pushes them: last read dropped, running order_base, no alignments hint.  The table is sized from the first
    file and grows ahead of a later one; every growth rewrites the EC-slot half of every (file, EC, cell) key.
    Checked with every cell kept and with a minimum count that some cell meets exactly and about half miss."""
    from alntools_b200 import synth
    files = [synth.make_columns(750_000, 100_000, 2, seed=40 + f, mode="diploid", n_cells=2000) for f in range(3)]
    pushes = [(c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"], True) for c in files]
    _, totals = _cell_totals(pushes)
    median = int(np.sort(totals)[len(totals) // 2])
    for min_cell_count in (1, median):
        want = _cells_oracle(pushes, min_cell_count)
        got, stats = _run_cells(native, pushes, 100_000, 2, min_cell_count)
        assert stats["table_grows"] >= 1 and stats["overflow_reads"] == 0
        _assert_cells(got, want)
    assert len(want["cell_order"]) < len(totals)


def test_cells_overflow_replay_records_the_cell(native):
    """A table of 1 024 slots against two files of 20 k diploid reads over 20 k targets and 300 cells: probes run
    out in the first push, the table grows in the middle of it (remapping the triples already recorded), and
    every replayed read must add its (file, EC, cell) count as well."""
    from alntools_b200 import synth
    files = [synth.make_columns(20_000, 20_000, 2, seed=50 + f, mode="diploid", n_cells=300) for f in range(2)]
    pushes = [(c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"], True) for c in files]
    for min_cell_count in (1, 40):
        want = _cells_oracle(pushes, min_cell_count)
        got, stats = _run_cells(native, pushes, 20_000, 2, min_cell_count, table_slots=1024)
        assert stats["overflow_reads"] > 0 and stats["table_grows"] >= 1
        _assert_cells(got, want)


def test_pipelined_cells_push_grows_between_its_pieces(native):
    """One host push of 8.4 M reads of two uniform alignments (16.8 M alignments, more than two pipeline pieces
    of 8 Mi), 50 000 cells, then a smaller second file, no alignments hint.  The table starts at n/4 rounded up
    (8 Mi slots) against about 8.3 M ECs: the first piece fills half of it and the projection grows it before the
    second piece, which shares the first one's file id."""
    rng = np.random.default_rng(61)
    pushes = []
    for n_reads, first_read in ((8_400_000, 0), (300_000, 5)):
        rg, tg, hp = _uniform_pairs(n_reads, 140_000, 8, rng, first_read)
        cell = np.repeat(rng.integers(0, 50_000, n_reads, dtype=np.int32), 2)
        pushes.append((rg, tg, hp, cell, True))
    assert len(pushes[0][0]) >= 2 * (8 << 20)
    _, totals = _cell_totals(pushes)
    min_cell_count = int(np.sort(totals)[len(totals) // 2])
    want = _cells_oracle(pushes, min_cell_count)
    with native.EcBuilder(140_000, 8, with_cells=True, alignments_hint=0) as b:
        b.push(*pushes[0][:4], order_base=0, drop_last_group=True)
        first = b.stats()
        assert first["table_grows"] >= 1 and first["overflow_reads"] == 0
        b.push(*pushes[1][:4], order_base=len(pushes[0][0]), drop_last_group=True)
        got = b.finalize(min_cell_count)
    _assert_cells(got, want)


# ---------------------------------------------------------------- per cell: shapes, geometry, boundaries
def test_cells_randomised_shapes_and_launch_geometry(native):
    """Many small per-cell jobs against the oracle: 1-5 files with read lengths around 8, 32 and 1 024, 1 to
    3 000 cells with dense or sparse ids, empty files and files of one (dropped) read, drop_last_group either
    way, random grids and chunk lengths, a 1 024-slot table on some jobs, and minimum counts of 0, 1, the exact
    total of some cell and more than any cell has.  Where nothing survives, the builder refuses as the reference
    does."""
    rng = np.random.default_rng(2025)
    pools = [[1, 7, 8, 9], [1, 2, 8, 16, 17], [31, 32, 33], [1, 30, 32, 64, 65], [1, 2, 1023, 1024, 1025]]
    seen = {"refused": 0, "empty_file": 0, "one_read_file": 0, "sparse": 0, "small_table": 0, "replayed": 0}
    for case in range(60):
        pool = pools[case % len(pools)]
        n_cells = [1, 2, 37, 3000][(case // 5) % 4]
        stride = 1 if case % 3 else int(rng.integers(2, 1_000_000 // n_cells))
        offset = int(rng.integers(0, stride))
        n_targets, n_haps = int(rng.choice([3, 50, 5000])), int(rng.choice([1, 2, 8]))
        n_files = int(rng.integers(1, 6))
        pushes = []
        for f in range(n_files):
            if case % 7 == 2 and f == 0:
                n_reads, drop = 0, bool(rng.integers(0, 2))                    # an empty push
            elif case % 7 == 4 and f == n_files - 1:
                n_reads, drop = 1, True                                        # one read, dropped
            else:
                n_reads = int(rng.integers(1, 25 if max(pool) > 100 else 1500))
                drop = bool(rng.integers(0, 2))
            lens = rng.choice(pool, n_reads)
            rg = np.repeat(np.arange(n_reads, dtype=np.int32) * 3 + 1, lens)
            n = len(rg)
            read_cell = ((rng.zipf(1.3, n_reads) - 1) % n_cells) * stride + offset
            pushes.append((rg, rng.integers(0, n_targets, n, dtype=np.int32), rng.integers(0, n_haps, n, dtype=np.int32),
                           np.repeat(read_cell, lens).astype(np.int32), drop))
            seen["empty_file"] += n_reads == 0
            seen["one_read_file"] += n_reads == 1 and drop
        seen["sparse"] += stride > 1
        ids, totals = _cell_totals(pushes)
        kind = case % 4
        min_cell_count = (0 if kind == 0 else 1 if kind == 1 or len(totals) == 0
                          else int(rng.choice(totals)) if kind == 2 else int(totals.max()) + 1)
        opts = {"grid_ctas": int(rng.choice([0, 1, 2, 7])), "chunk_len": int(rng.choice([0, 32, 64, 160, 1024]))}
        if rng.integers(0, 3) == 0:
            opts["table_slots"] = 1024
            seen["small_table"] += 1
        try:
            want = _cells_oracle(pushes, min_cell_count)
        except ValueError:
            want = None
        with native.EcBuilder(n_targets, n_haps, with_cells=True, alignments_hint=0, **opts) as b:
            base = 0
            for rg, tg, hp, cell, drop in pushes:
                b.push(rg, tg, hp, cell, order_base=base, drop_last_group=drop)
                base += len(rg)
            if want is None:
                with pytest.raises(native.EcbError) as info:
                    b.finalize(min_cell_count)
                assert info.value.code == native.ECB_ERR_EMPTY, case
                seen["refused"] += 1
            else:
                got = b.finalize(min_cell_count)
                _assert_cells(got, want)
            seen["replayed"] += b.stats()["overflow_reads"] > 0
    assert all(v >= 2 for v in seen.values()), seen


@pytest.mark.parametrize("n_kept", [255, 256, 257, 65535, 65536, 65537])
def test_kept_cell_counts_at_radix_pass_boundaries(native, n_kept):
    """Kept-cell counts on both sides of the 8-bit passes of the pair sort, whose key is the output column above
    the EC id (32 + bits_for(kept cells) bits: a column of 256 or of 65 536 needs one more pass).  The cell sort
    runs over several 2 048-key tiles from 2 049 cells on.  Kept cells have 3 or 4 reads and the minimum count is
    3, so many meet it exactly; 97 further cells of 1 or 2 reads are filtered.  Cell ids are shuffled against
    their first occurrence."""
    rng = np.random.default_rng(n_kept)
    min_cell_count, n_low = 3, 97
    totals = np.concatenate([rng.integers(3, 5, n_kept), rng.integers(1, 3, n_low)])
    ids = rng.permutation(len(totals)).astype(np.int32)
    read_cell = np.repeat(ids, totals)
    rng.shuffle(read_cell)
    n_reads = len(read_cell)
    lens = rng.integers(1, 3, n_reads)
    rg = np.repeat(np.arange(n_reads, dtype=np.int32), lens)
    tg = rng.integers(0, 300, len(rg), dtype=np.int32)
    hp = rng.integers(0, 2, len(rg), dtype=np.int32)
    cell = np.repeat(read_cell, lens).astype(np.int32)
    cut = _read_cuts(rg, len(rg) // 2)[1]
    pushes = [(rg[:cut], tg[:cut], hp[:cut], cell[:cut], False), (rg[cut:], tg[cut:], hp[cut:], cell[cut:], False)]
    want = _cells_oracle(pushes, min_cell_count)
    assert len(want["cell_order"]) == n_kept
    got, _ = _run_cells(native, pushes, 300, 2, min_cell_count)
    _assert_cells(got, want)


# ---------------------------------------------------------------- per cell: context reuse, device columns
def _cell_job(seed, n_files, n_reads, n_cells, mode):
    from alntools_b200 import synth
    files = [synth.make_columns(n_reads, 800, 2, seed=seed + f, mode=mode, n_cells=n_cells, dup_rate=0.02)
             for f in range(n_files)]
    return [(c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"], True) for c in files]


def test_cells_reset_between_jobs_equals_fresh_contexts(native):
    """Two different per-cell jobs, and the first again, on one context with reset() in between: every result
    equals that of a fresh context and the oracle's."""
    jobs = [(_cell_job(80, 2, 30_000, 200, "diploid"), 1), (_cell_job(90, 3, 12_000, 50, "light"), 10)]
    wants = [_cells_oracle(p, m) for p, m in jobs]
    for (pushes, m), want in zip(jobs, wants):
        _assert_cells(_run_cells(native, pushes, 800, 2, m)[0], want)
    with native.EcBuilder(800, 2, with_cells=True, alignments_hint=0) as b:
        for k in (0, 1, 0):
            pushes, m = jobs[k]
            base = 0
            for rg, tg, hp, cell, drop in pushes:
                b.push(rg, tg, hp, cell, order_base=base, drop_last_group=drop)
                base += len(rg)
            _assert_cells(b.finalize(m), wants[k])
            b.reset()


@pytest.mark.parametrize("misaligned", ["none", "all", "cell"])
def test_cells_device_resident_columns(native, misaligned):
    """All four columns pushed as CUDA tensors: aligned, as 4-byte-misaligned views (the push stages them), and
    with only the cell column misaligned, which the push reads in place: whether to stage is decided from the
    other three columns, and the cell is read with scalar loads."""
    import torch
    pushes = _cell_job(70, 3, 25_000, 500, "diploid")
    want = _cells_oracle(pushes, 5)

    def dev(a, shift):
        t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
        if shift:
            t = torch.cat([torch.zeros(1, dtype=torch.int32, device="cuda"), t])[1:]
        assert (t.data_ptr() % 16 != 0) == shift
        return t

    with native.EcBuilder(800, 2, with_cells=True, alignments_hint=0) as b:
        base = 0
        for rg, tg, hp, cell, drop in pushes:
            cols = [dev(a, misaligned == "all") for a in (rg, tg, hp)] + [dev(cell, misaligned != "none")]
            b.push(*cols, order_base=base, drop_last_group=drop)
            base += len(rg)
        got = b.finalize(5)
    _assert_cells(got, want)
