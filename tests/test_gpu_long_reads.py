"""Reads longer than 16384 alignments (ECB_OPT_MAX_READ, EcBuilder(max_read=...), ALNTOOLS_B200_MAX_READ).

The grouping kernel defers such reads and a sort-based pass keys, counts and harvests them (ecb_longread.cuh).  Every
result is compared with the C oracle, which has no read-length limit, as the reference has none
(alntools/bam_utils.py:322-323)."""
import os

import numpy as np
import pytest

from alntools_b200 import bam_utils, bam_utils_multisample, bin_utils, synth
from alntools_b200.header import TargetTables
from oracle import c_oracle, ec_oracle

pytestmark = pytest.mark.gpu

PUSH_LIMIT = (1 << 31) - 8192
N_TARGETS, N_HAPS = 5000, 4


@pytest.fixture(scope="module")
def native(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")
    from alntools_b200 import _native
    _native.load_library()
    return _native


# ---- columns ------------------------------------------------------------------------------------------------------
def _reads(spec, seed, n_targets=N_TARGETS, n_haps=N_HAPS):
    """spec: list of read lengths, or (length, kind) with kind "one" (a single distinct element), "all" (every target)
    or "narrow" (200 targets: many duplicates).  Plain lengths draw from every target."""
    rng = np.random.default_rng(seed)
    lens = np.asarray([item[0] if isinstance(item, tuple) else item for item in spec], dtype=np.int64)
    starts = np.r_[0, np.cumsum(lens)]
    rg = np.repeat(np.arange(len(lens)), lens)
    tg = rng.integers(0, n_targets, len(rg))
    hp = rng.integers(0, n_haps, len(rg))
    for i, item in enumerate(spec):
        if not isinstance(item, tuple):
            continue
        a, z = starts[i], starts[i + 1]
        if item[1] == "one":
            tg[a:z], hp[a:z] = 17, 1
        elif item[1] == "all":
            tg[a:z] = np.arange(z - a) % n_targets
        elif item[1] == "narrow":
            tg[a:z] = rng.integers(0, 200, z - a)
    return {"read_group": rg.astype(np.int32), "target_idx": tg.astype(np.int32), "hap_idx": hp.astype(np.int32)}


def _short(n, seed):
    rng = np.random.default_rng(seed)
    return [int(x) for x in rng.integers(1, 9, n)]


def _with_long(long_spec, n_short=20000, seed=0, where="middle"):
    short = _short(n_short, seed)
    if where == "first":
        spec = list(long_spec) + short
    elif where == "last":
        spec = short + list(long_spec)
    else:   # spread between the short reads
        spec = list(short)
        step = max(1, len(short) // (len(long_spec) + 1))
        for j, item in enumerate(long_spec):
            spec.insert((j + 1) * step + j, item)
    return _reads(spec, seed + 1)


def _n_long(cols):
    _, counts = np.unique(cols["read_group"], return_counts=True)
    return int((counts > 16384).sum())


def _oracle(cols, drop_last=False):
    return c_oracle.ec_from_columns(cols["read_group"], cols["target_idx"], cols["hap_idx"], drop_last)


def _assert_same(got, want):
    indptr, indices, data, counts, n_reads = want
    assert got["n_reads"] == n_reads
    assert got["n_ec"] == len(counts)
    assert np.array_equal(got["a_indptr"], indptr)
    assert np.array_equal(got["a_indices"], indices)
    assert np.array_equal(got["a_data"], data)
    assert np.array_equal(got["n_data"], counts)


def _run(native, cols, pushes=None, device=False, **options):
    options.setdefault("max_read", 0)
    with native.EcBuilder(N_TARGETS, N_HAPS, **options) as b:
        n = len(cols["read_group"])
        if device:
            import torch
            dev = {k: torch.from_numpy(cols[k]).cuda() for k in ("read_group", "target_idx", "hap_idx")}
            b.push(dev["read_group"], dev["target_idx"], dev["hap_idx"])
            torch.cuda.synchronize()
        elif pushes is None:
            b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
        else:
            stats = []
            for a, z in pushes:
                b.push(cols["read_group"][a:z], cols["target_idx"][a:z], cols["hap_idx"][a:z], order_base=a)
                stats.append(b.stats())
            return b.finalize(), stats
        assert n > 0
        return b.finalize(), b.stats()


# ---- the option -----------------------------------------------------------------------------------------------------
def test_option_values(native):
    with native.EcBuilder(100, 2) as b:
        for bad in (1, 16383, -1, PUSH_LIMIT + 1):
            with pytest.raises(native.EcbError) as info:
                b.set_option("max_read", bad)
            assert info.value.code == -1
        for good in (0, 16384, PUSH_LIMIT, 20000):
            b.set_option("max_read", good)
    for limit in (20000, 16384):
        for k, ok in ((limit, True), (limit + 1, False)):
            cols = _with_long([k], n_short=100)
            with native.EcBuilder(N_TARGETS, N_HAPS, max_read=limit) as b:
                if ok:
                    b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
                    _assert_same(b.finalize(), _oracle(cols))
                else:
                    with pytest.raises(native.EcbError) as info:
                        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
                    assert info.value.code == -4 and str(limit) in str(info.value)
    # the default keeps its message
    cols = _with_long([16385], n_short=10)
    with native.EcBuilder(N_TARGETS, N_HAPS) as b:
        with pytest.raises(native.EcbError) as info:
            b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
        assert info.value.code == -4 and "16384" in str(info.value)


# ---- columns against the oracle -------------------------------------------------------------------------------------
CASES = {
    "16385": ([16385], "middle"),
    "16416": ([16416], "middle"),
    "1e5": ([100_000], "middle"),
    "1e6": ([1_000_000], "middle"),
    "first": ([50_000], "first"),
    "last": ([50_000], "last"),
    "one_element": ([(40_000, "one")], "middle"),
    "every_target": ([(3 * N_TARGETS + 7 + 16384, "all")], "middle"),
    "narrow": ([(60_000, "narrow"), (17_000, "narrow")], "middle"),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_columns(native, case):
    spec, where = CASES[case]
    cols = _with_long(spec, where=where, seed=len(case))
    got, st = _run(native, cols)
    _assert_same(got, _oracle(cols))
    assert st["long_reads"] == _n_long(cols) == len(spec)
    assert st["long_ms"] > 0


def test_two_hundred_long_reads(native):
    rng = np.random.default_rng(5)
    cols = _with_long([int(k) for k in rng.integers(20_000, 70_001, 200)], n_short=50_000, seed=5)
    got, st = _run(native, cols)
    _assert_same(got, _oracle(cols))
    assert st["long_reads"] == 200


def test_grid_and_chunk_variations(native):
    cols = _with_long([100_000, 16_500], n_short=2000, seed=9)
    want = _oracle(cols)
    for grid, chunk in ((0, 0), (2, 256), (5, 32), (1, 4096)):
        got, st = _run(native, cols, grid_ctas=grid, chunk_len=chunk)
        _assert_same(got, want)
        assert st["long_reads"] == 2


def test_several_pushes_with_order_base(native):
    cols = _with_long([30_000, 100_000, 20_000, 16_385], n_short=30_000, seed=11)
    rg = cols["read_group"]
    starts = np.flatnonzero(np.r_[True, rg[1:] != rg[:-1]])
    cuts = [0] + [int(starts[np.searchsorted(starts, f * len(rg) // 4)]) for f in (1, 2, 3)] + [len(rg)]
    pieces = [(cuts[i], cuts[i + 1]) for i in range(4)]
    want = _oracle(cols)
    for order in (pieces, pieces[::-1], [pieces[2], pieces[0], pieces[3], pieces[1]]):
        got, stats = _run(native, cols, pushes=order)
        _assert_same(got, want)
        assert sum(s["long_reads"] for s in stats) == 4


def test_device_input(native):
    cols = _with_long([100_000, 40_000], seed=13)
    got, st = _run(native, cols, device=True)
    _assert_same(got, _oracle(cols))
    assert st["long_reads"] == 2


def test_pipelined_host_push_with_a_long_read_across_a_piece_cut(native):
    """A host push of at least 2 x 8 M alignments goes in read-aligned pieces of 8 M; the long read covers the first cut."""
    piece = 8 << 20
    rng = np.random.default_rng(17)
    head = []
    total = 0
    while total < piece - 50_000:
        k = int(rng.integers(1, 9))
        head.append(k)
        total += k
    spec = head + [100_000] + _short(2_200_000, 18) + [20_000]
    cols = _reads(spec, 19)
    n = len(cols["read_group"])
    assert n >= 2 * piece
    got, st = _run(native, cols)
    _assert_same(got, _oracle(cols))
    assert st["long_reads"] == 2


def test_table_growth_during_the_deferred_insert(native):
    cols = _with_long([20_000 + i for i in range(0, 3000, 100)], n_short=40_000, seed=23)
    got, st = _run(native, cols, table_slots=1024)
    _assert_same(got, _oracle(cols))
    assert st["table_grows"] >= 1 and st["long_reads"] == 30


def test_verify_keys(native):
    cols = _with_long([100_000, (30_000, "narrow"), (20_000, "one")], seed=29)
    got, st = _run(native, cols, verify_keys=1)
    _assert_same(got, _oracle(cols))
    assert st["long_reads"] == 3


# ---- one set, one EC ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("long_first", [True, False])
def test_long_and_short_read_with_one_set_are_one_ec(native, long_first):
    rng = np.random.default_rng(31)
    pairs = rng.choice(N_TARGETS * N_HAPS, 50, replace=False)
    t, h = (pairs // N_HAPS).astype(np.int32), (pairs % N_HAPS).astype(np.int32)
    k = 20_000
    idx = np.r_[np.arange(50), rng.integers(0, 50, k - 50)]
    long_read = (t[idx], h[idx])
    short_read = (t[::-1].copy(), h[::-1].copy())
    reads = [long_read, short_read] if long_first else [short_read, long_read]
    cols = {"read_group": np.repeat(np.arange(2), [len(r[0]) for r in reads]).astype(np.int32),
            "target_idx": np.concatenate([r[0] for r in reads]).astype(np.int32),
            "hap_idx": np.concatenate([r[1] for r in reads]).astype(np.int32)}
    got, st = _run(native, cols, verify_keys=1)
    want = _oracle(cols)
    _assert_same(got, want)
    assert got["n_ec"] == 1 and got["n_data"].tolist() == [2]
    assert st["long_reads"] == 1
    # the row is the set: every target once, the OR of its haplotype bits
    row = {}
    for a, b in zip(t.tolist(), h.tolist()):
        row[a] = row.get(a, 0) | (1 << b)
    assert got["a_indices"].tolist() == sorted(row)
    assert got["a_data"].tolist() == [row[a] for a in sorted(row)]


# ---- per cell -------------------------------------------------------------------------------------------------------
def _cells_file(spec, seed, n_cells):
    cols = _reads(spec, seed)
    rng = np.random.default_rng(seed + 100)
    cell_of_read = rng.integers(0, n_cells, len(spec))
    cols["cell_idx"] = cell_of_read[cols["read_group"]].astype(np.int32)
    return cols


def _first_appearance(files):
    """Cell ids renumbered by first appearance over the files in order (the ids the converters give)."""
    order = {}
    for f in files:
        for c in f["cell_idx"].tolist():
            order.setdefault(c, len(order))
    out = []
    for f in files:
        g = dict(f)
        g["cell_idx"] = np.asarray([order[c] for c in f["cell_idx"].tolist()], dtype=np.int32)
        out.append(g)
    return out, {v: k for k, v in order.items()}


def _cells_files(seed=37):
    f1 = _cells_file(_short(8000, seed)[:4000] + [30_000] + _short(4000, seed + 1) + [17_000], seed, 40)
    f2 = _cells_file([20_000] + _short(6000, seed + 2) + [100_000] + _short(3000, seed + 3), seed + 7, 40)
    f3 = _cells_file(_short(5000, seed + 4) + [(25_000, "narrow")], seed + 9, 40)
    return [f1, f2, f3]


@pytest.mark.parametrize("min_count", [1, 300])
def test_cells(native, min_count):
    files, _ = _first_appearance(_cells_files())
    want = c_oracle.ec_from_columns_cells([(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], True)
                                           for f in files], min_count)
    with native.EcBuilder(N_TARGETS, N_HAPS, with_cells=True, max_read=0) as b:
        base, deferred = 0, 0
        for f in files:
            b.push(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], order_base=base, drop_last_group=True)
            base += len(f["read_group"])
            deferred += b.stats()["long_reads"]
        got = b.finalize(min_count)
    assert deferred == 3   # the last read of files 1 and 3 is dropped, as by the reference
    for key in ("a_indptr", "a_indices", "a_data", "n_indptr", "n_indices", "n_data", "cell_order"):
        assert np.array_equal(got[key], want[key]), key


def test_convert_files(native, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    files, original = _first_appearance(_cells_files(41))
    paths = []
    for i, f in enumerate(files):
        p = str(tmp_path / ("f%d.bam" % i))
        raw = dict(f)
        raw["cell_idx"] = np.asarray([original[c] for c in f["cell_idx"].tolist()], dtype=np.int32)
        synth.columns_to_bam_cells(p, raw, N_TARGETS, N_HAPS)
        paths.append(p)
    out = str(tmp_path / "got.bin")
    bam_utils_multisample.convert_files(paths, out, None, 1)
    res = c_oracle.ec_from_columns_cells([(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], True)
                                          for f in files], 1)
    tables = _tables()
    want = str(tmp_path / "want.bin")
    bin_utils.ecsave2_arrays(want, tables.haplotypes, list(tables.main_targets), tables.lengths,
                             ["cell%07d" % original[c] for c in res["cell_order"].tolist()],
                             (res["a_indptr"], res["a_indices"], res["a_data"]),
                             (res["n_indptr"], res["n_indices"], res["n_data"]))
    with open(out, "rb") as a, open(want, "rb") as b:
        assert a.read() == b.read()


# ---- convert() -------------------------------------------------------------------------------------------------------
def _tables():
    refs = synth.reference_names(N_TARGETS, N_HAPS)
    return TargetTables([r[0] for r in refs], [r[1] for r in refs], None)


def _want_file(cols, path):
    indptr, indices, data, counts, _ = _oracle(cols)
    tables = _tables()
    bin_utils.ecsave2_arrays(path, tables.haplotypes, list(tables.main_targets), tables.lengths, ["s"],
                             (indptr, indices, data), ec_oracle.n_matrix_single(counts))
    with open(path, "rb") as fh:
        return fh.read()


def _write_shuffled(path, cols, seed):
    """The alignments of cols in a random order (names 'read%09d'); -> the columns regrouped by name, reads in order
    of their first alignment, which is what collation makes of the file."""
    from alntools_b200 import bam_io
    perm = np.random.default_rng(seed).permutation(len(cols["read_group"]))
    rg, tg, hp = cols["read_group"][perm], cols["target_idx"][perm], cols["hap_idx"][perm]
    tids = tg.astype(np.int64) * N_HAPS + hp
    bam_io.write_bam_columns(path, synth.reference_names(N_TARGETS, N_HAPS), rg, np.zeros(len(rg), dtype=np.uint16),
                             tids, level=1)
    _, first = np.unique(rg, return_index=True)
    rank = np.empty(len(first), dtype=np.int64)
    rank[np.argsort(first, kind="stable")] = np.arange(len(first))
    o = np.argsort(rank[rg], kind="stable")
    return {"read_group": rank[rg][o].astype(np.int32), "target_idx": tg[o], "hap_idx": hp[o]}


@pytest.fixture(scope="module")
def long_bam(tmp_path_factory):
    d = tmp_path_factory.mktemp("long_bam")
    cols = _with_long([100_000], n_short=60_000, seed=43)
    grouped = str(d / "grouped.bam")
    synth.columns_to_bam(grouped, cols, N_TARGETS, N_HAPS)
    shuffled = str(d / "shuffled.bam")
    regrouped = _write_shuffled(shuffled, cols, 44)
    return {"grouped": grouped, "want": _want_file(cols, str(d / "want.bin")), "shuffled": shuffled,
            "want_shuffled": _want_file(regrouped, str(d / "want_shuffled.bin"))}


def _convert(bam, tmp_path, tag, **kw):
    out = str(tmp_path / (tag + ".bin"))
    bam_utils.convert(bam, out, None, sample="s", **kw)
    with open(out, "rb") as fh:
        return fh.read()


def test_convert_default_limit_still_refuses(native, long_bam, tmp_path, monkeypatch):
    monkeypatch.delenv("ALNTOOLS_B200_MAX_READ", raising=False)
    with pytest.raises(native.EcbError) as info:
        _convert(long_bam["grouped"], tmp_path, "x")
    assert info.value.code == -4 and "16384" in str(info.value)


def test_convert_host_decode(native, long_bam, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    assert _convert(long_bam["grouped"], tmp_path, "host") == long_bam["want"]


def test_convert_device_decode_small_windows(native, long_bam, tmp_path, monkeypatch):
    """Windows of 256 kB: the long read (about 4.5 MB of records) is open across many windows."""
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")

    class SmallWindows(native.EcBuilder):
        def __init__(self, *a, **kw):
            super().__init__(*a, **kw)
            self.set_option("bam_window", 256 << 10)

    monkeypatch.setattr(bam_utils, "EcBuilder", SmallWindows)
    assert _convert(long_bam["grouped"], tmp_path, "device", decode="device") == long_bam["want"]


def test_convert_collated(native, long_bam, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    monkeypatch.delenv("ALNTOOLS_B200_COLLATE_BUDGET", raising=False)
    assert _convert(long_bam["shuffled"], tmp_path, "collated", collate=True) == long_bam["want_shuffled"]
    assert _convert(long_bam["grouped"], tmp_path, "collated_grouped", collate=True) == long_bam["want"]


def test_convert_collated_spill(native, long_bam, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    monkeypatch.setenv("ALNTOOLS_B200_COLLATE_BUDGET", str(16_000_000))
    from alntools_b200 import _native
    stats = []
    real_push = _native.Collator.push

    def push(self):
        r = real_push(self)
        stats.append(self.stats())
        return r

    monkeypatch.setattr(_native.Collator, "push", push)
    assert _convert(long_bam["shuffled"], tmp_path, "spill", collate=True) == long_bam["want_shuffled"]
    assert stats and stats[0]["spills"] >= 1


def test_convert_python_emitter(native, long_bam, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    monkeypatch.setenv("ALNTOOLS_B200_EMITTER", "python")
    assert _convert(long_bam["grouped"], tmp_path, "python") == long_bam["want"]


def test_convert_rank_world_one(native, long_bam, tmp_path, monkeypatch):
    import json
    import subprocess
    import sys
    from conftest import ROOT
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    out = str(tmp_path / "rank.bin")
    code = ("import json, sys; sys.path.insert(0, %r); from alntools_b200 import bam_utils; a = json.loads(sys.argv[1]); "
            "bam_utils.convert_rank(a[0], a[1], None, sample='s')" % ROOT)
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29547")
    subprocess.check_call([sys.executable, "-c", code, json.dumps([long_bam["grouped"], out])], env=env, cwd=ROOT,
                          timeout=600)
    with open(out, "rb") as fh:
        assert fh.read() == long_bam["want"]
