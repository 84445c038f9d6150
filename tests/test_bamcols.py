"""libbamcols.so (native host column emitter, include/bamcols.h) against the record-level Python
statement of the same rules (alntools_b200/emitter.py), on the reference's golden BAMs and on
generated BAMs that exercise the filters, the name trimming, the per-cell quirks, records that
straddle BGZF blocks and reads that straddle emit() calls.  No GPU involved."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_records
from alntools_b200 import bam_io, bamcols, emitter
from alntools_b200.header import TargetTables


@pytest.fixture(scope="module", autouse=True)
def _built(built):
    bamcols.load_library()


def _native_single(path, tables=None, chunk=1 << 20, n_threads=0):
    with bamcols.BamColumnReader(path, n_threads) as r:
        t = tables or TargetTables(r.references, r.lengths, None)
        r.set_tables(t)
        cols = r.read_all(chunk=chunk)
        return cols, r.all_alignments, r.n_groups, r.references, r.lengths


def _python_single(path, tables=None):
    header, recs = load_records(path)
    t = tables or TargetTables(header.references, header.lengths, None)
    return emitter.emit_single(recs, t), header


def _same_single(path, **kw):
    cols, all_aln, n_groups, refs, lens = _native_single(path, **kw)
    want, header = _python_single(path)
    assert refs == tuple(header.references) and lens == tuple(header.lengths)
    assert np.array_equal(cols["read_group"], want.read_group)
    assert np.array_equal(cols["target_idx"], want.target_idx)
    assert np.array_equal(cols["hap_idx"], want.hap_idx)
    assert all_aln == want.all_alignments and n_groups == want.n_groups
    return cols


@pytest.mark.parametrize("case", golden_cases("single"), ids=lambda c: c["name"])
def test_golden_single(case):
    _same_single(os.path.join(GOLDEN, case["bam"]))
    _same_single(os.path.join(GOLDEN, case["bam"]), n_threads=1)


@pytest.mark.parametrize("case", golden_cases("multisample"), ids=lambda c: c["name"])
def test_golden_multisample(case):
    tables, cell_ids = None, {}
    cells = bamcols.CellDictionary()
    for fn in case["file_order"]:
        path = os.path.join(GOLDEN, case["dir"], fn)
        header, recs = load_records(path)
        if tables is None:
            tables = TargetTables(header.references, header.lengths, None)
        want = emitter.emit_multisample(recs, tables, cell_ids)
        with bamcols.BamColumnReader(path) as r:
            r.set_tables(tables)
            got = r.read_all(cells=cells)
        for k, w in (("read_group", want.read_group), ("target_idx", want.target_idx),
                     ("hap_idx", want.hap_idx), ("cell_idx", want.cell_idx)):
            assert np.array_equal(got[k], w), (fn, k)
    assert cells.names() == [n for n, _ in sorted(cell_ids.items(), key=lambda kv: kv[1])]


REFS = [("T%d_%s" % (t, h), 100 + t) for t in range(6) for h in "AB"]


def _write(tmp_path, alignments, name="x.bam", block_payload=60000):
    p = str(tmp_path / name)
    bam_io.write_bam(p, REFS, alignments, block_payload=block_payload)
    return p


def test_filters_trimming_and_tiny_blocks(tmp_path, monkeypatch):
    """Unmapped / read2 / improper / mate-elsewhere alignments are skipped, names are cut at the first
    blank (not at a leading one), and with 70-byte BGZF blocks nearly every record straddles blocks."""
    rng = np.random.default_rng(5)
    alns = []
    for i in range(400):
        name = ["r%d" % (i // 3), "r%d extra words" % (i // 3), " lead%d" % (i // 2), "q%d x" % i][int(rng.integers(0, 4))]
        flag = int(rng.choice([0, 16, 4, 1 | 2 | 64, 1 | 2 | 128, 1 | 64, 1 | 2 | 64 | 16]))
        tid = int(rng.integers(0, len(REFS)))
        ntid = tid if rng.random() < 0.7 else int(rng.integers(0, len(REFS)))
        npos = int(rng.choice([-1, 5, 100]))
        alns.append((name, flag, tid, 7, ntid, npos))
    for bp in (70, 300, 60000):
        _same_single(_write(tmp_path, alns, "f%d.bam" % bp, block_payload=bp))
    # every worker thread gets a handful of records: thread boundaries fall inside reads
    monkeypatch.setenv("BAMCOLS_GRAIN", "7")
    for nt in (2, 3, 8):
        _same_single(_write(tmp_path, alns, "g%d.bam" % nt, block_payload=300), n_threads=nt)


def test_reads_are_never_split_between_emit_calls(tmp_path):
    rng = np.random.default_rng(9)
    alns = []
    for read in range(300):
        for _ in range(int(rng.integers(1, 9))):
            alns.append(("read%05d" % read, 0, int(rng.integers(0, len(REFS)))))
    path = _write(tmp_path, alns)
    want, _ = _python_single(path)
    with bamcols.BamColumnReader(path) as r:
        r.set_tables(TargetTables(r.references, r.lengths, None))
        rg_all = []
        bufs = [np.empty(11, dtype=np.int32) for _ in range(3)]
        while True:
            n, done = r.emit(*bufs)
            part = bufs[0][:n].copy()
            if n:
                assert not rg_all or part[0] != rg_all[-1][-1]       # a new read starts every call
            if n:
                rg_all.append(part)
            if done:
                break
        assert np.array_equal(np.concatenate(rg_all), want.read_group)
    with bamcols.BamColumnReader(path) as r:                       # a read longer than the buffers
        r.set_tables(TargetTables(r.references, r.lengths, None))
        small = [np.empty(1, dtype=np.int32) for _ in range(3)]
        with pytest.raises(ValueError):
            while not r.emit(*small)[1]:
                pass


def _cell_name(read, cell, extra=""):
    return "%s|||CR|||x|||CY|||x|||UR|||x|||UY|||x|||BC|||x|||QT|||x|||CID|||%s%s" % (read, cell, extra)


def test_per_cell_quirks(tmp_path):
    """The remembered name stays untrimmed after the first switch (names with blanks open a read per
    alignment), the cell is taken from the remembered name, ids follow first appearance."""
    rng = np.random.default_rng(11)
    alns = []
    for read in range(200):
        cell = "CELL%02d" % int(rng.integers(0, 7))
        extra = " tail" if read % 5 == 0 else ""
        for _ in range(int(rng.integers(1, 4))):
            alns.append((_cell_name("q%04d" % read, cell, extra), 0, int(rng.integers(0, len(REFS)))))
    path = _write(tmp_path, alns, block_payload=500)
    header, recs = load_records(path)
    tables = TargetTables(header.references, header.lengths, None)
    cell_ids = {}
    want = emitter.emit_multisample(recs, tables, cell_ids)
    cells = bamcols.CellDictionary()
    with bamcols.BamColumnReader(path) as r:
        r.set_tables(tables)
        got = r.read_all(cells=cells, chunk=64)
    assert np.array_equal(got["read_group"], want.read_group)
    assert np.array_equal(got["cell_idx"], want.cell_idx)
    assert np.array_equal(got["target_idx"], want.target_idx)
    assert cells.names() == [n for n, _ in sorted(cell_ids.items(), key=lambda kv: kv[1])]


def test_per_cell_short_name_raises_index_error_like_the_reference(tmp_path):
    alns = [(_cell_name("a", "C1"), 0, 0), ("only|||three|||fields", 0, 1), (_cell_name("b", "C2"), 0, 2)]
    path = _write(tmp_path, alns)
    header, recs = load_records(path)
    tables = TargetTables(header.references, header.lengths, None)
    with pytest.raises(IndexError):
        emitter.emit_multisample(recs, tables, {})
    with bamcols.BamColumnReader(path) as r:
        r.set_tables(tables)
        with pytest.raises(IndexError):
            r.read_all(cells=bamcols.CellDictionary())


def test_not_a_bam_and_missing_file(tmp_path):
    p = tmp_path / "junk.bam"
    p.write_bytes(b"this is not a bam file at all")
    with pytest.raises(ValueError):
        bamcols.BamColumnReader(str(p))
    with pytest.raises(IOError):
        bamcols.BamColumnReader(str(tmp_path / "absent.bam"))
    good = _write(tmp_path, [("r", 0, 0)])
    data = open(good, "rb").read()
    cut = tmp_path / "cut.bam"
    cut.write_bytes(data[:len(data) - 40])                          # EOF block and part of the last block gone
    with pytest.raises(ValueError):
        with bamcols.BamColumnReader(str(cut)) as r:
            r.set_tables(TargetTables(r.references, r.lengths, None))
            r.read_all()


def test_large_synthetic_multi_batch(tmp_path):
    """More than one inflate batch (> 2048 blocks) and all worker threads."""
    from alntools_b200 import synth
    cols = synth.make_columns(120000, 300, 2, seed=3, mode="diploid")
    path = str(tmp_path / "big.bam")
    bam_io.write_bam_columns(path, synth.reference_names(300, 2), cols["read_group"],
                             np.zeros(len(cols["read_group"]), dtype=np.uint16),
                             cols["target_idx"].astype(np.int64) * 2 + cols["hap_idx"], block_payload=4000)
    with bamcols.BamColumnReader(path) as r:
        tables = TargetTables(r.references, r.lengths, None)
        r.set_tables(tables)
        got = r.read_all(chunk=1 << 16)
    assert np.array_equal(got["read_group"], cols["read_group"])
    assert np.array_equal(got["target_idx"], cols["target_idx"])
    assert np.array_equal(got["hap_idx"], cols["hap_idx"])


def _range_cases():
    import json
    with open(os.path.join(GOLDEN, "manifest_range.json")) as fh:
        return json.load(fh)


@pytest.mark.parametrize("case", _range_cases(), ids=lambda c: c["name"])
def test_range_file_matches_the_reference(case, tmp_path):
    """--rangefile (bam_utils.py:282-286,735-766): per-reference min/max of reference_start over the valid
    alignments, written like the reference; goldens minted by oracle/make_golden_range.py."""
    from alntools_b200 import utils
    files = ([os.path.join(GOLDEN, case["bam"])] if case["kind"] == "single"
             else [os.path.join(GOLDEN, case["dir"], fn) for fn in case["file_order"]])
    tfile = os.path.join(GOLDEN, case["targets"]) if case.get("targets") else None
    tables = lo = hi = refs = None
    cells = bamcols.CellDictionary() if case["kind"] == "multisample" else None
    for path in files:
        with bamcols.BamColumnReader(path) as r:
            if tables is None:
                tables = TargetTables(r.references, r.lengths, tfile)
                refs = r.references
            r.set_tables(tables)
            r.track_ranges(True)
            r.read_all(cells=cells)
            a, b = r.ranges()
            lo = a if lo is None else np.minimum(lo, a)
            hi = b if hi is None else np.maximum(hi, b)
    out = str(tmp_path / "range.txt")
    utils.write_range_file(out, list(tables.main_targets.keys()), tables.haplotypes, refs, lo, hi)
    with open(out) as a, open(os.path.join(GOLDEN, case["range"])) as b:
        assert a.read() == b.read()


def test_randomised_small_bams(tmp_path, monkeypatch):
    """Random small BAMs (names with blanks, every filter combination, tiny BGZF blocks, forced thread
    splits) through the native emitter and the record-level Python emitter."""
    rng = np.random.default_rng(77)
    flags = [0, 16, 4, 20, 1 | 2 | 64, 1 | 2 | 128, 1 | 64, 1 | 2 | 64 | 16, 1 | 2 | 64 | 4, 256, 2048]
    for case in range(25):
        n = int(rng.integers(1, 600))
        alns, read = [], 0
        for _ in range(n):
            if rng.random() < 0.4:
                read += 1
            name = ("r%d" % read) if read % 4 else ("r%d tail %d" % (read, int(rng.integers(0, 3))))
            tid = int(rng.integers(0, len(REFS)))
            alns.append((name, int(rng.choice(flags)), tid, int(rng.integers(0, 500)),
                         tid if rng.random() < 0.8 else int(rng.integers(0, len(REFS))), int(rng.choice([-1, 0, 77]))))
        monkeypatch.setenv("BAMCOLS_GRAIN", str(int(rng.choice([1, 5, 4096]))))
        monkeypatch.setenv("BAMCOLS_BATCH_BLOCKS", str(int(rng.choice([1, 3, 2048]))))
        path = _write(tmp_path, alns, "rand%d.bam" % case, block_payload=int(rng.choice([64, 200, 5000])))
        _same_single(path, n_threads=int(rng.choice([1, 2, 5])))


def _tables_equal(a, b):
    assert list(a.main_targets.items()) == list(b.main_targets.items())
    assert a.haplotypes == b.haplotypes
    assert np.array_equal(a.tid_target, b.tid_target) and np.array_equal(a.tid_hap, b.tid_hap)
    assert np.array_equal(a.lengths, b.lengths) and a.lengths.dtype == b.lengths.dtype
    assert (a.num_targets, a.num_haplotypes) == (b.num_targets, b.num_haplotypes)


def test_native_header_tables_equal_the_python_tables(tmp_path):
    """bamcols_build_tables against alntools_b200/header.py (the statement of bam_utils.py:561-633) on the
    golden headers, with target files, and on names that exercise the '_' rules."""
    for case in golden_cases("single"):
        path = os.path.join(GOLDEN, case["bam"])
        tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
        with bamcols.BamColumnReader(path) as r:
            _tables_equal(r.build_tables(tfile), TargetTables(r.references, r.lengths, tfile))
    refs = [("G1_A", 1), ("G1_B", 2), ("G2", 3), ("_G3", 4), ("G5_x_A", 5), ("G6_", 6), ("Z_A", 7), ("G2_B", 8)]
    p = str(tmp_path / "quirks.bam")
    bam_io.write_bam(p, refs, [("r", 0, 0)])
    tf = str(tmp_path / "t.txt")
    with open(tf, "w") as fh:
        fh.write("# comment\nZ\nG9 second token ignored\nG1\n")
    with bamcols.BamColumnReader(p) as r:
        _tables_equal(r.build_tables(None), TargetTables(r.references, r.lengths, None))
    with bamcols.BamColumnReader(p) as r:
        got = r.build_tables(tf)
        _tables_equal(got, TargetTables(r.references, r.lengths, tf))
        assert list(got.main_targets)[:3] == ["Z", "G9", "G1"]
        cols = r.read_all()                                   # the lookups are installed
        assert cols["target_idx"].tolist() == [2] and cols["hap_idx"].tolist() == [1]
    clash = str(tmp_path / "clash.bam")
    bam_io.write_bam(clash, [("a", 1), ("a_", 2)], [("r", 0, 0)])
    with bamcols.BamColumnReader(clash) as r:
        with pytest.raises(ValueError):
            TargetTables(r.references, r.lengths, None)
        with pytest.raises(ValueError):
            r.build_tables(None)


def test_records_with_cigar_sequence_and_tags(tmp_path):
    """Real BAM records carry CIGAR, packed sequence, qualities and tags after the read name: the
    emitter must hop over them by block_size and still read the fixed-offset fields."""
    import struct
    rng = np.random.default_rng(31)
    payload = [bam_io.bam_header_bytes(REFS)]
    want_rg, want_tid, group, last = [], [], -1, None
    for i in range(700):
        name = ("frag%04d" % (i // 3)).encode() + b"\x00"
        n_cig, l_seq = int(rng.integers(0, 4)), int(rng.integers(0, 200))
        tid, flag = int(rng.integers(0, len(REFS))), int(rng.choice([0, 16, 4, 256]))
        tail = (rng.integers(0, 256, 4 * n_cig + (l_seq + 1) // 2 + l_seq + int(rng.integers(0, 40)), dtype=np.uint8)
                .tobytes())
        core = struct.pack("<iiBBHHHiiii", tid, int(rng.integers(0, 1000)), len(name), 30, 4680, n_cig, flag, l_seq,
                           -1, -1, 0) + name + tail
        payload.append(struct.pack("<i", len(core)) + core)
        if not flag & 4:
            if name != last:
                group, last = group + 1, name
            want_rg.append(group)
            want_tid.append(tid)
    raw = b"".join(payload)
    path = str(tmp_path / "full.bam")
    with open(path, "wb") as fh:
        for off in range(0, len(raw), 777):                     # blocks cut records anywhere
            fh.write(bam_io.bgzf_block(raw[off:off + 777]))
        fh.write(bam_io.BGZF_EOF)
    cols = _same_single(path)                                   # native == Python emitter
    tables = TargetTables([r[0] for r in REFS], [r[1] for r in REFS], None)
    assert cols["read_group"].tolist() == want_rg
    assert np.array_equal(cols["target_idx"], tables.tid_target[np.array(want_tid)])
    assert np.array_equal(cols["hap_idx"], tables.tid_hap[np.array(want_tid)])


def test_parallel_record_hop_rejects_decoys(tmp_path, monkeypatch):
    """The record boundaries of a window are found speculatively in parallel (bamcols.cpp:find_records): a
    worker guesses the first record of its byte segment from two plausible record headers in a row.  Here
    the tag area of every third record holds byte-exact copies of two small records - a guess that lands on
    them is wrong and must be thrown out by the join with the verified chain - and tiny segments
    (BAMCOLS_GRAIN) put many segment starts right in front of them.  A record with block_size < 32 on the
    true chain must still be reported."""
    import struct
    rng = np.random.default_rng(77)

    def record(name, tid, flag, tail=b""):
        nm = name.encode() + b"\x00"
        core = struct.pack("<iiBBHHHiiii", tid, 7, len(nm), 30, 4680, 0, flag, 0, -1, -1, 0) + nm + tail
        return struct.pack("<i", len(core)) + core

    decoy = record("decoyA", 1, 0) + record("decoyB", 2, 0)
    for grain in (1, 2, 7, 4096):
        monkeypatch.setenv("BAMCOLS_GRAIN", str(grain))
        monkeypatch.setenv("BAMCOLS_BATCH_BLOCKS", str(1 + grain % 3))    # many small windows
        payload, want_rg, want_tid, group, last = [bam_io.bam_header_bytes(REFS)], [], [], -1, None
        for i in range(900):
            name = "frag%04d" % (i // 2)
            tid = int(rng.integers(0, len(REFS)))
            filler = rng.integers(0, 256, int(rng.integers(0, 90)), dtype=np.uint8).tobytes()
            tail = filler
            if i % 3 == 0:       # decoys that lead back onto the true chain / that lead into random bytes
                tail = filler + decoy + decoy if i % 2 else filler + decoy + rng.integers(0, 256, 60, dtype=np.uint8).tobytes()
            payload.append(record(name, tid, 0, tail))
            if name != last:
                group, last = group + 1, name
            want_rg.append(group)
            want_tid.append(tid)
        raw = b"".join(payload)
        path = str(tmp_path / ("decoy%d.bam" % grain))
        with open(path, "wb") as fh:
            for off in range(0, len(raw), 3000):
                fh.write(bam_io.bgzf_block(raw[off:off + 3000]))
            fh.write(bam_io.BGZF_EOF)
        for threads in (1, 3, 8):
            cols = _same_single(path, n_threads=threads)
            assert cols["read_group"].tolist() == want_rg
            tables = TargetTables([r[0] for r in REFS], [r[1] for r in REFS], None)
            assert np.array_equal(cols["target_idx"], tables.tid_target[np.array(want_tid)])
    # a broken record on the true chain
    raw = bam_io.bam_header_bytes(REFS) + b"".join(record("r%03d" % i, 0, 0) for i in range(200)) + struct.pack("<i", 5) + b"x" * 64
    path = str(tmp_path / "broken.bam")
    with open(path, "wb") as fh:
        fh.write(bam_io.bgzf_block(raw))
        fh.write(bam_io.BGZF_EOF)
    monkeypatch.setenv("BAMCOLS_GRAIN", "3")
    tables = TargetTables([r[0] for r in REFS], [r[1] for r in REFS], None)
    with bamcols.BamColumnReader(path, n_threads=4) as r:
        r.set_tables(tables)
        with pytest.raises(Exception) as err:
            r.read_all()
    assert "block_size" in str(err.value)


def _multisample_both(path, tables, cell_ids, cells, **reader_kw):
    header, recs = load_records(path)
    want = emitter.emit_multisample(recs, tables, cell_ids)
    with bamcols.BamColumnReader(path, **reader_kw) as r:
        r.set_tables(tables)
        got = r.read_all(cells=cells, chunk=257)
    for k, w in (("read_group", want.read_group), ("target_idx", want.target_idx), ("hap_idx", want.hap_idx),
                 ("cell_idx", want.cell_idx)):
        assert np.array_equal(got[k], w), k
    assert cells.names() == [n for n, _ in sorted(cell_ids.items(), key=lambda kv: kv[1])]


def test_randomised_per_cell_bams(tmp_path, monkeypatch):
    """The parallel per-cell window code against the record-level Python emitter: names with blanks
    (every alignment its own read), filtered records between reads, reads that end a file alone, several
    files sharing one cell dictionary, tiny BGZF blocks, forced thread splits and window sizes."""
    rng = np.random.default_rng(123)
    flags = [0, 0, 0, 16, 4, 1 | 2 | 128, 1 | 2 | 64]
    tables = TargetTables([r[0] for r in REFS], [r[1] for r in REFS], None)
    for case in range(40):
        monkeypatch.setenv("BAMCOLS_GRAIN", str(int(rng.choice([1, 3, 64, 4096]))))
        monkeypatch.setenv("BAMCOLS_BATCH_BLOCKS", str(int(rng.choice([1, 2, 7, 2048]))))   # windows of a few records
        cell_ids, cells = {}, bamcols.CellDictionary()
        for f in range(int(rng.integers(1, 4))):
            alns = []
            for read in range(int(rng.integers(1, 300))):
                cell = "CELL%03d" % int(rng.integers(0, 12))
                extra = " x y" if rng.random() < 0.15 else ""
                lead = " " if rng.random() < 0.03 else ""
                name = lead + _cell_name("f%dq%04d" % (f, read), cell, extra)
                for _ in range(int(rng.integers(1, 5))):
                    tid = int(rng.integers(0, len(REFS)))
                    alns.append((name, int(rng.choice(flags)), tid, 5, tid, 9))
            path = _write(tmp_path, alns, "c%d_%d.bam" % (case, f), block_payload=int(rng.choice([90, 400, 60000])))
            _multisample_both(path, tables, cell_ids, cells, n_threads=int(rng.choice([1, 2, 5])))


def test_per_cell_short_name_raises_where_the_python_statement_does(tmp_path, monkeypatch):
    """A short name raises only when a later valid alignment exists, as in the record-level Python emitter;
    with every record on its own worker thread and with the window unsplit."""
    ok = [(_cell_name("a", "C1"), 0, 0), (_cell_name("a", "C1"), 0, 1), (_cell_name("b", "C2"), 0, 2)]
    tail_bad = ok + [("short|||name", 0, 3)]                      # ends the file alone: never looked up
    mid_bad = ok + [("short|||name", 0, 3), (_cell_name("c", "C3"), 0, 4)]
    tables = TargetTables([r[0] for r in REFS], [r[1] for r in REFS], None)
    for grain in (1, 4096):
        monkeypatch.setenv("BAMCOLS_GRAIN", str(grain))
        for name, alns in (("ok", ok), ("tail", tail_bad)):
            _multisample_both(_write(tmp_path, alns, name + ".bam"), tables, {}, bamcols.CellDictionary(), n_threads=4)
        path = _write(tmp_path, mid_bad, "mid.bam")
        header, recs = load_records(path)
        with pytest.raises(IndexError):
            emitter.emit_multisample(recs, tables, {})
        with bamcols.BamColumnReader(path, n_threads=4) as r:
            r.set_tables(tables)
            with pytest.raises(IndexError):
                r.read_all(cells=bamcols.CellDictionary())


def test_native_target_section_equals_the_python_one(tmp_path):
    """The EC file's targets section built by libbamcols (convert() writes it without creating a Python string
    per target) against bin_utils._target_section on the same tables; non-ASCII names are declined (the
    reference writes their length in characters) and the caller falls back to the name list."""
    from alntools_b200 import bin_utils
    refs = [("t1_A", 10), ("t1_B", 11), ("t2", 5), ("_x", 7), ("longer_name_here_C", 99), ("t3_A", 1)]
    path = str(tmp_path / "sec.bam")
    bam_io.write_bam(path, refs, [("r1", 0, 0, 0, -1, -1), ("r2", 0, 2, 0, -1, -1)])
    with bamcols.BamColumnReader(path) as r:
        t = r.build_tables(None)
        got = t.target_section()
        names = list(t.main_targets.keys())
        want = bin_utils._target_section(names, np.asarray(t.lengths).astype(int), len(t.haplotypes))
        assert got == want
    path2 = str(tmp_path / "uni.bam")
    bam_io.write_bam(path2, [("tr\u00e4_A", 3), ("t2_A", 4)], [("r1", 0, 0, 0, -1, -1)])
    with bamcols.BamColumnReader(path2) as r:
        t = r.build_tables(None)
        assert t.target_section() is None
        assert list(t.main_targets.keys()) == ["tr\u00e4", "t2"]


class _StubBuilder(object):
    """Stands in for EcBuilder: collects what stream_single / stream_files push (host logic only, no GPU)."""

    def __init__(self, fail_at=None):
        self.parts, self.bases, self.drops, self.fail_at = [], [], [], fail_at

    def push(self, rg, tg, hp, cell=None, order_base=0, n=None, drop_last_group=False):
        if self.fail_at is not None and len(self.parts) >= self.fail_at:
            raise RuntimeError("push failed")
        self.parts.append([np.array(x[:n]) for x in (rg, tg, hp) + (() if cell is None else (cell,))])
        self.bases.append(order_base)
        self.drops.append(drop_last_group)


def test_stream_single_pipeline(tmp_path):
    """emitter.stream_single: the pieces it pushes add up to the file; a read longer than the buffers makes
    them grow (as read_all does) instead of failing; when the consumer fails the decode thread has left the
    native library before the exception reaches the caller, so closing the reader is safe."""
    import threading
    rng = np.random.default_rng(12)
    alns = []
    for read in range(2000):
        k = 40 if read == 700 else int(rng.integers(1, 5))
        for _ in range(k):
            alns.append(("read%05d" % read, 0, int(rng.integers(0, len(REFS)))))
    path = _write(tmp_path, alns)
    want, _ = _python_single(path)
    for rows in (1 << 16, 64, 16):                                  # 16 < the 40-alignment read: buffers grow
        with bamcols.BamColumnReader(path) as r:
            r.set_tables(TargetTables(r.references, r.lengths, None))
            stub = _StubBuilder()
            n = emitter.stream_single(r, stub, chunk_rows=rows, pinned=False)
        assert n == len(want.read_group)
        assert stub.bases == list(np.cumsum([0] + [len(p[0]) for p in stub.parts[:-1]]))
        assert np.array_equal(np.concatenate([p[1] for p in stub.parts]), want.target_idx)
        assert np.array_equal(np.concatenate([p[2] for p in stub.parts]), want.hap_idx)
        starts = np.concatenate([p[0][1:] != p[0][:-1] for p in stub.parts if len(p[0]) > 1])
        assert int(starts.sum()) + len(stub.parts) == want.n_groups   # no read is split between pushes
    before = threading.active_count()
    with bamcols.BamColumnReader(path) as r:
        r.set_tables(TargetTables(r.references, r.lengths, None))
        with pytest.raises(RuntimeError, match="push failed"):
            emitter.stream_single(r, _StubBuilder(fail_at=3), chunk_rows=64, pinned=False)
        assert threading.active_count() == before                   # the producer was joined


def test_stream_files_pipeline(tmp_path):
    """emitter.stream_files, the per-cell decode-ahead: one push per file, in order, with drop_last_group and order
    keys from order_base on, equal to decoding the files one after another, and the ranges merged over the files.
    When the consumer fails, or a file cannot be read in the decode thread, the error reaches the caller once that
    thread has been joined."""
    import threading
    from alntools_b200 import bam_utils_multisample
    case = max(golden_cases("multisample"), key=lambda c: len(c["file_order"]))
    files = [os.path.join(GOLDEN, case["dir"], fn) for fn in case["file_order"]] * 2   # more files than the ring holds
    tables, _, _ = bam_utils_multisample._tables(files[0], None, False)
    want, lo, hi = [], None, None
    ref_cells = bamcols.CellDictionary()
    for path in files:
        with bamcols.BamColumnReader(path) as r:
            r.set_tables(tables)
            r.track_ranges(True)
            want.append(r.read_all(cells=ref_cells))
            l, h = r.ranges()
        lo, hi = (l, h) if lo is None else (np.minimum(lo, l), np.maximum(hi, h))
    ref_cells.close()
    stub, cells = _StubBuilder(), bamcols.CellDictionary()
    n, ranges = emitter.stream_files(files, tables, cells, stub, order_base=3 << 40, track_ranges=True)
    cells.close()
    sizes = [len(w["read_group"]) for w in want]
    assert n == sum(sizes) and stub.drops == [True] * len(files)
    assert stub.bases == [(3 << 40) + int(s) for s in np.cumsum([0] + sizes[:-1])]
    for got, w in zip(stub.parts, want):
        for g, key in zip(got, ("read_group", "target_idx", "hap_idx", "cell_idx")):
            assert np.array_equal(g, w[key])
    assert np.array_equal(ranges[0], lo) and np.array_equal(ranges[1], hi)
    assert emitter.stream_files([], tables, None, stub) == (0, None)
    before = threading.active_count()
    missing = str(tmp_path / "missing.bam")
    for paths, builder, err in ((files, _StubBuilder(fail_at=1), RuntimeError),
                                (files[:1] + [missing] + files[1:], _StubBuilder(), OSError)):
        cells = bamcols.CellDictionary()
        with pytest.raises(err):
            emitter.stream_files(paths, tables, cells, builder)
        assert threading.active_count() == before               # the decode thread was joined
        cells.close()


@pytest.mark.parametrize("payload,n_shards", [(300, 2), (300, 5), (4000, 3), (60000, 4), (70, 7)])
def test_shards_of_one_file_add_up_to_the_file(tmp_path, payload, n_shards):
    """bamcols_plan_shards / bamcols_set_range (SURVEY 8f N3: chunks as virtual offsets, no temporary BAMs): the
    shards are contiguous, start at read boundaries, and their columns concatenated are the file's columns -
    with records that straddle BGZF blocks (tiny payloads), reads of many alignments around the cuts, names
    with blanks, filtered records, and more shards than the file can feed."""
    rng = np.random.default_rng(payload + n_shards)
    alns = []
    for read in range(1500):
        k = 60 if read % 400 == 7 else int(rng.integers(1, 6))
        name = "read%05d" % read + (" tail words" if read % 5 == 0 else "")
        for _ in range(k):
            flag = int(rng.choice([0, 16, 4, 1 | 2 | 64, 1 | 2 | 128]))
            alns.append((name, flag, int(rng.integers(0, len(REFS)))))
    path = _write(tmp_path, alns, block_payload=payload)
    want, _ = _python_single(path)
    with bamcols.BamColumnReader(path) as r:
        plan = r.plan_shards(n_shards)
        whole_all = None
    assert len(plan) == n_shards + 1 and plan[-1] == -1 and plan[0] > 0
    starts = [v for v in plan[:-1] if v >= 0]
    assert starts == sorted(starts)
    parts, seen_records = [], 0
    for k in range(n_shards):
        with bamcols.BamColumnReader(path) as r:
            r.set_tables(TargetTables(r.references, r.lengths, None))
            assert r.plan_shards(n_shards) == plan                  # the plan depends on the file only
            r.set_range(plan[k], plan[k + 1])
            cols = r.read_all(chunk=1 << 12)
            seen_records += r.all_alignments
            parts.append(cols)
    assert seen_records == want.all_alignments
    tg = np.concatenate([p["target_idx"] for p in parts])
    hp = np.concatenate([p["hap_idx"] for p in parts])
    assert np.array_equal(tg, want.target_idx) and np.array_equal(hp, want.hap_idx)
    # read boundaries: inside a shard as in the file, and every non-empty shard begins a new read
    heads = np.concatenate([np.concatenate(([True], p["read_group"][1:] != p["read_group"][:-1])) if len(p["read_group"]) else
                            np.zeros(0, dtype=bool) for p in parts])
    want_heads = np.concatenate(([True], want.read_group[1:] != want.read_group[:-1]))
    assert np.array_equal(heads, want_heads)
    if payload >= 4000 and n_shards <= 4:
        assert sum(1 for p in parts if len(p["read_group"])) >= 2   # the work really is split
