"""Collation by read name, host side: the key rows of libbamcols (bamcols_emit_keys / BamColumnReader.emit_keys) against
the single-sample rows and the records themselves, the record-level statement emitter.emit_collated, and the
refusals of convert() that come before any file is opened."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_records
from alntools_b200 import bam_io, bamcols, emitter

REFS = [("T%d_%s" % (t, h), 100 + t) for t in range(6) for h in "AB"]
CAPACITIES = (1, 7, 4096, None)


class _Tables(object):
    """tid -> (target, haplotype) of REFS: tid = 2 * target + haplotype."""
    tid_target = np.arange(len(REFS), dtype=np.int32) // 2
    tid_hap = np.arange(len(REFS), dtype=np.int32) % 2


def _filters_file(path):
    """Filtered records, names with leading and inner blanks, 70-byte blocks."""
    rng = np.random.default_rng(5)
    names = ["r1", " r1", "r1 x", "r1 y", " lead", "in ner", "in ner2", "r2", "r2", "r3", " ", "  x"]
    alns = []
    for i in range(3000):
        name = names[int(rng.integers(0, len(names)))] if i % 7 else "q%04d" % (i // 5)
        flag = int(rng.choice([0, 0, 0, 4, 1 | 2, 1 | 2 | 0x80, 1, 16, 256]))
        tid = int(rng.integers(0, len(REFS)))
        ntid = tid if rng.random() < 0.8 else int(rng.integers(-1, len(REFS)))
        alns.append((name, flag, tid, int(rng.integers(0, 500)), ntid, int(rng.integers(-1, 300))))
    bam_io.write_bam(path, REFS, alns, block_payload=70)
    return path


def _lengths_file(path):
    """Names of 1 to 254 bytes (254 = the longest l_read_name allows with its NUL), some of them prefixes of others,
    each name used at two places of the file."""
    rng = np.random.default_rng(11)
    letters = np.frombuffer(b"ACGTacgt0123456789:_", dtype=np.uint8)
    base = bytes(letters[rng.integers(0, len(letters), 254)]).decode()
    names = [base[:k] for k in range(1, 255)] + [base[:k - 1] + "Z" for k in range(2, 255, 17)]
    order = list(range(len(names))) * 2
    rng.shuffle(order)
    alns = [(names[j], 0, int(rng.integers(0, len(REFS))), int(rng.integers(0, 900))) for j in order]
    bam_io.write_bam(path, REFS, alns, block_payload=4000)
    return path


@pytest.fixture(scope="module")
def files(built, tmp_path_factory):
    d = tmp_path_factory.mktemp("collate")
    golden = sorted({os.path.join(GOLDEN, c["bam"]) for c in golden_cases("single")})
    return golden + [_filters_file(str(d / "filters.bam")), _lengths_file(str(d / "lengths.bam"))]


def _keys(path, capacity):
    with bamcols.BamColumnReader(path) as r:
        r.build_tables(None)
        r.track_ranges(True)
        if capacity is None:
            cols = r.read_all_keys()
        else:
            parts = []
            while True:
                bufs = [np.empty(capacity, np.uint64), np.empty(capacity, np.uint64), np.empty(capacity, np.int32),
                        np.empty(capacity, np.int32)]
                n, done = r.emit_keys(*bufs)
                assert 0 <= n <= capacity
                parts.append([b[:n] for b in bufs])
                if done:
                    break
            cols = {k: np.concatenate([p[i] for p in parts]) for i, k in enumerate(("key_lo", "key_hi", "target_idx", "hap_idx"))}
        return cols, r.all_alignments, r.ranges()


def test_key_rows_match_the_single_sample_rows(files):
    for path in files:
        with bamcols.BamColumnReader(path) as r:
            r.build_tables(None)
            r.track_ranges(True)
            want = r.read_all()
            want_all, (want_lo, want_hi) = r.all_alignments, r.ranges()
        for cap in CAPACITIES:
            if cap == 1 and len(want["target_idx"]) > 50000:
                cap = 3
            got, all_alignments, (lo, hi) = _keys(path, cap)
            assert np.array_equal(got["target_idx"], want["target_idx"]), (path, cap)
            assert np.array_equal(got["hap_idx"], want["hap_idx"]), (path, cap)
            assert all_alignments == want_all, (path, cap)
            assert np.array_equal(lo, want_lo) and np.array_equal(hi, want_hi), (path, cap)


def test_keys_are_equal_exactly_when_trimmed_names_are(files):
    for path in files:
        _, records = load_records(path)
        names = [emitter._trim(q) for q, flag, tid, _p, ntid, npos in records if emitter._valid(flag, tid, ntid, npos)]
        got, _, _ = _keys(path, None)
        assert len(names) == len(got["key_lo"])
        keys = list(zip(got["key_lo"].tolist(), got["key_hi"].tolist()))
        assert all((lo & hi) != (1 << 64) - 1 for lo, hi in keys)
        by_name, by_key = {}, {}
        for name, key in zip(names, keys):
            assert by_name.setdefault(name, key) == key, (path, name)
            assert by_key.setdefault(key, name) == name, (path, name)


def _collated(records):
    return emitter.emit_collated(records, _Tables)


def test_emit_collated_hand_built_cases():
    c = _collated([("A", 0, 0, 0, -1, -1), ("A", 0, 1, 0, -1, -1), ("B", 0, 2, 0, -1, -1), ("A", 0, 3, 0, -1, -1)])
    assert c.read_group.tolist() == [0, 0, 0, 1] and c.n_groups == 2
    assert c.target_idx.tolist() == [0, 0, 1, 1] and c.hap_idx.tolist() == [0, 1, 1, 0]
    assert c.all_alignments == 4 and c.valid_alignments == 4
    # leading blanks keep the whole name; an inner blank cuts it
    c = _collated([(" x", 0, 0, 0, -1, -1), ("x", 0, 1, 0, -1, -1), ("x y", 0, 2, 0, -1, -1), (" x", 0, 3, 0, -1, -1)])
    assert c.read_group.tolist() == [0, 0, 1, 1] and c.target_idx.tolist() == [0, 1, 0, 1] and c.n_groups == 2
    # filtered records between the alignments of one read do not split it, and are counted
    c = _collated([("A", 0, 0, 0, -1, -1), ("A", 4, 1, 0, -1, -1), ("B", 1 | 2 | 0x80, 2, 0, 2, 0),
                   ("B", 0, 5, 0, -1, -1), ("A", 0, 4, 0, -1, -1)])
    assert c.read_group.tolist() == [0, 0, 1] and c.target_idx.tolist() == [0, 2, 2] and c.all_alignments == 5
    # one read
    c = _collated([("r", 0, t, 0, -1, -1) for t in (3, 1, 3, 0)])
    assert c.read_group.tolist() == [0] * 4 and c.n_groups == 1
    # every record its own read
    c = _collated([("r%d" % i, 0, i % 12, 0, -1, -1) for i in range(9)])
    assert c.read_group.tolist() == list(range(9)) and c.n_groups == 9
    # nothing valid
    c = _collated([("r", 4, 0, 0, -1, -1)])
    assert c.valid_alignments == 0 and c.n_groups == 0 and c.all_alignments == 1


def test_emit_collated_is_emit_single_of_the_regrouped_file(files):
    for path in files:
        header, records = load_records(path)
        tables = _Tables if len(header.references) == len(REFS) else None
        if tables is None:
            continue
        got = emitter.emit_collated(records, tables)
        first = {}
        for rec in records:
            if emitter._valid(rec[1], rec[2], rec[4], rec[5]):
                first.setdefault(emitter._trim(rec[0]), []).append(rec)
        want = emitter.emit_single([r for rs in first.values() for r in rs], tables)
        assert np.array_equal(got.read_group, want.read_group)
        assert np.array_equal(got.target_idx, want.target_idx) and np.array_equal(got.hap_idx, want.hap_idx)


def test_a_reader_does_not_switch_between_keys_and_read_groups(built):
    path = os.path.join(GOLDEN, "toy_single.bam")
    with bamcols.BamColumnReader(path) as r:
        r.build_tables(None)
        r.read_all_keys()
        with pytest.raises(ValueError, match="cannot switch"):
            r.read_all()
        with pytest.raises(ValueError, match="cannot switch"):
            r.read_all(cells=bamcols.CellDictionary())
    with bamcols.BamColumnReader(path) as r:
        r.build_tables(None)
        r.read_all(chunk=4)
        with pytest.raises(ValueError, match="cannot switch"):
            r.read_all_keys()


def test_collation_refuses_what_it_does_not_cover(tmp_path, monkeypatch):
    """These checks come before any file is opened or any GPU is touched."""
    from alntools_b200 import bam_utils, bam_utils_multisample
    missing = str(tmp_path / "missing.bam")
    with pytest.raises(NotImplementedError):
        bam_utils.convert(missing, None, None, devices=2, collate=True)
    with pytest.raises(NotImplementedError):
        bam_utils.convert(missing, None, None, decode="device", collate=True)
    with monkeypatch.context() as m:
        m.setenv("WORLD_SIZE", "2")
        m.setenv("RANK", "0")
        with pytest.raises(NotImplementedError):
            bam_utils.convert(missing, None, None, collate=True)
    with monkeypatch.context() as m:
        m.setenv("ALNTOOLS_B200_COLLATE", "1")
        with pytest.raises(NotImplementedError):
            bam_utils.convert(missing, None, None, devices=2)
        with pytest.raises(NotImplementedError):
            bam_utils.convert(missing, None, None, decode="device")
        with pytest.raises(NotImplementedError):
            bam_utils_multisample.convert_files([missing], None, None, 1)
        with pytest.raises(NotImplementedError):
            bam_utils_multisample.convert(str(tmp_path / "missing_dir"), None, None, 0, 1, 1, None, None, None)
    with monkeypatch.context() as m:
        m.setenv("ALNTOOLS_B200_COLLATE", "bogus")
        with pytest.raises(ValueError):
            bam_utils.convert(missing, None, None)
    assert emitter.collate_mode() is False
    monkeypatch.setenv("ALNTOOLS_B200_COLLATE", "0")
    assert emitter.collate_mode() is False and emitter.collate_mode(True) is True
