"""Several samples in one EC file (ecb_sample_close / ecb_finalize_samples, EcBuilder.close_sample /
finalize_samples, bam_utils.convert_samples).

Every result is compared byte for byte with tests/samples_oracle.py: the ECs, ids and A matrix of the concatenated
samples from the oracles, and each sample's counts as its column of N."""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
from alntools_b200 import bam_io, bam_utils, bin_utils, synth
import samples_oracle as so

pytestmark = pytest.mark.gpu

N_TARGETS, N_HAPS = 100_000, 2
DISTINCT = ["toy_single", "mixed_single", "synth_h2", "synth_h8_heavy", "range_single"]   # one per @SQ list


@pytest.fixture(scope="module")
def native(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")
    from alntools_b200 import _native
    _native.load_library()
    return _native


def _read(path):
    with open(path, "rb") as fh:
        return fh.read()


def _golden(name):
    return os.path.join(GOLDEN, next(c for c in golden_cases("single") if c["name"] == name)["bam"])


@pytest.fixture(scope="module")
def union(tmp_path_factory):
    """The distinct single-sample goldens on one header, and the same files shuffled (for collation)."""
    d = tmp_path_factory.mktemp("samples_union")
    paths = so.union_goldens([_golden(n) for n in DISTINCT], str(d))
    shuffled = []
    for i, p in enumerate(paths):
        header, records = so.load(p)
        perm = np.random.default_rng(i).permutation(len(records))
        q = str(d / ("s%d.bam" % i))
        bam_io.write_bam(q, list(zip(header.references, header.lengths)), [records[j] for j in perm],
                         block_payload=3000)
        shuffled.append(q)
    empty = str(d / "empty.bam")                       # no valid alignment: every record unmapped
    header, records = so.load(paths[0])
    bam_io.write_bam(empty, list(zip(header.references, header.lengths)),
                     [(q, 4, -1, 0, -1, -1) for q, *_ in records[:5]])
    return paths, shuffled, empty


def _names(paths):
    return ["sample_%d" % i for i in range(len(paths))]


def _convert(paths, out, **kw):
    ec = str(out / "got.bin")
    bam_utils.convert_samples(paths, ec, sample_names=_names(paths), **kw)
    return _read(ec)


# ---- files -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", golden_cases("single"), ids=lambda c: c["name"])
def test_one_sample_is_the_golden(case, native, tmp_path):
    bam = os.path.join(GOLDEN, case["bam"])
    targets = os.path.join(GOLDEN, case["targets"]) if case.get("targets") else None
    ec = str(tmp_path / "c.bin")
    rng = str(tmp_path / "c.range.txt") if case.get("range") else None
    bam_utils.convert_samples([bam], ec, target_filename=targets, range_filename=rng)
    assert hashlib.sha256(_read(ec)).hexdigest() == case["sha256"]
    if rng:
        assert _read(rng) == _read(os.path.join(GOLDEN, case["range"]))


@pytest.mark.parametrize("order", ["forward", "reversed"])
def test_goldens_as_samples(order, native, union, tmp_path):
    paths = union[0] if order == "forward" else union[0][::-1]
    assert _convert(paths, tmp_path) == so.ec_file_bytes(paths, _names(paths))


def test_concatenation_invariant_and_range_file(native, union, tmp_path):
    """A, the row sums of N and the range file are those of convert() of one BAM holding the files back to back."""
    paths = union[0]
    header, _ = so.load(paths[0])
    cat = str(tmp_path / "cat.bam")
    bam_io.write_bam(cat, list(zip(header.references, header.lengths)), [r for p in paths for r in so.load(p)[1]])
    rs, rc = str(tmp_path / "s.txt"), str(tmp_path / "c.txt")
    bam_utils.convert_samples(paths, str(tmp_path / "s.bin"), range_filename=rs)
    bam_utils.convert(cat, str(tmp_path / "c.bin"), None, range_filename=rc)
    assert _read(rs) == _read(rc)
    got, want = bin_utils.ecload_arrays(str(tmp_path / "s.bin")), bin_utils.ecload_arrays(str(tmp_path / "c.bin"))
    for a, b in zip(got["a"], want["a"]):
        assert np.array_equal(a, b)
    n_ec = len(got["a"][0]) - 1
    assert np.array_equal(np.bincount(got["n"][1], weights=got["n"][2], minlength=n_ec).astype(np.int64),
                          want["n"][2].astype(np.int64))
    assert got["samples"] == [os.path.basename(p) for p in paths]


@pytest.mark.parametrize("budget", [None, "400000"])   # 400 kB: files of more than a few thousand alignments spill
def test_collated_samples(budget, native, union, tmp_path, monkeypatch):
    if budget:
        monkeypatch.setenv("ALNTOOLS_B200_COLLATE_BUDGET", budget)
    paths = union[1]
    assert _convert(paths, tmp_path, collate=True) == so.ec_file_bytes(paths, _names(paths), collate=True)


def test_device_decode(native, union, tmp_path):
    paths = union[0]
    assert _convert(paths, tmp_path, decode="device") == so.ec_file_bytes(paths, _names(paths))


def test_python_emitter(native, union, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_EMITTER", "python")
    paths = union[0][:3]
    assert _convert(paths, tmp_path) == so.ec_file_bytes(paths, _names(paths))
    paths = union[1][:3]
    assert _convert(paths, tmp_path, collate=True) == so.ec_file_bytes(paths, _names(paths), collate=True)


@pytest.mark.parametrize("where", [0, 2, 5])
def test_sample_without_valid_alignment(where, native, union, tmp_path):
    paths = list(union[0])
    paths.insert(where, union[2])
    want = so.ec_file_bytes(paths, _names(paths))
    assert _convert(paths, tmp_path) == want
    got = bin_utils.ecload_arrays(str(tmp_path / "got.bin"))["n"][0]
    assert got[where] == got[where + 1]                # an empty column in its place


def test_only_empty_samples_raise(native, union, tmp_path):
    with pytest.raises(RuntimeError, match="three positive integers"):
        bam_utils.convert_samples([union[2], union[2]], str(tmp_path / "x.bin"))


def _columns_file(path, cols):
    synth.columns_to_bam(path, cols, N_TARGETS, N_HAPS)


def _check_file(ec_path, samples):
    got = bin_utils.ecload_arrays(ec_path)
    want = so.columns_result(samples)
    for a, b in zip(got["a"] + got["n"], want[:6]):
        assert np.array_equal(a, b)


def test_long_read_in_a_sample(native, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    rng = np.random.default_rng(5)
    a = synth.make_columns(20000, N_TARGETS, N_HAPS, 11, mode="diploid")
    lens = [3] * 500 + [40000] + [2] * 500          # one read of 40 000 alignments in the middle of the second file
    b = {"read_group": np.repeat(np.arange(len(lens)), lens).astype(np.int32),
         "target_idx": rng.integers(0, 3000, sum(lens)).astype(np.int32),
         "hap_idx": rng.integers(0, N_HAPS, sum(lens)).astype(np.int32)}
    paths = [str(tmp_path / "a.bam"), str(tmp_path / "b.bam")]
    _columns_file(paths[0], a)
    _columns_file(paths[1], b)
    ec = str(tmp_path / "x.bin")
    bam_utils.convert_samples(paths, ec)
    _check_file(ec, [[a], [b]])


# ---- the builder -----------------------------------------------------------------------------------------------
def _cols(n_reads, seed, mode="diploid"):
    return synth.make_columns(n_reads, N_TARGETS, N_HAPS, seed, mode=mode)


def _piece(cols, a, b):
    """Reads a..b of a column dict (read ids dense from 0)."""
    rg = cols["read_group"]
    lo, hi = np.searchsorted(rg, [a, b])
    return {k: cols[k][lo:hi] for k in ("read_group", "target_idx", "hap_idx")}


def _run(native, samples, **options):
    with native.EcBuilder(N_TARGETS, N_HAPS, **options) as b:
        nnz = []
        for pushes in samples:
            base = 0
            for p in pushes:
                b.push(p["read_group"], p["target_idx"], p["hap_idx"], order_base=base)
                base += len(p["read_group"])
            nnz.append(b.close_sample())
        res = b.finalize_samples()
        return res, nnz, b.stats()


def _same(res, want):
    keys = ("a_indptr", "a_indices", "a_data", "n_indptr", "n_indices", "n_data")
    for k, w in zip(keys, want[:6]):
        assert np.array_equal(res[k], w), k
    assert res["n_reads"] == want[6]


def test_several_pushes_per_sample_and_stats(native):
    c0, c1, c2 = _cols(60000, 1), _cols(50000, 2), _cols(40000, 3)
    samples = [[_piece(c0, 0, 20000), _piece(c0, 20000, 20001), _piece(c0, 20001, 60000)], [], [c1],
               [_piece(c2, 0, 1), _piece(c2, 1, 40000)], [_piece(c0, 0, 1)]]
    res, nnz, st = _run(native, samples)
    want = so.columns_result(samples)
    _same(res, want)
    assert nnz == list(np.diff(want[3]))
    assert res["n_samples"] == 5 and nnz[1] == 0 and nnz[4] == 1
    assert st["samples"] == 5 and st["sample_pairs"] == sum(nnz) and st["sample_ms"] > 0


def test_ec_first_seen_in_a_later_sample_and_equal_sets(native):
    a = {"read_group": np.array([0, 0, 1], np.int32), "target_idx": np.array([5, 6, 5], np.int32),
         "hap_idx": np.array([0, 1, 0], np.int32)}
    b = {"read_group": np.array([0, 1, 1, 2, 2], np.int32), "target_idx": np.array([9, 6, 5, 5, 6], np.int32),
         "hap_idx": np.array([1, 1, 0, 0, 1], np.int32)}
    res, nnz, _ = _run(native, [[a], [b], [a]])
    # ECs {5A, 6B}, {5A}, then {9B}: first seen in the second sample; the second sample's read {6B, 5A} is EC 0
    assert res["n_ec"] == 3 and nnz == [2, 2, 2]
    assert res["n_indptr"].tolist() == [0, 2, 4, 6]
    assert res["n_indices"].tolist() == [0, 1, 0, 2, 0, 1]
    assert res["n_data"].tolist() == [1, 1, 2, 1, 1, 1]
    _same(res, so.columns_result([[a], [b], [a]]))


def test_growth_and_replay_inside_a_sample(native):
    samples = [[_cols(20000, 4)], [_cols(300000, 5, mode="light")], [_cols(20000, 6)]]
    res, _, st = _run(native, samples, table_slots=1024)
    assert st["table_grows"] > 0 and st["overflow_reads"] > 0
    _same(res, so.columns_result(samples))


def test_long_read_with_max_read_zero(native):
    rng = np.random.default_rng(9)
    lens = [2] * 300 + [70000] + [4] * 300
    long = {"read_group": np.repeat(np.arange(len(lens)), lens).astype(np.int32),
            "target_idx": rng.integers(0, 5000, sum(lens)).astype(np.int32),
            "hap_idx": rng.integers(0, N_HAPS, sum(lens)).astype(np.int32)}
    samples = [[_cols(10000, 7)], [long], [_cols(10000, 8)]]
    res, _, st = _run(native, samples, max_read=0)
    _same(res, so.columns_result(samples))


def test_unclosed_push_is_refused(native):
    c = _cols(5000, 10)
    with native.EcBuilder(N_TARGETS, N_HAPS) as b:
        b.push(c["read_group"], c["target_idx"], c["hap_idx"])
        b.close_sample()
        b.push(c["read_group"], c["target_idx"], c["hap_idx"])
        with pytest.raises(native.EcbError, match="after the last ecb_sample_close") as err:
            b.finalize_samples()
        assert err.value.code == -1
        b.close_sample()
        _same(b.finalize_samples(), so.columns_result([[c], [c]]))
    with native.EcBuilder(N_TARGETS, N_HAPS, with_cells=True) as b:
        with pytest.raises(native.EcbError, match="single-sample"):
            b.close_sample()


def test_reset_and_reuse(native):
    s1 = [[_cols(30000, 12)], [_cols(30000, 13)]]
    s2 = [[_cols(20000, 14)], [], [_cols(25000, 15)]]
    with native.EcBuilder(N_TARGETS, N_HAPS) as b:
        for samples in (s1, s2, s1):
            for pushes in samples:
                for p in pushes:
                    b.push(p["read_group"], p["target_idx"], p["hap_idx"])
                b.close_sample()
            _same(b.finalize_samples(), so.columns_result(samples))
            b.reset()
            assert b.stats()["samples"] == 0


@pytest.mark.parametrize("where", ["pinned", "pageable", "device"])
def test_result_memory(where, native):
    import torch
    samples = [[_cols(40000, 16)], [_cols(40000, 17)], []]
    want = so.columns_result(samples)
    opts = {"pinned": {}, "pageable": {"pageable_results": 1}, "device": {"result_on_device": 1}}[where]
    with native.EcBuilder(N_TARGETS, N_HAPS, **opts) as b:
        for pushes in samples:
            for p in pushes:
                b.push(p["read_group"], p["target_idx"], p["hap_idx"])
            b.close_sample()
        if where != "device":
            _same(b.finalize_samples(), want)
            _same(b.finalize_samples(copy=False), want)       # a second finalize gives the same
            return
        r = b.finalize_samples_raw()
        dev = torch.device("cuda", 0)

        def view(p, n):
            return native._device_view(native.ctypes.cast(p, native.ctypes.c_void_p).value, (n,), "<i4",
                                       torch.int32, dev).cpu().numpy()
        got = {"a_indptr": view(r.a_indptr, r.n_ec + 1), "a_indices": view(r.a_indices, r.nnz_a),
               "a_data": view(r.a_data, r.nnz_a), "n_indptr": view(r.n_indptr, r.n_samples + 1),
               "n_indices": view(r.n_indices, r.nnz_n), "n_data": view(r.n_data, r.nnz_n), "n_reads": r.n_reads}
        _same(got, want)


def test_sixteen_files_of_a_million_reads(native):
    """16 cfg2-shaped samples (diploid, 100 000 targets) of 1 M reads each, against the C oracle."""
    samples = [[synth.make_columns(1_000_000, N_TARGETS, N_HAPS, 2000 + i, mode="diploid")] for i in range(16)]
    res, nnz, st = _run(native, samples)
    _same(res, so.columns_result(samples))
    assert st["samples"] == 16 and res["n_samples"] == 16
