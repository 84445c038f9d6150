"""Merging EC files on the GPU (ecb_push_ecs / ecb_sample_append, EcBuilder.push_ecs / append_samples,
bin_utils.merge_ec_files).

Outputs are compared by bytes, or array for array with the Python statement of the rule (tests/merge_oracle.py);
nothing is compared with a tolerance.  The properties: merging one file gives that file; merging the convert() outputs
of several BAM files gives what convert_samples writes for them; merging is associative."""
import glob
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
from alntools_b200 import bam_io, bam_utils, bin_utils, emitter, synth
import merge_oracle as mo
import samples_oracle as so

pytestmark = pytest.mark.gpu

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
    d = tmp_path_factory.mktemp("merge_union")
    paths = so.union_goldens([_golden(n) for n in DISTINCT], str(d))
    shuffled = []
    for i, p in enumerate(paths):
        header, records = so.load(p)
        perm = np.random.default_rng(i).permutation(len(records))
        q = str(d / ("s%d.bam" % i))
        bam_io.write_bam(q, list(zip(header.references, header.lengths)), [records[j] for j in perm],
                         block_payload=3000)
        shuffled.append(q)
    return paths, shuffled


def _convert_each(paths, out, **kw):
    ecs = []
    for i, p in enumerate(paths):
        ecs.append(str(out / ("c%d_%s.bin" % (i, os.path.basename(p)))))
        bam_utils.convert(p, ecs[-1], None, **kw)
    return ecs


def _merge(ins, out, name="m.bin", **kw):
    path = str(out / name)
    bin_utils.merge_ec_files(ins, path, **kw)
    return path


def _joint(paths, out, name="j.bin", **kw):
    path = str(out / name)
    bam_utils.convert_samples(paths, path, **kw)
    return path


def _same_arrays(got, want):
    for x, y in zip(got["a"] + got["n"], want["a"] + want["n"]):
        assert np.array_equal(np.asarray(x), np.asarray(y))


# ---- 1. merge([F]) == F ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "**", "*.bin"), recursive=True)),
                         ids=os.path.basename)
def test_one_file_is_itself(path, native, tmp_path):
    assert _read(_merge([path], tmp_path)) == _read(path)


# ---- 2. merge of convert() outputs == convert_samples ------------------------------------------------------------
@pytest.mark.parametrize("order", ["forward", "reversed"])
def test_merge_of_converts_is_convert_samples(order, native, union, tmp_path):
    paths = union[0] if order == "forward" else union[0][::-1]
    merged = _merge(_convert_each(paths, tmp_path), tmp_path)
    assert _read(merged) == _read(_joint(paths, tmp_path))


def test_merge_of_collated_converts_is_collated_convert_samples(native, union, tmp_path):
    paths = union[1]
    merged = _merge(_convert_each(paths, tmp_path, collate=True), tmp_path)
    assert _read(merged) == _read(_joint(paths, tmp_path, collate=True))


# ---- 3. associativity --------------------------------------------------------------------------------------------
def test_merging_is_associative(native, union, tmp_path):
    paths = union[0]
    c = _convert_each(paths, tmp_path)
    pair = _merge(c[:2], tmp_path, "pair.bin")
    assert _read(pair) == _read(_joint(paths[:2], tmp_path, "j2.bin"))
    triple = _merge(c[:3], tmp_path, "triple.bin")
    assert _read(_merge([pair, c[2]], tmp_path, "pair_then.bin")) == _read(triple)
    assert _read(_merge([c[0], _merge(c[1:3], tmp_path, "tail.bin")], tmp_path, "then_pair.bin")) == _read(triple)
    j12, j3 = _joint(paths[:2], tmp_path, "j12.bin"), _joint(paths[2:3], tmp_path, "j3.bin")
    assert _read(_merge([j12, j3], tmp_path, "jj.bin")) == _read(_joint(paths[:3], tmp_path, "j123.bin"))
    whole = _merge([_merge(c[:2], tmp_path, "a.bin"), _merge(c[2:4], tmp_path, "b.bin"), c[4]], tmp_path, "w.bin")
    assert _read(whole) == _read(_merge(c, tmp_path, "all.bin")) == _read(_joint(paths, tmp_path, "jall.bin"))


# ---- 4. random EC files against the statement --------------------------------------------------------------------
N_TARGETS, N_HAPS = 200_000, 31


def _pool(rng, short=3000, mid=20, long=2):
    """Distinct rows: many of 1 to 8 targets, some of 1000 to 5000, a few of 100 000; masks over all 31 bits."""
    sizes = ([int(x) for x in rng.integers(1, 9, size=short)] + [int(x) for x in rng.integers(1000, 5001, size=mid)]
             + [100_000] * long)
    rows = set()
    for k in sizes:
        t = np.sort(rng.choice(N_TARGETS, size=k, replace=False))
        m = rng.integers(1, 1 << N_HAPS, size=k)
        m[0] |= 1 << 30                                    # the highest haplotype bit is in use
        rows.add(tuple(zip(t.tolist(), m.tolist())))
    return sorted(rows, key=lambda r: (len(r), r))


def _random_files(seed, n_files=16, big_cols=1000):
    rng = np.random.default_rng(seed)
    pool = _pool(rng)
    files = []
    for k in range(n_files):
        n_rows = int(rng.integers(1, len(pool) // 3))
        n_cols = big_cols if k == 1 else int(rng.integers(1, 6))
        files.append(mo.random_file(rng, pool, n_rows, n_cols))
    return files


def _statement(files):
    rows, n = mo.merge_statement([(mo.rows_of(a), n) for a, n in files])
    return {"a": mo.a_csr(rows), "n": n}


def _write(path, a, n, n_samples):
    bin_utils.ecsave2_arrays(path, ["h%d" % h for h in range(N_HAPS)], ["t%d" % t for t in range(N_TARGETS)],
                             np.full((N_TARGETS, N_HAPS), 1000, np.int32), ["s%d" % s for s in range(n_samples)], a, n)


def test_random_files_through_merge_ec_files(native, tmp_path):
    files = _random_files(1)
    paths = []
    for k, (a, n) in enumerate(files):
        paths.append(str(tmp_path / ("r%d.bin" % k)))
        _write(paths[-1], a, n, len(n[0]) - 1)
    out = _merge(paths, tmp_path)
    _same_arrays(bin_utils.ecload_arrays(out), _statement(files))


@pytest.mark.parametrize("device_arrays", [False, True])
def test_random_files_with_table_growth(device_arrays, native, tmp_path):
    import torch
    files = _random_files(2)
    want = _statement(files)
    with native.EcBuilder(N_TARGETS, N_HAPS, table_slots=1024) as b:
        for a, n in files:
            if device_arrays:
                a = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in a]
                n = [torch.from_numpy(np.ascontiguousarray(x)).cuda() for x in n]
            b.push_ecs(*a)
            b.append_samples(*n)
        st = b.stats()
        got = b.finalize_samples()
    assert st["table_grows"] > 0
    assert st["ec_pushes"] == len(files) and st["ec_rows"] == sum(len(a[0]) - 1 for a, _ in files)
    assert st["ec_claimed"] == len(want["a"][0]) - 1 and st["samples"] == len(want["n"][0]) - 1
    _same_arrays({"a": (got["a_indptr"], got["a_indices"], got["a_data"]),
                  "n": (got["n_indptr"], got["n_indices"], got["n_data"])}, want)


# ---- 5. an EC-file row and a read with one set are one EC --------------------------------------------------------
def test_rows_and_reads_share_keys(native, union, tmp_path):
    b1, b2 = union[0][1], union[0][3]
    header, records = so.load(b1)
    tables = bam_utils.TargetTables(header.references, header.lengths, None)
    cols = emitter.emit_single(iter(records), tables)
    c2 = bin_utils.ecload_arrays(_convert_each([b2], tmp_path)[0])
    with native.EcBuilder(tables.num_targets, tables.num_haplotypes) as b:
        b.push(cols.read_group, cols.target_idx, cols.hap_idx)
        b.close_sample()
        b.push_ecs(*c2["a"])
        b.append_samples(*c2["n"])
        got = b.finalize_samples()
    want = bin_utils.ecload_arrays(_joint([b1, b2], tmp_path))
    _same_arrays({"a": (got["a_indptr"], got["a_indices"], got["a_data"]),
                  "n": (got["n_indptr"], got["n_indices"], got["n_data"])}, want)


# ---- 6. at size ------------------------------------------------------------------------------------------------
def test_at_size_merge_of_eight_converts(native, tmp_path):
    cols = synth.make_columns(8_000_000, 100_000, 2, 1002, mode="diploid")
    rg = cols["read_group"]
    n_reads = int(rg[-1]) + 1
    paths = []
    for i in range(8):
        lo, hi = np.searchsorted(rg, [n_reads * i // 8, n_reads * (i + 1) // 8])
        part = {k: np.ascontiguousarray(cols[k][lo:hi]) for k in ("read_group", "target_idx", "hap_idx")}
        paths.append(str(tmp_path / ("part%d.bam" % i)))
        synth.columns_to_bam(paths[-1], part, 100_000, 2)
    del cols
    merged = _merge(_convert_each(paths, tmp_path), tmp_path)
    joint = _joint(paths, tmp_path)
    assert hashlib.sha256(_read(merged)).hexdigest() == hashlib.sha256(_read(joint)).hexdigest()


# ---- 7. malformed input ------------------------------------------------------------------------------------------
GOOD_A = ([0, 2, 3], [1, 4, 2], [1, 3, 2])          # rows {(1, 1), (4, 3)} and {(2, 2)}
GOOD_N = ([0, 2], [0, 1], [5, 1])


def _arr(x):
    return np.asarray(x, dtype=np.int32)


BAD = [
    ("target", ([0, 2, 3], [1, 10, 2], [1, 3, 2]), GOOD_N, "target outside \\[0, 10\\) at entry 1 \\(row 0\\)"),
    ("negative_target", ([0, 1, 2], [-1, 2], [1, 1]), GOOD_N, "target outside \\[0, 10\\) at entry 0 \\(row 0\\)"),
    ("zero_mask", ([0, 2, 3], [1, 4, 2], [1, 0, 2]), GOOD_N, "haplotype mask .* at entry 1 \\(row 0\\)"),
    ("mask_bit", ([0, 2, 3], [1, 4, 2], [1, 3, 4]), GOOD_N, "haplotype mask .* at entry 2 \\(row 1\\)"),
    ("unsorted", ([0, 2, 3], [4, 1, 2], [1, 3, 2]), GOOD_N, "not strictly ascending at entry 1 \\(row 0\\)"),
    ("repeated_target", ([0, 2, 3], [1, 1, 2], [1, 3, 2]), GOOD_N, "not strictly ascending at entry 1"),
    ("empty_row", ([0, 2, 2, 3], [1, 4, 2], [1, 3, 2]), GOOD_N, "row 1 is empty"),
    ("decreasing", ([0, 2, 1, 3], [1, 4, 2], [1, 3, 2]), GOOD_N, "a_indptr decreases at 2"),
    ("duplicate", ([0, 1, 2, 3], [2, 1, 2], [2, 1, 2]), GOOD_N, "row [02] holds the set of another row"),
    ("n_index", GOOD_A, ([0, 2], [0, 2], [5, 1]), "EC index outside \\[0, 2\\) at entry 1"),
    ("n_count", GOOD_A, ([0, 2], [0, 1], [5, -1]), "negative count at entry 1"),
]


@pytest.mark.parametrize("kind,a,n,match", BAD, ids=[b[0] for b in BAD])
def test_malformed_rows_through_the_builder(kind, a, n, match, native):
    with native.EcBuilder(10, 2) as b:
        with pytest.raises(native.EcbError, match=match) as info:
            b.push_ecs(*map(_arr, a))
            b.append_samples(*map(_arr, n))
        assert info.value.code == native.ECB_ERR_FORMAT
        if kind == "duplicate":                              # the table changed: only a reset recovers
            with pytest.raises(native.EcbError, match="ecb_reset first"):
                b.push_ecs(*map(_arr, GOOD_A))
            b.reset()
        # the same builder merges a correct set afterwards, as the statement says
        files = [(tuple(map(_arr, GOOD_A)), tuple(map(_arr, GOOD_N))),
                 (tuple(map(_arr, ([0, 1, 3], [2, 1, 4], [2, 1, 3]))), tuple(map(_arr, ([0, 1, 2], [1, 0], [7, 2]))))]
        for fa, fn in files:
            b.push_ecs(*fa)
            b.append_samples(*fn)
        got = b.finalize_samples()
    _same_arrays({"a": (got["a_indptr"], got["a_indices"], got["a_data"]),
                  "n": (got["n_indptr"], got["n_indices"], got["n_data"])}, _statement(files))


@pytest.mark.parametrize("kind,a,n,match", BAD, ids=[b[0] for b in BAD])
def test_malformed_files_through_merge_ec_files(kind, a, n, match, native, tmp_path):
    good, bad = str(tmp_path / "good.bin"), str(tmp_path / ("bad_%s.bin" % kind))
    for path, (fa, fn) in ((good, (GOOD_A, GOOD_N)), (bad, (a, n))):
        bin_utils.ecsave2_arrays(path, ["A", "B"], ["t%d" % t for t in range(10)], np.ones((10, 2), np.int32), ["s"],
                                 tuple(map(_arr, fa)), tuple(map(_arr, fn)))
    out = str(tmp_path / "out.bin")
    with pytest.raises(ValueError, match="bad_%s.bin: .*%s" % (kind, match)):
        bin_utils.merge_ec_files([good, bad], out)
    assert not os.path.exists(out)


# ---- 8. state ----------------------------------------------------------------------------------------------------
def test_state_refusals(native):
    with native.EcBuilder(10, 2) as b:
        b.push_ecs(*map(_arr, GOOD_A))
        with pytest.raises(native.EcbError, match="await ecb_sample_append") as info:
            b.finalize_samples()
        assert info.value.code == -1
        with pytest.raises(native.EcbError, match="await ecb_sample_append") as info:
            b.push(_arr([0]), _arr([1]), _arr([0]))
        assert info.value.code == native.ECB_ERR_STATE
        with pytest.raises(native.EcbError, match="await ecb_sample_append"):
            b.close_sample()
        assert b.append_samples(*map(_arr, GOOD_N)) == 2
        with pytest.raises(native.EcbError, match="carry no reads") as info:
            b.finalize()
        assert info.value.code == native.ECB_ERR_STATE
        with pytest.raises(native.EcbError, match="no EC rows await"):
            b.append_samples(*map(_arr, GOOD_N))
        got = b.finalize_samples()
        assert got["n_ec"] == 2 and got["n_indices"].tolist() == [0, 1] and got["n_data"].tolist() == [5, 1]
        b.reset()
        b.push(_arr([0, 0, 1]), _arr([1, 4, 2]), _arr([0, 1, 1]))
        with pytest.raises(native.EcbError, match="close that sample first") as info:
            b.push_ecs(*map(_arr, GOOD_A))
        assert info.value.code == native.ECB_ERR_STATE
        assert b.finalize()["n_ec"] == 2                     # after a reset the context counts reads again
    with native.EcBuilder(10, 2, with_cells=True) as b:
        with pytest.raises(native.EcbError, match="single-sample contexts only") as info:
            b.push_ecs(*map(_arr, GOOD_A))
        assert info.value.code == -1
