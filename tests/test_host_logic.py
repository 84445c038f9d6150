"""Host logic without a GPU: header tables, the column emitter and the EC writer.  The emitter's
columns are pushed through the ORACLE's column-level EC build (the contract the CUDA kernels
implement) and the bytes must equal what the reference wrote."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_records
from alntools_b200 import bin_utils, emitter, utils
from alntools_b200.header import TargetTables
from oracle import ec_oracle


@pytest.mark.parametrize("case", golden_cases("single"), ids=lambda c: c["name"])
def test_emitter_columns_reproduce_reference_single(case, tmp_path):
    header, recs = load_records(os.path.join(GOLDEN, case["bam"]))
    tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
    tables = TargetTables(header.references, header.lengths, tfile)
    cols = emitter.emit_single(recs, tables)
    indptr, indices, data, counts = ec_oracle.ec_from_columns(cols.read_group, cols.target_idx, cols.hap_idx)
    out = str(tmp_path / "out.bin")
    bin_utils.ecsave2_arrays(out, tables.haplotypes, list(tables.main_targets), tables.lengths, [case["bam"]],
                             (indptr, indices, data), ec_oracle.n_matrix_single(counts))
    with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
        assert a.read() == b.read()


@pytest.mark.parametrize("case", golden_cases("multisample"), ids=lambda c: c["name"])
def test_emitter_columns_reproduce_reference_multisample(case, tmp_path):
    tables = None
    cell_ids = {}
    pushes = []
    for fn in case["file_order"]:
        header, recs = load_records(os.path.join(GOLDEN, case["dir"], fn))
        if tables is None:
            tables = TargetTables(header.references, header.lengths, None)
        cols = emitter.emit_multisample(recs, tables, cell_ids)
        pushes.append((cols.read_group, cols.target_idx, cols.hap_idx, cols.cell_idx, True))
    res = ec_oracle.ec_from_columns_cells(pushes, case["mincount"])
    names = {v: k for k, v in cell_ids.items()}
    out = str(tmp_path / "out.bin")
    bin_utils.ecsave2_arrays(out, tables.haplotypes, list(tables.main_targets), tables.lengths,
                             [names[c] for c in res["cell_order"].tolist()],
                             (res["a_indptr"], res["a_indices"], res["a_data"]),
                             (res["n_indptr"], res["n_indices"], res["n_data"]))
    with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
        assert a.read() == b.read()


def test_header_tables_quirks():
    refs = ["G1_A", "G1_B", "G2", "_G3", "G5_x_A"]
    t = TargetTables(refs, [1, 2, 3, 4, 5])
    assert t.haplotypes == ["", "A", "B"]                      # '' sorts first (bam_utils.py:602)
    assert list(t.main_targets) == ["G1", "G2", "_G3", "G5_x"]  # split at the LAST '_', not at index 0
    assert t.tid_target.tolist() == [0, 0, 1, 2, 3]
    assert t.tid_hap.tolist() == [1, 2, 0, 0, 1]
    assert t.lengths[0].tolist() == [0, 1, 2]


def test_header_tables_reject_ambiguous_names():
    with pytest.raises(ValueError):
        TargetTables(["a", "a_"], [1, 1])


def test_emitter_filters_and_trimming():
    t = TargetTables(["T_A", "T_B"], [1, 1])
    P, PP, R2, UN = 1, 2, 0x80, 4
    recs = [("r1 x", 0, 0, 0, -1, -1), ("r1", 0, 1, 0, -1, -1), ("r2", UN, -1, 0, -1, -1),
            ("r2", P | PP, 0, 0, 0, 5), ("r2", P | PP | R2, 0, 0, 0, 5), ("r2", P, 1, 0, 1, 5),
            ("r2", P | PP, 1, 0, 0, 5), ("r2", P | PP, 1, 0, 1, -1), (" r3", 0, 1, 0, -1, -1)]
    cols = emitter.emit_single(recs, t)
    assert cols.all_alignments == 9 and cols.valid_alignments == 4
    assert cols.read_group.tolist() == [0, 0, 1, 2]
    assert cols.hap_idx.tolist() == [0, 1, 0, 1]


def test_multisample_emitter_needs_15_fields():
    t = TargetTables(["T_A"], [1])
    with pytest.raises(IndexError):
        emitter.emit_multisample([("plainname", 0, 0, 0, -1, -1)], t, {})


def test_ec_file_round_trip(tmp_path):
    out = str(tmp_path / "x.bin")
    a = (np.array([0, 1, 3], np.int32), np.array([0, 0, 2], np.int32), np.array([3, 1, 2], np.int32))
    n = (np.array([0, 2], np.int32), np.array([0, 1], np.int32), np.array([7, 9], np.int32))
    bin_utils.ecsave2_arrays(out, ["A", "B"], ["t0", "t1", "t2"], np.arange(6).reshape(3, 2), ["s"], a, n)
    back = bin_utils.ecload_arrays(out)
    assert back["haplotypes"] == ["A", "B"] and back["targets"] == ["t0", "t1", "t2"] and back["samples"] == ["s"]
    for x, y in zip(back["a"] + back["n"], a + n):
        assert np.array_equal(x, y)


def test_partition_matches_reference_semantics():
    assert utils.partition(list(range(7)), 3) == [[0, 1, 2], [3, 4], [5, 6]]
    assert utils.partition(list(range(2)), 4) == [[0], [1]]


def test_shard_bounds_never_split_a_read():
    from alntools_b200 import multi_gpu
    rg = np.repeat(np.arange(50), np.random.default_rng(0).integers(1, 9, 50)).astype(np.int32)
    for world in (1, 2, 3, 8, 64):
        cuts = multi_gpu.shard_bounds(rg, world)
        assert cuts[0] == 0 and cuts[-1] == len(rg) and len(cuts) == world + 1
        assert all(b >= a for a, b in zip(cuts[:-1], cuts[1:]))
        for c in cuts[1:-1]:
            assert c == len(rg) or c == 0 or rg[c] != rg[c - 1]


class _StubBuilder(object):
    """Stands in for the GPU builder: accepts every push and returns fixed, well-formed result arrays, so that
    the host side of convert() (decode, tables, file writing) can run on a machine without a GPU."""

    def __init__(self, *a, **k):
        self.rows = 0

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def push(self, rg, tg, hp, cell=None, order_base=0, drop_last_group=False, n=None):
        self.rows += int(n) if n is not None else len(rg)

    def finalize(self, min_cell_count=0, copy=True):
        i32 = lambda *v: np.array(v, dtype=np.int32)
        return {"n_ec": 2, "n_reads": 3, "n_samples": 2, "a_indptr": i32(0, 1, 3), "a_indices": i32(0, 0, 1),
                "a_data": i32(1, 3, 1), "n_indptr": i32(0, 1, 2), "n_indices": i32(0, 1), "n_data": i32(2, 1),
                "cell_order": i32(0, 1)}


def test_convert_writes_the_same_file_with_native_and_python_target_sections(tmp_path, monkeypatch):
    """convert() / convert_files() write the EC file's targets block from libbamcols when the tables are native;
    the bytes must equal what the Python writer produces from the name list (stub builder: no GPU needed)."""
    from conftest import GOLDEN, golden_cases
    from alntools_b200 import bam_utils, bam_utils_multisample, bamcols
    monkeypatch.setattr(bam_utils, "EcBuilder", _StubBuilder)
    monkeypatch.setattr(bam_utils_multisample, "EcBuilder", _StubBuilder)
    real_build = bamcols.BamColumnReader.build_tables

    def build_without_section(self, target_filename=None):
        t = real_build(self, target_filename)
        t.target_section = lambda: None
        return t

    outputs = {}
    for mode in ("native", "python"):
        if mode == "python":
            monkeypatch.setattr(bamcols.BamColumnReader, "build_tables", build_without_section)
        case = golden_cases("single")[0]
        out = str(tmp_path / ("single_%s.bin" % mode))
        tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
        bam_utils.convert(os.path.join(GOLDEN, case["bam"]), out, None, num_chunks=1, number_processes=1,
                          target_filename=tfile)
        mcase = golden_cases("multisample")[0]
        mout = str(tmp_path / ("multi_%s.bin" % mode))
        files = [os.path.join(GOLDEN, mcase["dir"], fn) for fn in mcase["file_order"]]
        bam_utils_multisample.convert_files(files, mout, None, mcase["mincount"])
        outputs[mode] = (open(out, "rb").read(), open(mout, "rb").read())
    assert outputs["native"][0] == outputs["python"][0]
    assert outputs["native"][1] == outputs["python"][1]
    assert len(outputs["native"][0]) > 60 and len(outputs["native"][1]) > 60


@pytest.mark.parametrize("emitter_mode", ["native", "python"])
def test_convert_files_without_files_raises(tmp_path, monkeypatch, emitter_mode):
    """convert_files([]) has no file to take the target tables from: it raises ValueError at once, with either
    emitter, instead of waiting for tables that never come."""
    import threading
    from alntools_b200 import bam_utils_multisample
    monkeypatch.setenv("ALNTOOLS_B200_EMITTER", emitter_mode)
    outcome = []

    def run():
        try:
            bam_utils_multisample.convert_files([], str(tmp_path / "x.bin"), None, 1)
        except Exception as exc:     # noqa: BLE001 - checked below
            outcome.append(exc)

    worker = threading.Thread(target=run, daemon=True)
    worker.start()
    worker.join(1.0)
    assert not worker.is_alive(), "convert_files([]) did not return within a second"
    assert len(outcome) == 1 and isinstance(outcome[0], ValueError), outcome
    assert not os.path.exists(str(tmp_path / "x.bin"))


def test_sliced_ec_file_writer_reproduces_the_golden_bytes(tmp_path):
    """bin_utils.ecsave2_slice: the EC file written in EC-id ranges by several writers (what the ranks of the
    multi-GPU convert do) is the file ecsave2 writes, for 1, 2, 3 and 5 writers, empty slices included."""
    import json
    from conftest import GOLDEN
    from alntools_b200 import bin_utils
    with open(os.path.join(GOLDEN, "manifest.json")) as fh:
        cases = [c for c in json.load(fh) if c["kind"] == "single"]
    for case in cases:
        src = os.path.join(GOLDEN, case["ec"])
        ec = bin_utils.ecload_arrays(src)
        header = bin_utils.ec_header_bytes(ec["haplotypes"], ec["targets"], ec["lengths"], ec["samples"])
        indptr, indices, data = ec["a"]
        counts = ec["n"][2]
        n_ec, nnz = len(counts), len(indices)
        for world in (1, 2, 3, 5, n_ec + 3):
            out = str(tmp_path / ("%s.%d.bin" % (case["name"], world)))
            per = (n_ec + world - 1) // world
            for r in range(world):
                a, b = min(n_ec, r * per), min(n_ec, (r + 1) * per)
                lo, hi = int(indptr[a]), int(indptr[b])
                bin_utils.ecsave2_slice(out, header, n_ec, nnz, a, lo, indptr[a:b + 1] - indptr[a], indices[lo:hi],
                                        data[lo:hi], counts[a:b], create=(r == 0))
            with open(out, "rb") as x, open(src, "rb") as y:
                assert x.read() == y.read(), (case["name"], world)


def test_multi_gpu_convert_fails_loudly_and_promptly_without_gpus(tmp_path):
    """convert(..., devices=2) starts one worker process per GPU.  Where the GPUs are missing the workers die at
    once; the call must report that (no CPU fallback) and must not leave a worker waiting for its peers."""
    import time
    import torch
    from alntools_b200 import bam_utils
    if torch.cuda.is_available() and torch.cuda.device_count() >= 2:
        pytest.skip("this machine has the GPUs; tests/multigpu_convert_check.py covers the working path")
    case = [c for c in golden_cases("single")][0]
    t0 = time.time()
    with pytest.raises(RuntimeError, match="multi-GPU bam2ec failed"):
        bam_utils.convert(os.path.join(GOLDEN, case["bam"]), str(tmp_path / "out.bin"), None, devices=2)
    assert time.time() - t0 < 120
    assert not os.path.exists(str(tmp_path / "out.bin"))
