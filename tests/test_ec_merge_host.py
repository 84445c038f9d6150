"""merge_ec_files and `ec-merge` without a GPU: the rule of a merge stated in Python (tests/merge_oracle.py) and checked
against hand-built cases, the host plumbing (reading, sections, writing) with a builder that follows that statement,
every refusal before a builder is made or the output is touched, and the command line."""
import glob
import os
import struct

import numpy as np
import pytest
from click.testing import CliRunner

from conftest import GOLDEN
from alntools_b200 import bin_utils, cli
import merge_oracle as mo

A, B, C, D = ((0, 1),), ((0, 1), (2, 3)), ((1, 2),), ((3, 1),)


def _n(cols):
    """cols: per column a list of (row, count) -> CSC arrays."""
    indptr = np.cumsum([0] + [len(c) for c in cols]).astype(np.int32)
    return (indptr, np.asarray([e for c in cols for e, _ in c], np.int32), np.asarray([v for c in cols for _, v in c],
                                                                                      np.int32))


def _lists(n):
    return tuple(np.asarray(x).tolist() for x in n)


# ---- the rule ----------------------------------------------------------------------------------------------------
def test_overlap_across_files():
    rows, n = mo.merge_statement([([A, B], _n([[(0, 2), (1, 1)]])), ([B, C], _n([[(0, 4), (1, 3)]]))])
    assert rows == [A, B, C]
    assert _lists(n) == ([0, 2, 4], [0, 1, 1, 2], [2, 1, 4, 3])


def test_ec_first_seen_in_a_later_file():
    rows, n = mo.merge_statement([([A], _n([[(0, 1)]])), ([C, A], _n([[(0, 5), (1, 6)]]))])
    assert rows == [A, C]
    assert _lists(n) == ([0, 1, 3], [0, 0, 1], [1, 6, 5])   # ids ascend inside a column


def test_local_ids_in_another_order_in_a_later_file():
    rows, n = mo.merge_statement([([A, B, C], _n([[(0, 1), (1, 1), (2, 1)]])), ([C, B, A], _n([[(0, 7), (2, 9)]]))])
    assert rows == [A, B, C]
    assert _lists(n) == ([0, 3, 5], [0, 1, 2, 0, 2], [1, 1, 1, 9, 7])


def test_columns_zeros_and_rows_without_entries():
    files = [([A, B], _n([[(0, 3)], [], [(0, 0), (1, 2)]])), ([D, A], _n([[(1, 1)], [(0, 0)]]))]
    rows, n = mo.merge_statement(files)
    assert rows == [A, B, D]                                   # D has no entry but is an EC
    assert _lists(n) == ([0, 1, 1, 2, 3, 3], [0, 1, 0], [3, 2, 1])


def test_one_file_is_itself():
    a, n = [A, B, C], _n([[(2, 1), (0, 4)], [(1, 2)]])
    rows, got = mo.merge_statement([(a, n)])
    assert rows == a and _lists(got) == ([0, 2, 3], [0, 2, 1], [4, 1, 2])   # ids ascend inside a column


# ---- the host plumbing, with a builder that follows the statement --------------------------------------------------
class _StatementBuilder(object):
    made = []

    def __init__(self, n_targets, n_haps, **kw):
        self.files, self.pending, self.seen = [], None, set()
        _StatementBuilder.made.append(self)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def push_ecs(self, a_indptr, a_indices, a_data, order_base=0):
        assert self.pending is None and order_base == 0
        self.pending = mo.rows_of((a_indptr, a_indices, a_data))
        self.seen.update(self.pending)

    def append_samples(self, n_indptr, n_indices, n_data):
        self.files.append((self.pending, tuple(np.array(x) for x in (n_indptr, n_indices, n_data))))
        self.pending = None
        return int(np.count_nonzero(n_data))

    def stats(self):
        return {"ec_claimed": len(self.seen)}

    def finalize_samples(self, copy=True):
        rows, n = mo.merge_statement(self.files)
        a = mo.a_csr(rows)
        return {"n_ec": len(rows), "nnz_a": len(a[1]), "nnz_n": len(n[1]), "n_samples": len(n[0]) - 1,
                "a_indptr": a[0], "a_indices": a[1], "a_data": a[2], "n_indptr": n[0], "n_indices": n[1],
                "n_data": n[2]}


@pytest.fixture
def statement_builder(monkeypatch):
    from alntools_b200 import _native
    monkeypatch.setattr(_native, "EcBuilder", _StatementBuilder)
    for var in ("ALNTOOLS_GPUS", "WORLD_SIZE", "RANK"):
        monkeypatch.delenv(var, raising=False)
    _StatementBuilder.made = []
    return _StatementBuilder


def _goldens():
    return sorted(glob.glob(os.path.join(GOLDEN, "**", "*.bin"), recursive=True))


def _read(path):
    with open(path, "rb") as fh:
        return fh.read()


@pytest.mark.parametrize("path", _goldens(), ids=os.path.basename)
def test_one_golden_gives_its_bytes(path, statement_builder, tmp_path):
    out = str(tmp_path / "m.bin")
    summary = bin_utils.merge_ec_files([path], out)
    assert _read(out) == _read(path)
    assert summary["ecs_added"] == [summary["n_ec"]]


def test_two_files_give_the_statement(statement_builder, tmp_path):
    a, b = os.path.join(GOLDEN, "toy_multi.m2.bin"), os.path.join(GOLDEN, "toy_multi.m-1.bin")
    out = str(tmp_path / "m.bin")
    summary = bin_utils.merge_ec_files([a, b, a], out, sample_names=["c%d" % i for i in range(13)])
    got, want = bin_utils.ecload_arrays(out), mo.merge_files([a, b, a])
    for x, y in zip(got["a"] + got["n"], want["a"] + want["n"]):
        assert np.array_equal(x, y)
    assert got["samples"] == ["c%d" % i for i in range(13)]
    assert summary["n_samples"] == 13 and summary["ecs_added"][2] == 0


# ---- refusals ------------------------------------------------------------------------------------------------------
class _NoBuilder(object):
    def __init__(self, *a, **kw):
        raise AssertionError("no builder may be created")


@pytest.fixture
def nobuild(tmp_path, monkeypatch):
    from alntools_b200 import _native
    monkeypatch.setattr(_native, "EcBuilder", _NoBuilder)
    for var in ("ALNTOOLS_GPUS", "WORLD_SIZE", "RANK"):
        monkeypatch.delenv(var, raising=False)
    return str(tmp_path / "out.bin")


def _check_refused(inputs, out, error, match, **kw):
    with pytest.raises(error, match=match):
        bin_utils.merge_ec_files(inputs, out, **kw)
    assert not os.path.exists(out)


TOY = os.path.join(GOLDEN, "toy_single.bin")


def test_no_file(nobuild):
    _check_refused([], nobuild, ValueError, "at least one EC file")


def test_sample_names_must_match_columns(nobuild):
    m2, m3 = os.path.join(GOLDEN, "toy_multi.m2.bin"), os.path.join(GOLDEN, "toy_multi.m3.bin")   # 4 and 2 columns
    _check_refused([m2, m3], nobuild, ValueError, "2 sample names for 6 columns", sample_names=["a", "b"])


def test_emase_output_is_refused(nobuild, tmp_path):
    _check_refused([TOY], str(tmp_path / "out.h5"), NotImplementedError, "ec2emase")


@pytest.mark.parametrize("how", ["env", "launcher"])
def test_more_than_one_gpu_is_refused(how, nobuild, monkeypatch):
    if how == "env":
        monkeypatch.setenv("ALNTOOLS_GPUS", "2")
    else:
        monkeypatch.setenv("WORLD_SIZE", "2")
        monkeypatch.setenv("RANK", "0")
    _check_refused([TOY], nobuild, NotImplementedError, "one GPU")


def test_header_mismatch_names_the_file(nobuild):
    other = os.path.join(GOLDEN, "synth_h2.bin")
    _check_refused([TOY, TOY, other], nobuild, ValueError, "synth_h2.bin: its haplotype or target section differs")
    _check_refused([TOY, os.path.join(GOLDEN, "range_single_targets.bin")], nobuild, ValueError,
                   "range_single_targets.bin")


def _edited(tmp_path, name, fn):
    raw = bytearray(_read(TOY))
    raw = fn(raw)
    p = str(tmp_path / name)
    with open(p, "wb") as fh:
        fh.write(bytes(raw))
    return p


@pytest.mark.parametrize("kind,fn,match", [
    ("format", lambda r: struct.pack("<i", 1) + r[4:], "not an EC file of format 2"),
    ("truncated", lambda r: r[:-3], "truncated"),
    ("cut_header", lambda r: r[:10], "truncated"),
    ("trailing", lambda r: r + b"\0\0\0\0", "trailing bytes"),
    ("n_sizes", lambda r: r[:-16] + struct.pack("<i", 3) + r[-12:], None),
    ("no_sample", None, "at least one sample"),
])
def test_malformed_files_are_refused(kind, fn, match, nobuild, tmp_path):
    if kind == "no_sample":
        sec = bin_utils._ec_sections(TOY)
        at = len(sec["header"])
        raw = _read(TOY)
        # drop the one sample name: count 0, then the matrices
        p = str(tmp_path / "none.bin")
        with open(p, "wb") as fh:
            fh.write(raw[:at] + struct.pack("<i", 0) + raw[sec["matrices_at"]:])
    else:
        p = _edited(tmp_path, kind + ".bin", fn)
    if kind == "n_sizes":
        # toy_single ends with N = (2, 3, [0, 3], [0, 1, 2], [c0, c1, c2]); the entry count is changed
        raw = _read(TOY)
        n_at = len(raw) - 4 * (2 + 2 + 3 + 3)
        with open(p, "wb") as fh:
            fh.write(raw[:n_at] + struct.pack("<ii", 3, 3) + raw[n_at + 8:])
        match = "inconsistent N sizes"
    _check_refused([TOY, p], nobuild, ValueError, os.path.basename(p) + ": .*" + match)


# ---- the command line --------------------------------------------------------------------------------------------
def test_command_reaches_merge_ec_files(tmp_path, monkeypatch):
    calls = []
    monkeypatch.setattr(bin_utils, "merge_ec_files", lambda *a, **kw: calls.append((a, kw)))
    ins = [TOY, os.path.join(GOLDEN, "toy_multi.m2.bin")]
    out = str(tmp_path / "o.bin")
    runner = CliRunner()
    res = runner.invoke(cli.main, ["ec-merge", out] + ins + ["-s", "x", "--sample", "y", "-v"])
    assert res.exit_code == 0, res.output + repr(res.exception)
    assert calls == [((ins, out), dict(sample_names=["x", "y"]))]
    calls.clear()
    res = runner.invoke(cli.main, ["ec-merge", out] + ins)
    assert res.exit_code == 0, res.output
    assert calls == [((ins, out), dict(sample_names=None))]
    assert runner.invoke(cli.main, ["ec-merge", out]).exit_code != 0                     # at least one input
    assert runner.invoke(cli.main, ["ec-merge", out, str(tmp_path / "no.bin")]).exit_code != 0
    params = {p.name: sorted(p.opts) for p in cli.main.get_command(None, "ec-merge").params}
    assert params == {"ec_file": ["ec_file"], "in_files": ["in_files"], "samples": ["--sample", "-s"],
                      "verbose": ["--verbose", "-v"]}


def test_module_command_line_has_every_command():
    """`python -m alntools_b200` runs cli.main: the converter group's commands and ec-merge."""
    import click
    ctx = click.Context(cli.main)
    assert sorted(cli.main.list_commands(ctx)) == sorted(list(cli.cli.commands) + ["ec-merge"])
    for name in cli.cli.commands:
        assert cli.main.get_command(ctx, name) is cli.cli.commands[name]
