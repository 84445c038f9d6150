"""convert_samples and `bam2ec-samples` without a GPU: the refusals, the command line, and the rules of several samples
in one EC file, stated in Python (samples_statement) and checked against hand-built cases.  The host plumbing of
convert_samples runs with a builder that follows that statement, against the EC file bytes of tests/samples_oracle.py."""
import os

import numpy as np
import pytest
from click.testing import CliRunner

from conftest import GOLDEN, golden_cases
from alntools_b200 import bam_io, bam_utils, cli
import samples_oracle as so


# ---- the rules -------------------------------------------------------------------------------------------------
def samples_statement(samples):
    """samples: per sample, its reads in order, each read a list of elements.  An EC is a set of elements; its id is
    the rank of its first occurrence over sample 1, then sample 2, ...; entry (e, s) of N counts the reads of sample s
    in EC e.  -> (EC sets in id order, n_indptr, n_indices, n_data), N as CSC with ids ascending in a column."""
    ids, columns = {}, []
    for reads in samples:
        counts = {}
        for read in reads:
            e = ids.setdefault(frozenset(read), len(ids))
            counts[e] = counts.get(e, 0) + 1
        columns.append(counts)
    indptr, indices, data = so.n_csc(columns)
    return list(ids), indptr.tolist(), indices.tolist(), data.tolist()


def test_empty_sample_is_an_empty_column():
    ecs, indptr, indices, data = samples_statement([[["a"]], [], [["a"], ["a"]]])
    assert ecs == [{"a"}] and indptr == [0, 1, 1, 2] and indices == [0, 0] and data == [1, 2]


def test_one_read_sample():
    assert samples_statement([[["x", "y"]]]) == ([{"x", "y"}], [0, 1], [0], [1])


def test_ec_first_seen_in_a_later_sample():
    ecs, indptr, indices, data = samples_statement([[["a"], ["a"]], [["b"], ["a"]]])
    assert ecs == [{"a"}, {"b"}]
    assert indptr == [0, 1, 3] and indices == [0, 0, 1] and data == [2, 1, 1]    # ids ascend inside a column


def test_equal_sets_are_one_ec_across_samples():
    ecs, indptr, indices, data = samples_statement([[["a", "b"], ["b", "a", "a"]], [["b", "a"]], [["a"]]])
    assert ecs == [{"a", "b"}, {"a"}]
    assert indptr == [0, 1, 2, 3] and indices == [0, 0, 1] and data == [2, 1, 1]


def test_one_sample_is_the_single_sample_count():
    reads = [["a"], ["b", "c"], ["a"], ["c", "b"]]
    ecs, indptr, indices, data = samples_statement([reads])
    assert indptr == [0, len(ecs)] and indices == list(range(len(ecs))) and data == [2, 2]


# ---- convert_samples on the host, with a builder that follows the statement --------------------------------------
class _StatementBuilder(object):
    """Stands in for EcBuilder: pushes are read into reads of (target, haplotype) elements, closes end samples, and
    finalize_samples builds A and N from samples_statement."""
    made = []

    def __init__(self, n_targets, n_haps, with_cells=False, **kw):
        self.samples, self.open, self.bases = [], [], []
        _StatementBuilder.made.append(self)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def push(self, rg, tg, hp, cell=None, order_base=0, drop_last_group=False, n=None):
        n = len(rg) if n is None else int(n)
        rg, tg, hp = (np.asarray(x)[:n] for x in (rg, tg, hp))
        self.bases.append(order_base)
        for r in np.unique(rg):
            sel = rg == r
            self.open.append(list(zip(tg[sel].tolist(), hp[sel].tolist())))

    def close_sample(self):
        self.samples.append(self.open)
        self.open = []
        return 0

    def finalize_samples(self, copy=True):
        assert not self.open
        ecs, indptr, indices, data = samples_statement(self.samples)
        a_indptr, a_indices, a_data = [0], [], []
        for ec in ecs:
            masks = {}
            for t, h in ec:
                masks[t] = masks.get(t, 0) | (1 << h)
            a_indices += sorted(masks)
            a_data += [masks[t] for t in sorted(masks)]
            a_indptr.append(len(a_indices))
        i32 = lambda v: np.asarray(v, dtype=np.int32)
        return {"n_ec": len(ecs), "n_reads": sum(len(s) for s in self.samples), "n_samples": len(self.samples),
                "a_indptr": i32(a_indptr), "a_indices": i32(a_indices), "a_data": i32(a_data),
                "n_indptr": i32(indptr), "n_indices": i32(indices), "n_data": i32(data)}


@pytest.fixture
def statement_builder(built, monkeypatch):
    monkeypatch.setattr(bam_utils, "EcBuilder", _StatementBuilder)
    _StatementBuilder.made = []
    return _StatementBuilder


@pytest.fixture(scope="module")
def union(tmp_path_factory):
    names = ["toy_single", "mixed_single", "range_single"]
    cases = {c["name"]: c for c in golden_cases("single")}
    return so.union_goldens([os.path.join(GOLDEN, cases[n]["bam"]) for n in names],
                            str(tmp_path_factory.mktemp("samples_host")))


@pytest.mark.parametrize("emitter", ["native", "python"])
def test_host_plumbing_matches_the_oracle(emitter, statement_builder, union, tmp_path, monkeypatch):
    monkeypatch.setenv("ALNTOOLS_B200_EMITTER", emitter)
    for paths in (union, union[::-1], union[:1]):
        names = ["s%d" % i for i in range(len(paths))]
        ec = str(tmp_path / "x.bin")
        bam_utils.convert_samples(paths, ec, sample_names=names)
        with open(ec, "rb") as fh:
            assert fh.read() == so.ec_file_bytes(paths, names)
        b = statement_builder.made[-1]
        assert len(b.samples) == len(paths) and set(b.bases) == {0}    # each sample pushed from order_base 0


def test_one_golden_gives_its_bytes(statement_builder, tmp_path):
    import hashlib
    for case in golden_cases("single"):
        ec = str(tmp_path / "x.bin")
        targets = os.path.join(GOLDEN, case["targets"]) if case.get("targets") else None
        bam_utils.convert_samples([os.path.join(GOLDEN, case["bam"])], ec, target_filename=targets)
        with open(ec, "rb") as fh:
            assert hashlib.sha256(fh.read()).hexdigest() == case["sha256"], case["name"]


# ---- refusals ----------------------------------------------------------------------------------------------------
class _NoBuilder(object):
    def __init__(self, *a, **kw):
        raise AssertionError("no builder may be created")


@pytest.fixture
def missing(tmp_path, monkeypatch):
    """Paths that do not exist: a call that opened one would fail differently."""
    monkeypatch.setattr(bam_utils, "EcBuilder", _NoBuilder)
    for var in ("ALNTOOLS_GPUS", "WORLD_SIZE", "RANK", "ALNTOOLS_B200_MAX_READ", "ALNTOOLS_B200_COLLATE",
                "ALNTOOLS_B200_COLLATE_BUDGET", "ALNTOOLS_B200_DECODE", "ALNTOOLS_B200_EMITTER"):
        monkeypatch.delenv(var, raising=False)
    return [str(tmp_path / "a.bam"), str(tmp_path / "b.bam")], str(tmp_path / "out.bin")


def test_no_file(missing):
    with pytest.raises(ValueError, match="at least one BAM file"):
        bam_utils.convert_samples([], missing[1])


def test_names_must_match_files(missing):
    with pytest.raises(ValueError, match="3 sample names for 2 BAM files"):
        bam_utils.convert_samples(missing[0], missing[1], sample_names=["a", "b", "c"])
    assert not os.path.exists(missing[1])


@pytest.mark.parametrize("how", ["devices", "env", "launcher"])
def test_more_than_one_gpu_is_refused(how, missing, monkeypatch):
    kw = {}
    if how == "devices":
        kw["devices"] = 2
    elif how == "env":
        monkeypatch.setenv("ALNTOOLS_GPUS", "4")
    else:
        monkeypatch.setenv("WORLD_SIZE", "2")
        monkeypatch.setenv("RANK", "0")
    with pytest.raises(NotImplementedError, match="one GPU"):
        bam_utils.convert_samples(*missing, **kw)
    assert not os.path.exists(missing[1])


def test_emase_output_is_refused(missing, tmp_path):
    with pytest.raises(NotImplementedError, match="EMASE"):
        bam_utils.convert_samples(missing[0], str(tmp_path / "out.h5"))


@pytest.mark.parametrize("var,value", [("ALNTOOLS_B200_MAX_READ", "16k"), ("ALNTOOLS_B200_COLLATE", "yes"),
                                       ("ALNTOOLS_B200_COLLATE_BUDGET", "-1"), ("ALNTOOLS_B200_DECODE", "gpu")])
def test_bad_environment_is_refused(var, value, missing, monkeypatch):
    monkeypatch.setenv(var, value)
    if var == "ALNTOOLS_B200_COLLATE_BUDGET":
        monkeypatch.setenv("ALNTOOLS_B200_COLLATE", "1")
    with pytest.raises(ValueError):
        bam_utils.convert_samples(*missing)
    assert not os.path.exists(missing[1])


@pytest.mark.parametrize("combination", [dict(decode="device", collate=True), dict(range_python=True)])
def test_combinations_convert_refuses_are_refused(combination, missing, monkeypatch):
    if combination.pop("range_python", False):
        monkeypatch.setenv("ALNTOOLS_B200_EMITTER", "python")
        combination = dict(range_filename=missing[1] + ".range")
    with pytest.raises(NotImplementedError):
        bam_utils.convert_samples(*missing, **combination)


def _with_header(path, refs, records=()):
    bam_io.write_bam(path, refs, list(records))
    return path


@pytest.mark.parametrize("emitter", ["native", "python"])
def test_header_mismatch_is_refused_before_any_push(emitter, built, tmp_path, monkeypatch):
    monkeypatch.setattr(bam_utils, "EcBuilder", _NoBuilder)
    monkeypatch.setenv("ALNTOOLS_B200_EMITTER", emitter)
    rec = [("r1", 0, 0, 5, -1, -1)]
    refs = [("T0_A", 100), ("T0_B", 100)]
    a = _with_header(str(tmp_path / "a.bam"), refs, rec)
    same = _with_header(str(tmp_path / "same.bam"), refs, rec)
    longer = _with_header(str(tmp_path / "longer.bam"), [("T0_A", 100), ("T0_B", 101)], rec)
    renamed = _with_header(str(tmp_path / "renamed.bam"), [("T0_A", 100), ("T1_B", 100)], rec)
    fewer = _with_header(str(tmp_path / "fewer.bam"), refs[:1], rec)
    for bad in (longer, renamed, fewer):
        with pytest.raises(ValueError, match=os.path.basename(bad) + " does not have the @SQ list"):
            bam_utils.convert_samples([a, same, bad, longer], str(tmp_path / "x.bin"))
    assert not os.path.exists(str(tmp_path / "x.bin"))


# ---- the command line --------------------------------------------------------------------------------------------
def test_command_options(tmp_path, monkeypatch):
    calls = []
    monkeypatch.setattr(bam_utils, "convert_samples", lambda *a, **kw: calls.append((a, kw)))
    bams = [os.path.join(GOLDEN, c["bam"]) for c in golden_cases("single")[:2]]
    targets = os.path.join(GOLDEN, "range_single.targets.txt")
    out, rng = str(tmp_path / "o.bin"), str(tmp_path / "r.txt")
    runner = CliRunner()
    res = runner.invoke(cli.cli, ["bam2ec-samples", out] + bams + ["-s", "x", "--sample", "y", "-t", targets,
                                                                    "--rangefile", rng, "-v"])
    assert res.exit_code == 0, res.output + repr(res.exception)
    assert calls == [((bams, out), dict(sample_names=["x", "y"], target_filename=targets, range_filename=rng))]
    calls.clear()
    res = runner.invoke(cli.cli, ["bam2ec-samples", out] + bams)
    assert res.exit_code == 0, res.output
    assert calls == [((bams, out), dict(sample_names=None, target_filename=None, range_filename=None))]
    assert runner.invoke(cli.cli, ["bam2ec-samples", out]).exit_code != 0                 # at least one BAM file
    assert runner.invoke(cli.cli, ["bam2ec-samples", out, str(tmp_path / "no.bam")]).exit_code != 0
    names = sorted(cli.cli.commands)
    assert names == ["bam2ec", "bam2ec-samples", "bam2emase", "ec2emase"]
    params = {p.name: sorted(p.opts) for p in cli.cli.commands["bam2ec-samples"].params}
    assert params == {"ec_file": ["ec_file"], "bam_files": ["bam_files"], "samples": ["--sample", "-s"],
                      "rangefile": ["--rangefile"], "targets": ["--targets", "-t"], "verbose": ["--verbose", "-v"]}
