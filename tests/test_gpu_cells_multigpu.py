"""The multi-GPU per-cell path as users run it: the NCCL job of tests/multigpu_cells_check.py (at world 2 or 4 where
the GPUs are there, else at world 1, which still runs the whole orchestration), and, with at least 2 GPUs,
convert_files(devices=N) and the CLI with ALNTOOLS_GPUS=N on the multisample goldens."""
import hashlib
import os
import subprocess
import sys

import pytest

from conftest import GOLDEN, ROOT, golden_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def native(built):
    import torch
    assert torch.cuda.is_available(), "these tests need a B200"
    from alntools_b200 import _native
    _native.load_library()
    return _native


def test_multigpu_cells_exchange_matches_oracle(native):
    import torch
    n = torch.cuda.device_count()
    world = 1 if n < 2 else 2 if n < 4 else 4
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                          "--master-addr", "127.0.0.1", "--master-port", "29541",
                          os.path.join(ROOT, "tests", "multigpu_cells_check.py"), "300000"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert out.stdout.count("OK") == 2 and "MISMATCH" not in out.stdout, out.stdout[-2000:]


def _sha(path):
    with open(path, "rb") as fh:
        return hashlib.sha256(fh.read()).hexdigest()


def _generated_dir(tmp_path):
    """6 per-cell BAM files, about 1.5 M reads over 5 000 cells.  -> (file paths in order, minimum count)."""
    from alntools_b200 import multi_gpu, synth
    d = tmp_path / "gen"
    d.mkdir()
    cols = synth.make_columns(1_500_000, 20000, 2, seed=91, mode="diploid", n_cells=5000, dup_rate=0.01)
    cuts = multi_gpu.shard_bounds(cols["read_group"], 6)
    files = []
    for i in range(6):
        part = {k: cols[k][cuts[i]:cuts[i + 1]] for k in ("read_group", "target_idx", "hap_idx", "cell_idx")}
        files.append(str(d / ("f%d.bam" % i)))
        synth.columns_to_bam_cells(files[-1], part, 20000, 2)
    return files, 50


def _rank_body_world1(files, out, min_count, rng=None):
    """bam_utils_multisample.convert_files_rank as the only rank of a job (the orchestration of the multi-GPU
    convert - decode, name merge, exchange, header, slice writes, range all-reduce - on one GPU)."""
    import json
    code = ("import json, sys; sys.path.insert(0, %r); from alntools_b200 import bam_utils_multisample as m; "
            "a = json.loads(sys.argv[1]); m.convert_files_rank(a[0], a[1], None, a[2], range_filename=a[3])" % ROOT)
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29543")
    subprocess.check_call([sys.executable, "-c", code, json.dumps([files, out, min_count, rng])], env=env, cwd=ROOT,
                          timeout=600)


def test_cells_rank_body_matches_one_gpu_file(native, tmp_path):
    """The multi-GPU rank body at world 1 writes the golden EC files, and on a generated 6-file directory the
    same EC and range files as the one-GPU convert_files."""
    from alntools_b200 import bam_utils_multisample
    for case in golden_cases("multisample"):
        files = [os.path.join(GOLDEN, case["dir"], f) for f in case["file_order"]]
        out = str(tmp_path / ("%s.rank.bin" % case["name"]))
        _rank_body_world1(files, out, case["mincount"])
        assert _sha(out) == case["sha256"], case["name"]
    files, min_count = _generated_dir(tmp_path)
    one, one_rng = str(tmp_path / "gen.1.bin"), str(tmp_path / "gen.1.range")
    bam_utils_multisample.convert_files(files, one, None, min_count, range_filename=one_rng)
    out, out_rng = str(tmp_path / "gen.rank.bin"), str(tmp_path / "gen.rank.range")
    _rank_body_world1(files, out, min_count, out_rng)
    assert _sha(out) == _sha(one)
    assert _sha(out_rng) == _sha(one_rng)


def test_multigpu_cells_convert_writes_the_golden_files(native, tmp_path):
    """convert_files(devices=N) and the CLI with ALNTOOLS_GPUS=N at N = 2 and all GPUs: the multisample goldens
    byte-identical, and a generated 6-file, 1.5 M-read directory identical to the one-GPU file."""
    import torch
    from alntools_b200 import bam_utils_multisample
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")

    def cli(directory, out, gpus, min_count):
        env = dict(os.environ, ALNTOOLS_GPUS=str(gpus), PYTHONPATH=ROOT)
        subprocess.check_call([sys.executable, "-m", "alntools_b200", "bam2ec", directory, out, "--multisample",
                               "-m", str(min_count)], env=env, cwd=ROOT)

    files, min_count = _generated_dir(tmp_path)
    cases = [(c["name"], [os.path.join(GOLDEN, c["dir"], f) for f in c["file_order"]], c["mincount"], c["sha256"])
             for c in golden_cases("multisample")] + [("generated", files, min_count, None)]
    for name, paths, mc, sha in cases:
        one = str(tmp_path / ("%s.1.bin" % name))
        bam_utils_multisample.convert_files(paths, one, None, mc)
        if sha is not None:
            assert _sha(one) == sha, name
        cli_one = str(tmp_path / ("%s.cli1.bin" % name))
        cli(os.path.dirname(paths[0]), cli_one, 1, mc)
        for w in sorted({2, n}):
            out = str(tmp_path / ("%s.%d.bin" % (name, w)))
            bam_utils_multisample.convert_files(paths, out, None, mc, devices=w)
            assert _sha(out) == _sha(one), (name, w)
            cli_out = str(tmp_path / ("%s.cli%d.bin" % (name, w)))
            cli(os.path.dirname(paths[0]), cli_out, w, mc)
            assert _sha(cli_out) == _sha(cli_one), (name, w)
