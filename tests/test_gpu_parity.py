"""Parity tests proper: the CUDA path, called through the C ABI (ctypes -> libecb200.so), against the
oracle on the same seeded inputs, against the reference's golden EC files, and - at BASELINE.json's
full sizes - through size-independent properties plus the C oracle.  Bit-exact everywhere (integer work)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def native(built):
    import torch
    assert torch.cuda.is_available(), "these tests need a B200"
    from alntools_b200 import _native
    _native.load_library()
    return _native


def _oracle(cols, drop_last=False):
    from oracle import c_oracle
    return c_oracle.ec_from_columns(cols["read_group"], cols["target_idx"], cols["hap_idx"], drop_last)


def _assert_same(got, want):
    indptr, indices, data, counts, n_reads = want
    assert got["n_reads"] == n_reads
    assert got["n_ec"] == len(counts)
    assert np.array_equal(got["a_indptr"], indptr)
    assert np.array_equal(got["a_indices"], indices)
    assert np.array_equal(got["a_data"], data)
    assert np.array_equal(got["n_data"], counts)
    assert got["n_indptr"].tolist() == [0, len(counts)]
    assert np.array_equal(got["n_indices"], np.arange(len(counts), dtype=np.int32))


def _run(native, cols, n_targets, n_haps, **options):
    with native.EcBuilder(n_targets, n_haps, alignments_hint=len(cols["read_group"]), **options) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
        return b.finalize(), b.stats()


# ---------------------------------------------------------------- golden files (reference outputs)
@pytest.mark.parametrize("case", golden_cases("single"), ids=lambda c: c["name"])
def test_convert_reproduces_reference_file_single(native, case, tmp_path):
    from alntools_b200 import bam_utils
    out = str(tmp_path / "out.bin")
    tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
    bam_utils.convert(os.path.join(GOLDEN, case["bam"]), out, None, num_chunks=1, number_processes=1,
                      target_filename=tfile)
    with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
        assert a.read() == b.read()


@pytest.mark.parametrize("case", golden_cases("multisample"), ids=lambda c: c["name"])
def test_convert_reproduces_reference_file_multisample(native, case, tmp_path):
    from alntools_b200 import bam_utils_multisample
    out = str(tmp_path / "out.bin")
    files = [os.path.join(GOLDEN, case["dir"], fn) for fn in case["file_order"]]
    bam_utils_multisample.convert_files(files, out, None, case["mincount"])
    with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
        assert a.read() == b.read()


def test_convert_with_rangefile_reproduces_reference_files(native, tmp_path):
    """EC file and --rangefile report together, single-sample and per-cell (goldens of make_golden_range.py)."""
    import json
    from alntools_b200 import bam_utils, bam_utils_multisample
    with open(os.path.join(GOLDEN, "manifest_range.json")) as fh:
        cases = json.load(fh)
    for case in cases:
        out, rng = str(tmp_path / (case["name"] + ".bin")), str(tmp_path / (case["name"] + ".range.txt"))
        if case["kind"] == "single":
            tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
            bam_utils.convert(os.path.join(GOLDEN, case["bam"]), out, None, num_chunks=1, number_processes=1,
                              range_filename=rng, target_filename=tfile)
        else:
            files = [os.path.join(GOLDEN, case["dir"], fn) for fn in case["file_order"]]
            bam_utils_multisample.convert_files(files, out, None, case["mincount"], range_filename=rng)
        with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
            assert a.read() == b.read(), case["name"]
        with open(rng) as a, open(os.path.join(GOLDEN, case["range"])) as b:
            assert a.read() == b.read(), case["name"]


# ---------------------------------------------------------------- seeded columns vs the oracle
@pytest.mark.parametrize("n_reads,n_targets,n_haps,mode,dup", [
    (1, 5, 2, "light", 0.0),
    (7, 5, 2, "light", 0.5),
    (1000, 50, 2, "light", 0.05),          # tiny target space: few, very hot ECs
    (1023, 300, 2, "diploid", 0.0),
    (50000, 2000, 2, "light", 0.02),       # cfg1 shape, scaled down
    (200000, 2000, 2, "diploid", 0.02),
    (30000, 1500, 8, "heavy", 0.01),       # reads longer than a warp and than a tile
    (4000, 1000, 8, 64, 0.0),              # fixed 64 transcripts per read (cfg5)
    (300000, 100000, 2, "diploid", 0.0),   # cfg2 shape, scaled down
])
def test_columns_match_oracle(native, n_reads, n_targets, n_haps, mode, dup):
    from alntools_b200 import synth
    cols = synth.make_columns(n_reads, n_targets, n_haps, seed=n_reads % 97 + 1, mode=mode, dup_rate=dup)
    got, _ = _run(native, cols, n_targets, n_haps)
    _assert_same(got, _oracle(cols))


def test_tile_and_chunk_boundaries(native):
    """Sizes around the 32-alignment window and reads that straddle window / work-chunk boundaries."""
    from alntools_b200 import synth
    for n_reads in (15, 16, 17, 31, 32, 33, 340, 341, 342, 512, 1024, 1025, 2047, 2048, 2049, 4096):
        cols = synth.make_columns(n_reads, 40, 3, seed=n_reads, mode="diploid", dup_rate=0.1)
        want = _oracle(cols)
        for grid, chunk in ((0, 0), (1, 32), (3, 64), (2, 96), (148, 32)):
            got, _ = _run(native, cols, 40, 3, grid_ctas=grid, chunk_len=chunk)
            _assert_same(got, want)
    # exactly one tile, exactly two tiles, one alignment per read
    for n in (1024, 2048, 3072):
        rg = np.arange(n, dtype=np.int32)
        cols = {"read_group": rg, "target_idx": (rg % 7).astype(np.int32), "hap_idx": (rg % 2).astype(np.int32)}
        got, _ = _run(native, cols, 7, 2, grid_ctas=2)
        _assert_same(got, _oracle(cols))


def test_giant_read_spanning_many_tiles(native):
    """One read of 5000 alignments (> 4 tiles) between ordinary reads; 5000 <= ECB_MAX_READ_ALIGNMENTS."""
    rng = np.random.default_rng(3)
    rg = np.concatenate([np.repeat(np.arange(300), 3), np.full(5000, 300), np.repeat(np.arange(301, 700), 2)])
    tg = rng.integers(0, 900, len(rg))
    hp = rng.integers(0, 4, len(rg))
    cols = {"read_group": rg.astype(np.int32), "target_idx": tg.astype(np.int32), "hap_idx": hp.astype(np.int32)}
    want = _oracle(cols)
    for grid, chunk in ((0, 0), (2, 256), (5, 32), (1, 4096)):
        got, _ = _run(native, cols, 900, 4, grid_ctas=grid, chunk_len=chunk)
        _assert_same(got, want)


def test_read_longer_than_the_limit_is_an_error(native):
    n = 16384 + 40
    cols = {"read_group": np.zeros(n, np.int32), "target_idx": (np.arange(n) % 30000).astype(np.int32),
            "hap_idx": np.zeros(n, np.int32)}
    with native.EcBuilder(30000, 1) as b:
        with pytest.raises(native.EcbError) as info:
            b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
            b.finalize()
    assert info.value.code == -4


def test_out_of_range_values_are_an_error(native):
    with native.EcBuilder(10, 2) as b:
        with pytest.raises(native.EcbError) as info:
            b.push(np.array([0, 1], np.int32), np.array([3, 10], np.int32), np.array([0, 1], np.int32))
    assert info.value.code == -1


def test_empty_input_raises_like_the_reference(native):
    with native.EcBuilder(10, 2) as b:
        e = np.zeros(0, np.int32)
        b.push(e, e, e)
        with pytest.raises(native.EcbError) as info:
            b.finalize()
    assert info.value.code == native.ECB_ERR_EMPTY


def test_table_growth_and_overflow_replay(native):
    """A deliberately tiny table forces probe exhaustion, growth (rehash) and the replay kernel."""
    from alntools_b200 import synth
    cols = synth.make_columns(60000, 20000, 2, seed=21, mode="diploid")
    got, stats = _run(native, cols, 20000, 2, table_slots=1024)
    _assert_same(got, _oracle(cols))
    assert stats["table_grows"] >= 1 and stats["overflow_reads"] > 0


def test_hot_cache_off_gives_the_same_result(native):
    from alntools_b200 import synth
    cols = synth.make_columns(40000, 300, 2, seed=22, mode="light", dup_rate=0.02)
    a, _ = _run(native, cols, 300, 2, hot_cache=1)
    b, _ = _run(native, cols, 300, 2, hot_cache=0)
    for k in ("a_indptr", "a_indices", "a_data", "n_data"):
        assert np.array_equal(a[k], b[k])
    _assert_same(a, _oracle(cols))


def test_multiple_pushes_equal_one_push(native):
    """Chunk independence (bam_utils.py:680-698): pushing read-aligned pieces with their order_base
    gives the same matrices as one push, in any arrival order."""
    from alntools_b200 import synth
    cols = synth.make_columns(50000, 3000, 2, seed=23, mode="diploid", dup_rate=0.02)
    rg = cols["read_group"]
    want = _oracle(cols)
    cuts = [0]
    for k in range(1, 5):
        c = len(rg) * k // 5
        while rg[c] == rg[c - 1]:
            c += 1
        cuts.append(c)
    cuts.append(len(rg))
    pieces = list(zip(cuts[:-1], cuts[1:]))
    for order in (pieces, pieces[::-1], [pieces[2], pieces[0], pieces[4], pieces[1], pieces[3]]):
        with native.EcBuilder(3000, 2, alignments_hint=len(rg)) as b:
            for a, e in order:
                b.push(np.ascontiguousarray(rg[a:e]), np.ascontiguousarray(cols["target_idx"][a:e]),
                       np.ascontiguousarray(cols["hap_idx"][a:e]), order_base=a)
            _assert_same(b.finalize(), want)


def test_overlapping_order_bases_are_detected(native):
    from alntools_b200 import synth
    cols = synth.make_columns(2000, 3000, 2, seed=24, mode="light")
    with native.EcBuilder(3000, 2) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"], order_base=0)
        b.push(cols["read_group"], (cols["target_idx"] + 1) % 3000, cols["hap_idx"], order_base=0)
        with pytest.raises(native.EcbError):
            b.finalize()


def test_device_resident_columns_and_results(native):
    """on_device=1 pushes (torch only hands over device pointers), incl. a 4-byte-misaligned view."""
    import torch
    from alntools_b200 import synth
    cols = synth.make_columns(80000, 5000, 2, seed=25, mode="diploid", dup_rate=0.01)
    want = _oracle(cols)
    dev = {k: torch.from_numpy(cols[k]).cuda() for k in ("read_group", "target_idx", "hap_idx")}
    with native.EcBuilder(5000, 2, alignments_hint=len(cols["read_group"])) as b:
        b.push(dev["read_group"], dev["target_idx"], dev["hap_idx"])
        _assert_same(b.finalize(), want)
        b.reset()
        pad = {k: torch.cat([torch.zeros(1, dtype=torch.int32, device="cuda"), v])[1:] for k, v in dev.items()}
        assert pad["read_group"].data_ptr() % 16 != 0
        b.push(pad["read_group"], pad["target_idx"], pad["hap_idx"])
        _assert_same(b.finalize(), want)
    with native.EcBuilder(5000, 2, alignments_hint=len(cols["read_group"]), result_on_device=1) as b:
        b.push(dev["read_group"], dev["target_idx"], dev["hap_idx"])
        res = b.finalize_raw()
        assert res.n_ec == len(want[3]) and res.nnz_a == len(want[1])


def test_reset_reuses_the_context(native):
    from alntools_b200 import synth
    with native.EcBuilder(500, 2) as b:
        for seed in (31, 32, 33):
            cols = synth.make_columns(20000, 500, 2, seed=seed, mode="light", dup_rate=0.02)
            b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
            _assert_same(b.finalize(), _oracle(cols))
            b.reset()


def test_drop_last_group(native):
    from alntools_b200 import synth
    cols = synth.make_columns(5000, 200, 2, seed=34, mode="diploid")
    with native.EcBuilder(200, 2) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"], drop_last_group=True)
        _assert_same(b.finalize(), _oracle(cols, drop_last=True))


# ---------------------------------------------------------------- per-cell path vs the oracle
@pytest.mark.parametrize("n_files,reads,n_cells,mincount", [(1, 3000, 10, 1), (3, 5000, 40, 1), (4, 20000, 300, 120),
                                                            (2, 60000, 2000, 25)])
def test_cells_match_oracle(native, n_files, reads, n_cells, mincount):
    from alntools_b200 import synth
    from oracle import ec_oracle
    pushes = []
    for f in range(n_files):
        c = synth.make_columns(reads, 800, 2, seed=100 + f, mode="light", n_cells=n_cells, dup_rate=0.02)
        pushes.append((c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"], True))
    want = ec_oracle.ec_from_columns_cells(pushes, mincount)
    total = sum(len(p[0]) for p in pushes)
    with native.EcBuilder(800, 2, with_cells=True, alignments_hint=total) as b:
        base = 0
        for rg, tg, hp, cell, drop in pushes:
            b.push(rg, tg, hp, cell, order_base=base, drop_last_group=drop)
            base += len(rg)
        got = b.finalize(mincount)
    for k in ("a_indptr", "a_indices", "a_data", "n_indptr", "n_indices", "n_data", "cell_order"):
        assert np.array_equal(got[k], want[k]), k


# ---------------------------------------------------------------- full-size properties (BASELINE configs)
_CFG2 = {}


def _cfg2():
    """cfg2's columns and the C oracle's result on them, made once for the tests that use them."""
    if not _CFG2:
        from alntools_b200 import synth
        _CFG2["cols"] = synth.make_columns(30_000_000, 100_000, 2, seed=2, mode="diploid")
        _CFG2["want"] = _oracle(_CFG2["cols"])
    return _CFG2["cols"], _CFG2["want"]


def test_full_size_cfg2_properties_and_oracle(native):
    """cfg2 shape at full size (30 M reads, 2 haplotypes x 100 k transcripts): size-independent
    properties on the GPU result, then the C oracle on the same columns."""
    cols, want = _cfg2()
    got, stats = _run(native, cols, 100_000, 2)
    n_aln = len(cols["read_group"])
    assert got["n_reads"] == cols["n_reads"] and got["n_alignments"] == n_aln
    assert int(got["n_data"].astype(np.int64).sum()) == cols["n_reads"]       # every read counted once
    assert np.all(np.diff(got["a_indptr"]) >= 1)                              # no empty EC
    rows = np.repeat(np.arange(got["n_ec"]), np.diff(got["a_indptr"]))
    same_row = rows[1:] == rows[:-1]
    assert np.all(got["a_indices"][1:][same_row] > got["a_indices"][:-1][same_row])  # sorted, unique targets
    assert got["a_data"].min() >= 1 and got["a_data"].max() <= 3
    # idempotence: a second context gives identical bytes
    again, _ = _run(native, cols, 100_000, 2)
    for k in ("a_indptr", "a_indices", "a_data", "n_data"):
        assert np.array_equal(got[k], again[k])
    _assert_same(got, want)


def test_full_size_cfg2_key_verification(native):
    """EC identity on the device is the 128-bit set hash (DESIGN.md section 3).  ECB_OPT_VERIFY_KEYS re-derives
    every read's set of (target, haplotype) pairs and compares it with the row of the EC it was counted in: at
    cfg2's full size (30 M reads, 4 M ECs) no two different sets may share a key, and the result is the oracle's."""
    cols, want = _cfg2()
    got, _ = _run(native, cols, 100_000, 2, verify_keys=1)      # a collision raises EcbError(ECB_ERR_LIMIT)
    _assert_same(got, want)
    _CFG2.clear()


def test_full_size_cfg3_heavy_with_key_verification(native):
    """cfg3 shape at the size the bench runs per GPU (8 haplotypes x 140 k transcripts, heavy multimapping,
    100 M alignments): key verification on, result against the C oracle."""
    from alntools_b200 import synth
    cols = synth.make_columns(3_000_000, 140_000, 8, seed=3, mode="heavy")
    assert len(cols["read_group"]) > 90_000_000
    got, _ = _run(native, cols, 140_000, 8, verify_keys=1)
    assert int(got["n_data"].astype(np.int64).sum()) == cols["n_reads"]
    _assert_same(got, _oracle(cols))


@pytest.mark.parametrize("degree", [1, 64])
def test_full_size_cfg5_sweep_ends(native, degree):
    """cfg5, the two ends of the multimapping-degree sweep at the bench's size (64 M alignments, exactly
    `degree` alignments per read, 8 haplotypes x 140 k transcripts) against the C oracle."""
    from alntools_b200 import synth
    cols = synth.make_columns(64_000_000 // degree, 140_000, 8, seed=5, mode="aln%d" % degree)
    got, _ = _run(native, cols, 140_000, 8)
    _assert_same(got, _oracle(cols))


def test_full_size_cfg4_cells_50k(native):
    """cfg4 at the bench's size on one GPU: 20 M reads, 50 000 cells (Zipf sizes), 4 files with their last
    read dropped, cells below 1000 reads filtered - against the C statement of the per-cell merge
    (oracle/ec_oracle.c: ec_oracle_build_cells, itself pinned to the Python statement on small cases)."""
    from alntools_b200 import synth
    from oracle import c_oracle
    cols = synth.make_columns(20_000_000, 140_000, 8, seed=4, mode="diploid", n_cells=50_000)
    n = len(cols["read_group"])
    cuts = [0]
    for k in range(1, 4):
        c = n * k // 4
        while c < n and cols["read_group"][c] == cols["read_group"][c - 1]:
            c += 1
        cuts.append(c)
    cuts.append(n)
    pushes = [(cols["read_group"][a:b], cols["target_idx"][a:b], cols["hap_idx"][a:b], cols["cell_idx"][a:b], True)
              for a, b in zip(cuts[:-1], cuts[1:])]
    with native.EcBuilder(140_000, 8, with_cells=True, alignments_hint=n) as b:
        for (rg, tg, hp, cell, drop), base in zip(pushes, cuts[:-1]):
            b.push(rg, tg, hp, cell, order_base=base, drop_last_group=drop)
        got = b.finalize(1000)
    want = c_oracle.ec_from_columns_cells(pushes, 1000)
    assert got["n_reads"] == want["n_reads"]
    for k in ("a_indptr", "a_indices", "a_data", "n_indptr", "n_indices", "n_data", "cell_order"):
        assert np.array_equal(got[k], want[k]), k


# ---------------------------------------------------------------- multi-GPU exchange
def test_multigpu_exchange_matches_oracle(native):
    """The NCCL job of tests/multigpu_check.py: at world 2 or 4 where the GPUs are there, else at world 1, which
    still runs the whole orchestration (arena, stream barriers, both dispatches, id_base)."""
    import subprocess
    import sys
    import torch
    from conftest import ROOT
    n = torch.cuda.device_count()
    world = 1 if n < 2 else 2 if n < 4 else 4
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                          "--master-addr", "127.0.0.1", "--master-port", "29533",
                          os.path.join(ROOT, "tests", "multigpu_check.py"), "300000"],
                         capture_output=True, text=True, timeout=400)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert out.stdout.count("OK") == 3 and "MISMATCH" not in out.stdout, out.stdout[-2000:]


def test_multigpu_convert_writes_the_golden_files(native):
    """convert() / the CLI sharded over GPUs (ALNTOOLS_GPUS; one worker process per GPU, shards of the one BAM
    planned as virtual offsets): golden EC files and a 1.5 M-read file byte-identical at 2 and at all GPUs."""
    import subprocess
    import sys
    import torch
    from conftest import ROOT
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least 2 GPUs")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "multigpu_convert_check.py")],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    assert "multigpu convert check: ok" in out.stdout


def _single_rank_body_world1(bam, out, target_filename=None, range_filename=None):
    """bam_utils.convert_rank as the only rank of a job (the orchestration of the multi-GPU convert - shard plan,
    decode, rebase, exchange, header, slice writes, range all-reduce - on one GPU)."""
    import json
    import subprocess
    import sys
    from conftest import ROOT
    code = ("import json, sys; sys.path.insert(0, %r); from alntools_b200 import bam_utils; a = json.loads(sys.argv[1]); "
            "bam_utils.convert_rank(a[0], a[1], None, range_filename=a[2], target_filename=a[3])" % ROOT)
    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0", MASTER_ADDR="127.0.0.1", MASTER_PORT="29545")
    subprocess.check_call([sys.executable, "-c", code, json.dumps([bam, out, range_filename, target_filename])], env=env,
                          cwd=ROOT, timeout=600)


def test_single_rank_body_matches_one_gpu_file(native, tmp_path):
    """The single-sample multi-GPU rank body at world 1 writes every golden EC file (and the golden range files), and
    on a generated 1.5 M-read file the same EC and range files as the one-GPU convert()."""
    from alntools_b200 import bam_utils, synth
    for case in golden_cases("single"):
        out, rng = str(tmp_path / (case["name"] + ".rank.bin")), str(tmp_path / (case["name"] + ".rank.range"))
        tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
        _single_rank_body_world1(os.path.join(GOLDEN, case["bam"]), out, tfile, rng if case.get("range") else None)
        with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
            assert a.read() == b.read(), case["name"]
        if case.get("range"):
            with open(rng) as a, open(os.path.join(GOLDEN, case["range"])) as b:
                assert a.read() == b.read(), case["name"]
    cols = synth.make_columns(1_500_000, 20000, 2, seed=77, mode="diploid", dup_rate=0.01)
    bam = str(tmp_path / "big.bam")
    synth.columns_to_bam(bam, cols, 20000, 2)
    one, one_rng = str(tmp_path / "big.1.bin"), str(tmp_path / "big.1.range")
    bam_utils.convert(bam, one, None, range_filename=one_rng)
    out, out_rng = str(tmp_path / "big.rank.bin"), str(tmp_path / "big.rank.range")
    _single_rank_body_world1(bam, out, range_filename=out_rng)
    for x, y in ((out, one), (out_rng, one_rng)):
        with open(x, "rb") as a, open(y, "rb") as b:
            assert a.read() == b.read(), x


def test_rebase_moves_the_order_keys(native):
    """ecb_rebase: pushes made with order_base counted from 0 and then moved by a delta give the result of
    pushes made at their final positions (two contexts merged through the single-GPU exchange emulation would
    need more plumbing; here: the EC order of ONE context must not change, and finalize must still work)."""
    from alntools_b200 import synth
    cols = synth.make_columns(50000, 900, 2, seed=61, mode="diploid", dup_rate=0.02)
    want = _oracle(cols)
    with native.EcBuilder(900, 2) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"], order_base=0)
        b.rebase(123456789)
        _assert_same(b.finalize(), want)


@pytest.mark.parametrize("world,mode", [(1, "diploid"), (2, "diploid"), (3, "diploid"), (4, "heavy"), (3, "empty-rank")])
def test_peer_memory_exchange_single_gpu(native, world, mode):
    """The exchange of the multi-GPU path - dispatch by key, owner merge, dispatch by first occurrence, slices
    ordered over the rank's own positions with rows from the LOCAL context - with the ranks emulated on ONE GPU
    (arenas in the same process instead of IPC mappings).  The slices concatenated are the oracle's matrices."""
    from alntools_b200 import synth, multi_gpu
    if mode == "heavy":
        cols, nt, nh = synth.make_columns(6000, 3000, 8, seed=43, mode="heavy", dup_rate=0.02), 3000, 8
    else:
        cols, nt, nh = synth.make_columns(120000, 4000, 2, seed=41, mode="diploid", dup_rate=0.02), 4000, 2
    rg, tg, hp = cols["read_group"], cols["target_idx"], cols["hap_idx"]
    want = _oracle(cols)
    cuts = multi_gpu.shard_bounds(rg, world)
    if mode == "empty-rank":
        cuts[1] = cuts[2]                                        # rank 1 holds nothing
    locals_, owners = [], []
    for r in range(world):
        a, b = cuts[r], cuts[r + 1]
        lb = native.EcBuilder(nt, nh, alignments_hint=max(b - a, 1))
        if b > a:
            lb.push(np.ascontiguousarray(rg[a:b]), np.ascontiguousarray(tg[a:b]), np.ascontiguousarray(hp[a:b]), order_base=a)
        locals_.append(lb)
        owners.append(native.EcBuilder(nt, nh, alignments_hint=len(rg)))
    cap_ec = 2 * len(want[3]) + 64
    bases = [ob.arena_create(cap_ec)[1] for ob in owners]
    spans = [lb.export_to_arenas(bases, cap_ec) for lb in locals_]
    for ob in owners:
        ob.import_arena()
        ob.arena_reset()
    lo, hi = [s[0] for s in spans], [s[1] for s in spans]
    assert [h > l for l, h in zip(lo, hi)] == [cuts[r + 1] > cuts[r] for r in range(world)]
    for ob in owners:
        ob.order_dispatch(bases, cap_ec, lo, hi)
    at = 0
    for r, ob in enumerate(owners):
        sl = ob.order_build(locals_[r], lo[r], hi[r])
        a, b = at, at + sl["n_ec"]
        assert np.array_equal(sl["a_indptr"].cpu().numpy(), want[0][a:b + 1] - want[0][a])
        assert np.array_equal(sl["a_indices"].cpu().numpy(), want[1][want[0][a]:want[0][b]])
        assert np.array_equal(sl["a_data"].cpu().numpy(), want[2][want[0][a]:want[0][b]])
        assert np.array_equal(sl["n_data"].cpu().numpy(), want[3][a:b])
        at = b
    assert at == len(want[3])
    for b in locals_ + owners:
        b.close()


def test_randomised_read_shapes_and_launch_geometry(native):
    """Many small random inputs against the oracle: read lengths around the 32-alignment window and the
    8-alignment shuffle-de-dup limit, heavy duplication, tiny target spaces (hot keys), and random work
    chunk lengths / grids / cache settings, so that chunk, window and batch boundaries fall everywhere."""
    rng = np.random.default_rng(2024)
    length_pools = [
        [1], [1, 2], [1, 2, 3, 4], [7, 8, 9], [1, 8, 9, 16, 17], [30, 31, 32, 33, 34], [1, 31, 32, 33, 63, 64, 65],
        [1, 2, 3, 100, 200], [1, 1, 1, 1, 1500],
    ]
    for case in range(48):
        pool = length_pools[case % len(length_pools)]
        n_reads = int(rng.integers(1, 4000))
        lens = rng.choice(pool, n_reads)
        n_targets = int(rng.choice([1, 3, 50, 5000]))
        n_haps = int(rng.choice([1, 2, 8]))
        rg = np.repeat(np.arange(n_reads, dtype=np.int32) * 3 + 5, lens)      # any increasing labels
        n = len(rg)
        tg = rng.integers(0, n_targets, n).astype(np.int32)
        hp = rng.integers(0, n_haps, n).astype(np.int32)
        if case % 3 == 0:                                                     # runs of verbatim duplicates
            rep = rng.integers(0, 4, n) == 0
            tg[1:][rep[1:]] = tg[:-1][rep[1:]]
            hp[1:][rep[1:]] = hp[:-1][rep[1:]]
        cols = {"read_group": rg, "target_idx": tg, "hap_idx": hp}
        opts = {"chunk_len": int(rng.choice([0, 32, 64, 160, 1024])), "grid_ctas": int(rng.choice([0, 1, 2, 7])),
                "hot_cache": int(rng.integers(0, 2))}
        if case % 5 == 0:
            opts["table_slots"] = 1024                                        # growth + replay
        got, _ = _run(native, cols, n_targets, n_haps, **opts)
        _assert_same(got, _oracle(cols))


def test_key_verification_option_finds_no_collision(native):
    """ECB_OPT_VERIFY_KEYS re-derives every read's element set and compares it with its EC's row: on
    real-shaped inputs it must pass (no 128-bit key collision) and leave the result unchanged."""
    from alntools_b200 import synth
    for n_reads, n_targets, n_haps, mode, dup in ((60000, 3000, 2, "diploid", 0.05), (4000, 500, 8, "heavy", 0.02)):
        cols = synth.make_columns(n_reads, n_targets, n_haps, seed=9, mode=mode, dup_rate=dup)
        got, _ = _run(native, cols, n_targets, n_haps, verify_keys=1)
        _assert_same(got, _oracle(cols))
