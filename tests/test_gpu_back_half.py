"""The back half of the EC build: the single-pass device scan (ecb_scan.cuh) and the id-ordered finalize
(ecb_finalize.cuh: rank, then one emit pass that scans the row lengths and copies the rows in tiles).

The scan is reached through finalize's rank of the first-occurrence bitmap: the order_base of a second push sets the
bitmap's length in words, so the scan runs at a chosen number of items around its tile size.  Every result is
compared with the C oracle."""
import numpy as np
import pytest

from oracle import c_oracle

pytestmark = pytest.mark.gpu

SCAN_BLOCK = 256 * 16     # items per scan tile (ecb_scan.cuh)
EMIT_TILE = 256 * 4       # ids per emit tile (ecb_finalize.cuh)
N_TARGETS, N_HAPS = 40000, 4


@pytest.fixture(scope="module")
def native(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")
    from alntools_b200 import _native
    _native.load_library()
    return _native


def _oracle(cols):
    return c_oracle.ec_from_columns(cols["read_group"], cols["target_idx"], cols["hap_idx"])


def _assert_same(got, want):
    indptr, indices, data, counts, n_reads = want
    assert got["n_reads"] == n_reads
    assert got["n_ec"] == len(counts)
    assert np.array_equal(got["a_indptr"], indptr)
    assert np.array_equal(got["a_indices"], indices)
    assert np.array_equal(got["a_data"], data)
    assert np.array_equal(got["n_indptr"], [0, len(counts)])
    assert np.array_equal(got["n_indices"], np.arange(len(counts)))
    assert np.array_equal(got["n_data"], counts)


def _distinct(n_reads, first=0):
    """n_reads single-alignment reads, every one its own EC."""
    i = np.arange(first, first + n_reads)
    return {"read_group": i.astype(np.int32), "target_idx": (i % N_TARGETS).astype(np.int32),
            "hap_idx": ((i // N_TARGETS) % N_HAPS).astype(np.int32)}


def _rows(lengths, seed):
    """One read per length; a read of k alignments on k distinct targets gives a row of k entries.  Short reads of
    1..8 alignments are repeated, so their ECs also count several reads."""
    rng = np.random.default_rng(seed)
    rg, tg, hp = [], [], []
    for r, k in enumerate(lengths):
        rg.append(np.full(k, r))
        tg.append((rng.integers(0, N_TARGETS) + np.arange(k)) % N_TARGETS if k > 8 else rng.integers(0, 50, k))
        hp.append(rng.integers(0, N_HAPS, k))
    return {"read_group": np.concatenate(rg).astype(np.int32), "target_idx": np.concatenate(tg).astype(np.int32),
            "hap_idx": np.concatenate(hp).astype(np.int32)}


def _concat(a, b):
    rg_b = b["read_group"].astype(np.int64) + int(a["read_group"].max()) + 1
    return {"read_group": np.concatenate([a["read_group"], rg_b.astype(np.int32)]),
            "target_idx": np.concatenate([a["target_idx"], b["target_idx"]]),
            "hap_idx": np.concatenate([a["hap_idx"], b["hap_idx"]])}


@pytest.mark.parametrize("n_ec", [1, 2, EMIT_TILE - 1, EMIT_TILE, EMIT_TILE + 1, 3 * EMIT_TILE + 5, 128 * 33 + 7])
def test_emit_tile_edges(native, n_ec):
    cols = _distinct(n_ec)
    with native.EcBuilder(N_TARGETS, N_HAPS) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
        _assert_same(b.finalize(), _oracle(cols))


def test_rows_straddle_warps_and_tiles(native):
    """Rows of 1, 8, 9, 33, 1024 and 16384 entries and a deferred read of more than 16384 alignments, placed so that
    long rows start and end inside warps and cross emit tiles."""
    rng = np.random.default_rng(5)
    lengths = [int(x) for x in rng.integers(1, 9, 6000)]
    for j, k in enumerate([1, 8, 9, 33, 1024, 16384, 20000, 9, 33, 1024, 16384, 8, 1]):
        lengths.insert(97 + j * 431, k)
    cols = _rows(lengths, 6)
    with native.EcBuilder(N_TARGETS, N_HAPS, max_read=0) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
        got = b.finalize()
        assert b.stats()["long_reads"] == 1
    _assert_same(got, _oracle(cols))


@pytest.mark.parametrize("words", [70, SCAN_BLOCK - 1, SCAN_BLOCK, SCAN_BLOCK + 1, 2 * SCAN_BLOCK + 1, 100_000_003])
def test_rank_scan_lengths(native, words):
    """The popcount scan of the first-occurrence bitmap at `words` words: two pushes, the second placed so that the
    alignments span 32 * (words - 1) positions."""
    a, bb = _distinct(1500), _distinct(700, first=1500)
    n_a, n_b = len(a["read_group"]), len(bb["read_group"])
    span = 32 * (words - 1)
    base_b = max(n_a, span - n_b)
    with native.EcBuilder(N_TARGETS, N_HAPS) as b:
        b.push(a["read_group"], a["target_idx"], a["hap_idx"], order_base=0)
        b.push(bb["read_group"], bb["target_idx"], bb["hap_idx"], order_base=base_b)
        _assert_same(b.finalize(), _oracle(_concat(a, bb)))


def test_replayed_push_gets_its_rows(native):
    """A push that overflows a tiny table: the ECs the replay claims get their rows like the others."""
    from alntools_b200 import synth
    cols = synth.make_columns(60000, 5000, 2, seed=31, mode="diploid", dup_rate=0.01)
    with native.EcBuilder(5000, 2, table_slots=1024) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
        got = b.finalize()
        st = b.stats()
    assert st["overflow_reads"] > 0 and st["table_grows"] > 0
    want = _oracle(cols)
    assert np.array_equal(got["a_indptr"], want[0])
    assert np.array_equal(got["a_indices"], want[1])
    assert np.array_equal(got["a_data"], want[2])
    assert np.array_equal(got["n_data"], want[3])


def test_overlapping_order_bases_then_reuse(native):
    """Overlapping order_base ranges leave ids no EC takes: finalize reports the overlap, and the context gives the
    right result after a reset."""
    from alntools_b200 import synth
    cols = synth.make_columns(50000, 5000, 2, seed=32, mode="diploid")
    with native.EcBuilder(5000, 2) as b:
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"], order_base=0)
        b.push(cols["read_group"], (cols["target_idx"] + 1) % 5000, cols["hap_idx"], order_base=10)
        with pytest.raises(native.EcbError, match="overlap"):
            b.finalize()
        b.reset()
        b.push(cols["read_group"], cols["target_idx"], cols["hap_idx"])
        want = _oracle(cols)
        got = b.finalize()
        assert np.array_equal(got["a_indptr"], want[0])
        assert np.array_equal(got["a_indices"], want[1])
        assert np.array_equal(got["a_data"], want[2])
        assert np.array_equal(got["n_data"], want[3])
