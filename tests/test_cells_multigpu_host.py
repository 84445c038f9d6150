"""Host parts of the multi-GPU per-cell convert: the file partition, the merge of the ranks' cell names into global
ids, and the EC file written in slices by several ranks (byte-identical to the goldens)."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases


def test_partition_files_contiguous_balanced():
    from alntools_b200.bam_utils_multisample import partition_files
    rng = np.random.default_rng(5)
    for _ in range(200):
        n = int(rng.integers(1, 30))
        world = int(rng.integers(1, 12))
        sizes = rng.integers(1, 1000, n).tolist()
        cuts = partition_files(sizes, world)
        assert len(cuts) == world + 1 and cuts[0] == 0 and cuts[-1] == n
        assert all(a <= b for a, b in zip(cuts, cuts[1:]))             # contiguous runs, in order
        total, biggest = sum(sizes), max(sizes)
        for r in range(world):
            assert sum(sizes[cuts[r]:cuts[r + 1]]) <= total / world + biggest
    # equal sizes split evenly; more ranks than files leave ranks empty
    assert partition_files([10] * 8, 4) == [0, 2, 4, 6, 8]
    cuts = partition_files([5, 5], 4)
    assert cuts[0] == 0 and cuts[-1] == 2 and sum(b > a for a, b in zip(cuts, cuts[1:])) == 2


def test_merge_cell_names_is_one_first_appearance_pass():
    from alntools_b200.bam_utils_multisample import merge_cell_names
    rng = np.random.default_rng(9)
    for _ in range(100):
        pool = ["c%d" % i for i in range(int(rng.integers(1, 40)))]
        lists = []
        for _r in range(int(rng.integers(1, 6))):
            k = int(rng.integers(0, len(pool) + 1))
            lists.append(list(dict.fromkeys(rng.choice(pool, k).tolist())))   # a rank's names are distinct
        names, maps = merge_cell_names(lists)
        want = list(dict.fromkeys(n for lst in lists for n in lst))
        assert names == want
        for lst, m in zip(lists, maps):
            assert m.dtype == np.int32 and [names[g] for g in m.tolist()] == lst


def _slice_pieces(ec, lo, hi):
    """A rank's pieces of the per-cell matrices for EC ids [lo, hi), as distributed_finalize_cells returns them."""
    a_indptr, a_indices, a_data = ec["a"]
    n_indptr, n_indices, n_data = ec["n"]
    S = len(n_indptr) - 1
    a = (a_indptr[lo:hi + 1] - a_indptr[lo], a_indices[a_indptr[lo]:a_indptr[hi]], a_data[a_indptr[lo]:a_indptr[hi]])
    counts, offset, idx, dat = np.zeros(S, np.int64), np.zeros(S, np.int64), [], []
    for c in range(S):
        rows = n_indices[n_indptr[c]:n_indptr[c + 1]]
        keep = (rows >= lo) & (rows < hi)
        counts[c] = keep.sum()
        offset[c] = (rows < lo).sum()
        idx.append(rows[keep] - lo)
        dat.append(n_data[n_indptr[c]:n_indptr[c + 1]][keep])
    return a, (n_indptr, counts, offset, np.concatenate(idx).astype(np.int32), np.concatenate(dat).astype(np.int32))


@pytest.mark.parametrize("case", golden_cases("multisample"), ids=lambda c: c["name"])
def test_cells_slices_write_the_golden_bytes(case, tmp_path):
    from alntools_b200 import bin_utils
    ec = bin_utils.ecload_arrays(os.path.join(GOLDEN, case["ec"]))
    header = bin_utils.ec_header_bytes(ec["haplotypes"], ec["targets"], ec["lengths"], ec["samples"])
    E = len(ec["a"][0]) - 1
    rng = np.random.default_rng(len(case["name"]))
    for world in (1, 2, 3, 4):
        inner = sorted(rng.integers(0, E + 1, world - 1).tolist())
        if world > 1:
            inner[int(rng.integers(0, world - 1))] = inner[0]      # at least one empty slice
        cuts = [0] + sorted(inner) + [E]
        out = str(tmp_path / ("w%d.bin" % world))
        # the creator first, the others in a shuffled order
        for r in [0] + rng.permutation(np.arange(1, world)).tolist():
            lo, hi = cuts[r], cuts[r + 1]
            a, n = _slice_pieces(ec, lo, hi)
            bin_utils.ecsave2_cells_slice(out, header, E, len(ec["a"][1]), lo, int(ec["a"][0][lo]), *a, *n,
                                          create=(r == 0))
        with open(out, "rb") as fh:
            assert hashlib.sha256(fh.read()).hexdigest() == case["sha256"], (world, cuts)
