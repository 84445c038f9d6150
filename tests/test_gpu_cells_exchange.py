"""The per-cell (multisample) multi-GPU exchange with the ranks emulated on ONE GPU (arenas in the same process
instead of IPC mappings), driven step by step as multi_gpu.distributed_finalize_cells drives it: cell summary,
cell decision, dispatch by key with exact arena sizing, owner merge, dispatch by first occurrence, slice build.
The slices put together must equal the oracle bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

RANK_STRIDE = 1 << 40


@pytest.fixture(scope="module")
def native(built):
    import torch
    assert torch.cuda.is_available(), "these tests need a B200"
    from alntools_b200 import _native
    _native.load_library()
    return _native


def _oracle(files, min_count):
    pushes = [(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], True) for f in files]
    if sum(len(p[0]) for p in pushes) > 100_000:
        from oracle import c_oracle
        return c_oracle.ec_from_columns_cells(pushes, min_count)
    from oracle import ec_oracle
    return ec_oracle.ec_from_columns_cells(pushes, min_count)


def _local_ids(files, rng):
    """A rank's local cell ids: a random permutation of the global ids it holds.  -> (files with local cell
    columns, int32 map local -> global)."""
    held = np.unique(np.concatenate([f["cell_idx"] for f in files])) if files else np.zeros(0, np.int32)
    cell_map = rng.permutation(held).astype(np.int32)
    inv = {int(g): l for l, g in enumerate(cell_map.tolist())}
    lut = np.zeros(int(held.max()) + 1 if len(held) else 1, dtype=np.int32)
    for g, l in inv.items():
        lut[g] = l
    out = [dict(f, cell_idx=np.ascontiguousarray(lut[f["cell_idx"]])) for f in files]
    return out, cell_map


def _exchange(native, rank_files, nt, nh, min_count, n_cells, rng=None, resize=True):
    """Run the exchange over emulated ranks.  rank_files[r]: that rank's files (dicts of int32 columns with
    GLOBAL cell ids).  -> (assembled result dict, info dict)."""
    import torch
    world = len(rank_files)
    rng = rng or np.random.default_rng(0)
    dev = torch.device("cuda", 0)
    locals_, owners, maps = [], [], []
    try:
        for r, files in enumerate(rank_files):
            lfiles, cell_map = _local_ids(files, rng)
            lb = native.EcBuilder(nt, nh, with_cells=True, alignments_hint=0)
            base = r * RANK_STRIDE
            for f in lfiles:
                lb.push(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], order_base=base, drop_last_group=True)
                base += len(f["read_group"])
            locals_.append(lb)
            owners.append(native.EcBuilder(nt, nh))
            maps.append(torch.from_numpy(cell_map).to(dev) if len(cell_map) else None)
        sums = [lb.cells_summary(m, n_cells) for lb, m in zip(locals_, maps)]
        keys_all = torch.cat([k for k, _ in sums])
        totals = sum(t for _, t in sums)
        decided = [lb.cells_order(keys_all, totals, min_count, m, world) for lb, m in zip(locals_, maps)]
        n_samples, cell_order = decided[0]
        for s, o in decided[1:]:
            assert s == n_samples and torch.equal(o, cell_order)           # the same decision everywhere
        cell_order = cell_order.cpu().numpy()                               # (a view of library memory)
        counts = sum(lb.cells_dispatch_counts(world) for lb in locals_).tolist()
        cap_ec, cap_pairs = max(1, max(counts[:world])), max(1, max(counts[world:]))
        bases = [ob.cells_arena_create(cap_ec, cap_pairs)[1] for ob in owners]
        spans = [lb.cells_export_to_arenas(bases, cap_ec, cap_pairs) for lb in locals_]
        for ob in owners:
            ob.cells_import_arena()
        lo, hi = [s[0] for s in spans], [s[1] for s in spans]
        counts2 = sum(ob.cells_dispatch_counts(world, lo, hi) for ob in owners).tolist()
        need_ec, need_pairs = max(counts2[:world]), max(counts2[world:])
        resized = need_ec > cap_ec or need_pairs > cap_pairs
        if resized and resize:
            cap_ec, cap_pairs = max(cap_ec, need_ec), max(cap_pairs, need_pairs)
            bases = [ob.cells_arena_create(cap_ec, cap_pairs)[1] for ob in owners]
        else:
            for ob in owners:
                ob.arena_reset()
        for ob in owners:
            ob.cells_order_dispatch(bases, cap_ec, cap_pairs, lo, hi)
        slices = []
        for r, ob in enumerate(owners):
            sl = ob.cells_order_build(locals_[r], lo[r], hi[r], n_samples)
            slices.append((lo[r], r, {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in sl.items()}))
    finally:
        for b in locals_ + owners:
            b.close()
    # put the slices together in id order (the order of the ranks' shards)
    slices = [s[2] for s in sorted(s for s in slices if s[2]["n_ec"] or s[2]["nnz_n"])]
    a_indptr, a_indices, a_data, at = [np.zeros(1, np.int64)], [], [], 0
    for sl in slices:
        a_indptr.append(sl["a_indptr"][1:].astype(np.int64) + at)
        at += sl["nnz"]
        a_indices.append(sl["a_indices"])
        a_data.append(sl["a_data"])
    cols = [[] for _ in range(n_samples)]
    base = 0
    for sl in slices:
        starts = np.concatenate([[0], np.cumsum(sl["n_col_counts"])])
        for c in range(n_samples):
            s, e = starts[c], starts[c + 1]
            cols[c].append((sl["n_indices"][s:e].astype(np.int64) + base, sl["n_data"][s:e]))
        base += sl["n_ec"]
    n_idx = [np.concatenate([p[0] for p in col]) if col else np.zeros(0) for col in cols]
    n_dat = [np.concatenate([p[1] for p in col]) if col else np.zeros(0) for col in cols]
    got = {"n_ec": base, "a_indptr": np.concatenate(a_indptr), "a_indices": np.concatenate(a_indices),
           "a_data": np.concatenate(a_data), "n_indptr": np.concatenate([[0], np.cumsum([len(x) for x in n_idx])]),
           "n_indices": np.concatenate(n_idx), "n_data": np.concatenate(n_dat), "cell_order": cell_order}
    return got, {"resized": resized, "counts": counts, "counts2": counts2}


def _assert_equal(got, want):
    for k in ("a_indptr", "a_indices", "a_data", "n_indptr", "n_indices", "n_data", "cell_order"):
        assert np.array_equal(np.asarray(got[k], dtype=np.int64), np.asarray(want[k], dtype=np.int64)), k


def _files(total_reads, n_files, nt, nh, seed, cells):
    """Synthetic files with global cell ids drawn from `cells` (an int array)."""
    from alntools_b200 import synth, multi_gpu
    cols = synth.make_columns(total_reads, nt, nh, seed=seed, mode="diploid", n_cells=len(cells), dup_rate=0.02)
    cols["cell_idx"] = np.ascontiguousarray(np.asarray(cells, dtype=np.int32)[cols["cell_idx"]])
    cuts = multi_gpu.shard_bounds(cols["read_group"], n_files) if n_files else [0]
    return [{k: np.ascontiguousarray(cols[k][cuts[i]:cuts[i + 1]]) for k in ("read_group", "target_idx", "hap_idx", "cell_idx")}
            for i in range(n_files)]


def test_cells_exchange_randomised_sweep(native):
    rng = np.random.default_rng(2026)
    for case in range(24):
        world = 1 + case % 4
        n_cells = int(rng.integers(20, 400))
        shared = rng.choice(n_cells, n_cells // 2, replace=False)
        private = np.setdiff1d(np.arange(n_cells), shared)
        priv = np.array_split(rng.permutation(private), world)
        rank_files = []
        for r in range(world):
            n_files = int(rng.integers(0, 4)) if world > 1 else int(rng.integers(1, 4))
            pool = np.concatenate([shared, priv[r]]) if case % 3 else shared
            rank_files.append(_files(int(rng.integers(500, 6000)) * max(n_files, 1), n_files, 300, 4,
                                     seed=1000 + 10 * case + r, cells=pool) if n_files else [])
        files = [f for fl in rank_files for f in fl]
        if not files:
            continue
        read_cells = []
        for f in files:                                                 # reads per cell (last read of a file dropped)
            rg = f["read_group"]
            starts = np.flatnonzero(np.concatenate(([True], rg[1:] != rg[:-1])))[:-1]
            read_cells.append(f["cell_idx"][starts])
        totals = np.bincount(np.concatenate(read_cells), minlength=n_cells)
        min_count = int(rng.choice([0, 1, 2, int(np.median(totals[totals > 0])), int(totals.max()), int(totals.max()) + 1]))
        want = _oracle(files, min_count)
        if len(want["cell_order"]) == 0:                                # the builder refuses where nothing is kept
            from alntools_b200 import _native
            with pytest.raises(_native.EcbError) as exc:
                _exchange(native, rank_files, 300, 4, min_count, n_cells, rng=rng)
            assert exc.value.code == _native.ECB_ERR_EMPTY
            continue
        got, _ = _exchange(native, rank_files, 300, 4, min_count, n_cells, rng=rng)
        assert got["n_ec"] == len(want["a_indptr"]) - 1, case
        _assert_equal(got, want)


def _explicit(reads):
    """reads: list of (targets tuple, cell) -> one file's columns (haplotype 0)."""
    rg, tg, hp, cell = [], [], [], []
    for i, (ts, c) in enumerate(reads):
        for t in ts:
            rg.append(i)
            tg.append(t)
            hp.append(0)
            cell.append(c)
    a = lambda v: np.asarray(v, dtype=np.int32)
    return {"read_group": a(rg), "target_idx": a(tg), "hap_idx": a(hp), "cell_idx": a(cell)}


def test_ec_first_seen_where_its_cells_are_filtered(native):
    """EC (7, 8) first occurs on rank 0 in cell 0, which the minimum count drops; on rank 1 it is kept in cell 1.
    Its id still comes from its first occurrence on rank 0."""
    r0 = _explicit([((1,), 1), ((7, 8), 0), ((2,), 1), ((1,), 1), ((3,), 2)])
    r1 = _explicit([((3,), 1), ((7, 8), 1), ((7, 8), 1), ((2,), 2), ((4,), 2), ((4,), 2), ((9,), 1)])
    want = _oracle([r0, r1], 2)
    got, _ = _exchange(native, [[r0], [r1]], 16, 1, 2, 3)
    _assert_equal(got, want)


def test_cell_first_seen_on_earlier_rank_with_larger_local_key(native):
    """Cell 5 appears late on rank 0 (a large local key there) and at the very first read of rank 1 (key 0): its
    global place comes from rank 0."""
    r0 = _explicit([((1,), 1), ((2,), 2), ((3,), 3), ((4,), 4), ((5,), 5), ((6,), 6)])
    r1 = _explicit([((5,), 5), ((1,), 1), ((2,), 2), ((3,), 3), ((4,), 7), ((4,), 7)])
    want = _oracle([r0, r1], 0)
    got, _ = _exchange(native, [[r0], [r1]], 16, 1, 0, 8)
    _assert_equal(got, want)


def test_skewed_second_dispatch_resizes_the_arena(native):
    """Rank 0's file holds the first occurrence of almost every EC and the cells spread over all ranks, so
    dispatch 2 sends rank 0 about world x one rank's pairs: the arena is re-created from the exact counts.  Kept
    at the dispatch-1 size, the overflow flag makes the build fail instead of losing records."""
    from alntools_b200 import _native
    world = 4
    cells = np.arange(2000)
    base = _files(6000, 1, 200, 2, seed=77, cells=cells)[0]
    rank_files = []
    for r in range(world):
        f = dict(base)
        f["cell_idx"] = np.ascontiguousarray(((base["cell_idx"] + 500 * r) % 2000).astype(np.int32))
        rank_files.append([f])
    files = [fl[0] for fl in rank_files]
    want = _oracle(files, 0)
    got, info = _exchange(native, rank_files, 200, 2, 0, 2000)
    assert info["resized"], info
    _assert_equal(got, want)
    with pytest.raises(_native.EcbError) as exc:
        _exchange(native, rank_files, 200, 2, 0, 2000, resize=False)
    assert "arena too small" in str(exc.value)


def test_no_kept_cell_fails_on_every_rank(native):
    from alntools_b200 import _native
    import torch
    r0 = _explicit([((1,), 0), ((2,), 1), ((3,), 0)])
    r1 = _explicit([((1,), 2), ((2,), 2), ((3,), 1)])
    builders = []
    try:
        for r, f in enumerate((r0, r1)):
            b = native.EcBuilder(8, 1, with_cells=True)
            b.push(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], order_base=r * RANK_STRIDE,
                   drop_last_group=True)
            builders.append(b)
        sums = [b.cells_summary(None, 3) for b in builders]
        keys, totals = torch.cat([k for k, _ in sums]), sum(t for _, t in sums)
        for b in builders:
            with pytest.raises(_native.EcbError) as exc:
                b.cells_order(keys, totals, 100, None, 2)
            assert exc.value.code == _native.ECB_ERR_EMPTY and "no cell reaches the minimum count 100" in str(exc.value)
    finally:
        for b in builders:
            b.close()


def test_world_one_equals_single_gpu_finalize(native):
    files = _files(40000, 3, 500, 4, seed=5, cells=np.arange(300))
    for min_count in (0, 50):
        with native.EcBuilder(500, 4, with_cells=True) as b:
            base = 0
            for f in files:
                b.push(f["read_group"], f["target_idx"], f["hap_idx"], f["cell_idx"], order_base=base, drop_last_group=True)
                base += len(f["read_group"])
            one = b.finalize(min_count)
        got, _ = _exchange(native, [files], 500, 4, min_count, 300)
        _assert_equal(got, one)


def test_cells_exchange_cfg4_scale(native):
    """cfg4's shape at scale: 20 M reads, 50 000 cells, 4 files over 2 emulated ranks, against the C oracle."""
    files = _files(20_000_000, 4, 140_000, 8, seed=4, cells=np.arange(50_000))
    want = _oracle(files, 1000)
    got, _ = _exchange(native, [files[:2], files[2:]], 140_000, 8, 1000, 50_000)
    _assert_equal(got, want)
