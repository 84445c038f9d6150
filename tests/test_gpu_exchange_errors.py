"""Caller errors that reach the slice build of both multi-GPU exchanges, with the ranks emulated on ONE GPU (arenas in
the same process instead of IPC mappings, as in test_gpu_parity.py and test_gpu_cells_exchange.py).  Each comes back as
EcbError with its message before any row is copied.  The same owner then runs one correct exchange, whose slices
must equal the oracle: the failed call left the device and the contexts usable."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ERR_INVALID, ERR_LIMIT = -1, -4          # ECB_ERR_INVALID, ECB_ERR_LIMIT (include/ecb200.h)
NT = 16

# A: ECs {1, 2}, {3}, {4, 5, 6}, {10} first at positions 0, 2, 4, 7; B: ECs {7}, {8, 9}, {11} first at 0, 1, 5.
# The per-cell pushes drop their last read, and with it EC {10} or {11}.
A = [(1, 2), (3,), (1, 2), (4, 5, 6), (10,)]
B = [(7,), (8, 9), (7,), (11,)]
UNSEEN = [(12,), (13,), (14,), (12,), (15,)]    # as many ECs as A, none of them A's


@pytest.fixture(scope="module")
def native(built):
    import torch
    assert torch.cuda.is_available(), "these tests need a B200"
    from alntools_b200 import _native
    _native.load_library()
    return _native


def _cols(reads):
    """reads: target tuples -> int32 columns, haplotype 0, read i in cell i % 3."""
    lens = [len(t) for t in reads]
    rg = np.repeat(np.arange(len(reads), dtype=np.int32), lens)
    return {"read_group": rg, "target_idx": np.asarray([t for ts in reads for t in ts], dtype=np.int32),
            "hap_idx": np.zeros(len(rg), np.int32), "cell_idx": (rg % 3).astype(np.int32)}


def _local(native, pushes, nt=NT, cells=False):
    """A LOCAL context with pushes [(columns, order_base)] (per-cell: drop_last_group, as convert_files_rank)."""
    b = native.EcBuilder(nt, 1, with_cells=cells)
    for c, base in pushes:
        b.push(c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"] if cells else None, order_base=base,
               drop_last_group=cells)
    return b


def _np(sl):
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in sl.items()}


def _single(native, owners, bases, cap, ranks, nt=NT, build_local=None, span=None):
    """One single-sample exchange: ranks[r] = rank r's pushes.  The slices are built against build_local (default:
    each rank's own local context) over `span` positions from the shard's start (default: the whole shard)."""
    locals_ = [_local(native, pushes, nt) for pushes in ranks]
    try:
        for ob in owners:
            ob.reset()
            ob.arena_reset()
        spans = [lb.export_to_arenas(bases, cap) for lb in locals_]
        for ob in owners:
            ob.import_arena()
            ob.arena_reset()
        lo, hi = [s[0] for s in spans], [s[1] for s in spans]
        for ob in owners:
            ob.order_dispatch(bases, cap, lo, hi)
        return [_np(ob.order_build(build_local or locals_[r], lo[r], hi[r] if span is None else lo[r] + span))
                for r, ob in enumerate(owners)]
    finally:
        for b in locals_:
            b.close()


def _assert_single_oracle(slices, cols):
    from oracle import c_oracle
    indptr, indices, data, counts, _ = c_oracle.ec_from_columns(cols["read_group"], cols["target_idx"], cols["hap_idx"])
    at = 0
    for sl in slices:
        a, b = at, at + sl["n_ec"]
        assert np.array_equal(sl["a_indptr"], indptr[a:b + 1] - indptr[a])
        assert np.array_equal(sl["a_indices"], indices[indptr[a]:indptr[b]])
        assert np.array_equal(sl["a_data"], data[indptr[a]:indptr[b]])
        assert np.array_equal(sl["n_data"], counts[a:b])
        at = b
    assert at == len(counts)


def _single_ok(native, owners, bases, cap, reads, nt=NT):
    """A correct exchange on the same owners: `reads` sharded over the ranks, against the oracle."""
    from alntools_b200 import multi_gpu
    cols = _cols(reads)
    cuts = multi_gpu.shard_bounds(cols["read_group"], len(owners))
    ranks = [[({k: np.ascontiguousarray(v[a:b]) for k, v in cols.items()}, a)] if b > a else []
             for a, b in zip(cuts[:-1], cuts[1:])]
    _assert_single_oracle(_single(native, owners, bases, cap, ranks, nt), cols)


def _cells(native, owner, pushes, build_local=None, span=None):
    """One per-cell exchange at world 1 (every cell kept), the arena sized from the exact counts."""
    local = _local(native, pushes, cells=True)
    try:
        owner.reset()
        key, total = local.cells_summary(None, 3)
        n_samples, order = local.cells_order(key, total, 0, None, 1)
        order = order.cpu().numpy()
        counts = local.cells_dispatch_counts(1).tolist()
        cap_ec, cap_pairs = max(1, counts[0]), max(1, counts[1])
        base = owner.cells_arena_create(cap_ec, cap_pairs)[1]
        lo, hi = local.cells_export_to_arenas([base], cap_ec, cap_pairs)
        owner.cells_import_arena()
        owner.arena_reset()
        owner.cells_order_dispatch([base], cap_ec, cap_pairs, [lo], [hi])
        sl = _np(owner.cells_order_build(build_local or local, lo, hi if span is None else lo + span, n_samples))
        return sl, order
    finally:
        local.close()


def _cells_ok(native, owner):
    from oracle import ec_oracle
    a, b = _cols(A), _cols(B)
    sl, order = _cells(native, owner, [(a, 0), (b, len(a["read_group"]))])
    want = ec_oracle.ec_from_columns_cells([(c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"], True)
                                            for c in (a, b)], 0)
    assert np.array_equal(sl["a_indptr"], want["a_indptr"])
    assert np.array_equal(sl["a_indices"], want["a_indices"])
    assert np.array_equal(sl["a_data"], want["a_data"])
    assert np.array_equal(np.concatenate([[0], np.cumsum(sl["n_col_counts"])]), want["n_indptr"])
    assert np.array_equal(sl["n_indices"], want["n_indices"])
    assert np.array_equal(sl["n_data"], want["n_data"])
    assert np.array_equal(order, want["cell_order"])


def _raises(code, message, fn):
    from alntools_b200 import _native
    with pytest.raises(_native.EcbError) as exc:
        fn()
    assert exc.value.code == code
    assert str(exc.value) == "libecb200 error %d: %s" % (code, message)


CASES = {   # name: (message, keyword arguments of the failing exchange besides its pushes)
    "shared_first_read": ("second dispatch: two ECs share a first read", {}),
    "unseen_ec": ("second dispatch: an EC arrived that the local context has never seen", {"unseen": True}),
    # a shard of 4 positions still has room for A's ECs, but not for its EC first at position 4
    "outside_shard": ("second dispatch: a record outside the shard's positions arrived", {"span": 4}),
}


def _pushes(name):
    a = _cols(A)
    return [(a, 0), (_cols(B), 0)] if name == "shared_first_read" else [(a, 0)]


@pytest.mark.parametrize("name", list(CASES))
def test_single_sample_build_reports_the_caller_error(native, name):
    message, kw = CASES[name]
    owner = native.EcBuilder(NT, 1)
    unseen = _local(native, [(_cols(UNSEEN), 0)]) if kw.get("unseen") else None
    try:
        bases = [owner.arena_create(64)[1]]
        _raises(ERR_INVALID, message, lambda: _single(native, [owner], bases, 64, [_pushes(name)], build_local=unseen,
                                                      span=kw.get("span")))
        _single_ok(native, [owner], bases, 64, A + B)
    finally:
        for b in (owner, unseen):
            if b is not None:
                b.close()


@pytest.mark.parametrize("name", list(CASES))
def test_cells_build_reports_the_caller_error(native, name):
    message, kw = CASES[name]
    owner = native.EcBuilder(NT, 1)
    unseen = _local(native, [(_cols(UNSEEN), 0)], cells=True) if kw.get("unseen") else None
    try:
        _raises(ERR_INVALID, message, lambda: _cells(native, owner, _pushes(name), build_local=unseen, span=kw.get("span")))
        _cells_ok(native, owner)
    finally:
        for b in (owner, unseen):
            if b is not None:
                b.close()


def test_single_sample_import_reports_a_small_arena(native):
    with native.EcBuilder(NT, 1) as owner:
        bases = [owner.arena_create(2)[1]]
        _raises(ERR_LIMIT, "exchange arena too small: 3 records arrived, capacity 2",
                lambda: _single(native, [owner], bases, 2, [[(_cols(A[:4]), 0)]]))
        _single_ok(native, [owner], bases, 2, A[:3])     # two ECs


def test_single_sample_build_reports_a_small_arena(native):
    """Rank 0 holds the first occurrence of all n ECs, rank 1 one repeat.  Dispatch 1 splits the ECs between the
    owners by key, about n/2 each, which the arenas of 0.6 n records take; dispatch 2 sends all n to rank 0, whose
    arena then lacks room for their 24-byte records (3 n words against 2.4 n)."""
    n, cap = 10_000, 6_000
    owners = [native.EcBuilder(n, 1) for _ in range(2)]
    try:
        bases = [ob.arena_create(cap)[1] for ob in owners]
        rank0 = {"read_group": np.arange(n, dtype=np.int32), "target_idx": np.arange(n, dtype=np.int32),
                 "hap_idx": np.zeros(n, np.int32), "cell_idx": np.zeros(n, np.int32)}
        rank1 = {k: v[:1].copy() for k, v in rank0.items()}
        _raises(ERR_LIMIT, "exchange arena too small for the second dispatch",
                lambda: _single(native, owners, bases, cap, [[(rank0, 0)], [(rank1, n)]], nt=n))
        rng = np.random.default_rng(3)
        _single_ok(native, owners, bases, cap, [tuple(rng.choice(n, int(k), replace=False)) for k in rng.integers(1, 4, 3000)],
                   nt=n)
    finally:
        for b in owners:
            b.close()
