"""What bin_utils.merge_ec_files must produce, stated in Python, for the merge tests.

An EC is a distinct A row: a tuple of (target, mask) pairs.  A dict maps every row to its merged id, taken in the order
of first appearance over (file index, row id in that file); every file's columns follow in order, their entries moved
to the merged ids of their rows, zeros dropped, ids ascending in a column."""
import numpy as np

from alntools_b200 import bin_utils
import samples_oracle as so


def rows_of(a):
    """(indptr, indices, data) of an A matrix -> its rows as tuples of (target, mask)."""
    indptr, indices, data = (np.asarray(x).tolist() for x in a)
    return [tuple(zip(indices[indptr[e]:indptr[e + 1]], data[indptr[e]:indptr[e + 1]])) for e in range(len(indptr) - 1)]


def a_csr(rows):
    indptr = np.cumsum([0] + [len(r) for r in rows]).astype(np.int32)
    pairs = [p for r in rows for p in r]
    return (indptr, np.asarray([t for t, _ in pairs], np.int32), np.asarray([m for _, m in pairs], np.int32))


def merge_statement(files):
    """files: per file (rows, n) with rows a list of row tuples and n = (indptr, indices, data), N as CSC over those
    rows.  -> (merged rows in id order, N of the merge as (indptr, indices, data))."""
    ids = {}
    for rows, _ in files:
        for row in rows:
            ids.setdefault(row, len(ids))
    columns = []
    for rows, n in files:
        indptr, indices, data = (np.asarray(x).tolist() for x in n)
        for s in range(len(indptr) - 1):
            col = {}
            for i in range(indptr[s], indptr[s + 1]):
                if data[i]:
                    e = ids[rows[indices[i]]]
                    col[e] = col.get(e, 0) + data[i]
            columns.append(col)
    return list(ids), so.n_csc(columns)


def merge_files(paths):
    """The statement applied to EC files.  -> dict(a, n, samples) as bin_utils.ecload_arrays gives them."""
    loaded = [bin_utils.ecload_arrays(p) for p in paths]
    rows, n = merge_statement([(rows_of(d["a"]), d["n"]) for d in loaded])
    return {"a": a_csr(rows), "n": n, "samples": [s for d in loaded for s in d["samples"]]}


def random_file(rng, pool, n_rows, n_cols, max_count=5):
    """An EC file's matrices: n_rows distinct rows drawn from `pool` (row tuples) in random order, and n_cols columns
    with random counts (some entries explicit zeros, some rows without any entry).  -> (a, n)."""
    pick = rng.choice(len(pool), size=n_rows, replace=False)
    rows = [pool[i] for i in pick]
    cols = []
    for _ in range(n_cols):
        k = int(rng.integers(0, n_rows + 1))
        idx = np.sort(rng.choice(n_rows, size=k, replace=False))
        cols.append((idx, rng.integers(0, max_count + 1, size=k)))
    indptr = np.cumsum([0] + [len(i) for i, _ in cols]).astype(np.int32)
    n = (indptr, np.concatenate([i for i, _ in cols] + [np.zeros(0, np.int64)]).astype(np.int32),
         np.concatenate([v for _, v in cols] + [np.zeros(0, np.int64)]).astype(np.int32))
    return a_csr(rows), n
