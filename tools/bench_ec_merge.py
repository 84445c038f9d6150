"""Merging EC files (bin_utils.merge_ec_files, ecb_push_ecs, ecb_sample_append).

  files    bench.py's bam_e2e sample (8 M cfg2-shaped reads) split into 8 BAM files as bench_samples.split splits it:
           convert_samples of the 8 files, the 8 convert() calls, and merge_ec_files of their outputs, alternating,
           `--runs` passes each; wall times, the merge's breakdown (reading, pushing, finalize, writing), the device
           time from the builder's stats, and whether the merged and the joint file have one sha256.
  scale    `--scale-files` EC files of `--scale-ecs` ECs each, half of every file's rows shared with the first file and
           half its own, built with numpy (row j is a distinct set by construction: targets j >> 10 and 2^17 + (j & 1023),
           every third row a third target; random masks over 2 haplotypes), written with ecsave2_arrays and merged;
           ECs/s and A entries/s of the pushes from their device time, the exact check's share of it, and the Python
           statement (tests/merge_oracle.py) on the first `--statement-files` files as a CPU reference.
  ab       bench.py's default workload (cfg2_diploid_30M, one GPU, no CPU arm) on the parent's library (--parent-lib)
           and the tree's, alternating: the read path must not pay for the merge.

Prints one JSON document with the GPU's name, power limit and max SM clock (read in the same run) and writes it to
--out.

    python tools/bench_ec_merge.py --parent-lib /path/to/parent/libecb200.so --out profiles/r9_ec_merge.json
"""
import argparse
import hashlib
import json
import os
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

from alntools_b200 import _native, bam_utils, bin_utils, synth  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402
from bench_samples import FILES, WL, run_ab, split  # noqa: E402


def _sha(path):
    with open(path, "rb") as fh:
        return hashlib.sha256(fh.read()).hexdigest()


def _merge_stats(ins, out):
    """merge_ec_files with the builder's stats of the run (the builder is made inside the call)."""
    seen = {}
    real = _native.EcBuilder

    class Watched(real):
        def finalize_samples(self, copy=True):
            res = real.finalize_samples(self, copy)
            seen.update(self.stats())
            return res

    _native.EcBuilder = Watched
    try:
        summary = bin_utils.merge_ec_files(ins, out)
    finally:
        _native.EcBuilder = real
    return summary, seen


def run_files(paths, tmp, runs):
    out = {"joint_s": [], "converts_s": [], "merge_s": [], "merge_breakdown_s": [], "merge_device": [], "same_sha256": []}
    ecs = [os.path.join(tmp, "one%d.bin" % j) for j in range(len(paths))]
    for _ in range(runs):
        t0 = time.perf_counter()
        bam_utils.convert_samples(paths, os.path.join(tmp, "joint.bin"))
        out["joint_s"].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        for p, e in zip(paths, ecs):
            bam_utils.convert(p, e, None)
        out["converts_s"].append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        summary, st = _merge_stats(ecs, os.path.join(tmp, "merged.bin"))
        out["merge_s"].append(time.perf_counter() - t0)
        out["merge_breakdown_s"].append(summary["seconds"])
        out["merge_device"].append({"ec_ms": st["ec_ms"], "ec_check_ms": st["ec_check_ms"], "sample_ms": st["sample_ms"],
                                    "finalize_ms": st["finalize_ms"], "ec_rows": st["ec_rows"],
                                    "ec_claimed": st["ec_claimed"]})
        out["same_sha256"].append(_sha(os.path.join(tmp, "merged.bin")) == _sha(os.path.join(tmp, "joint.bin")))
    out["n_ec"], out["nnz_n"] = summary["n_ec"], summary["nnz_n"]
    out["ec_file_bytes"] = [os.path.getsize(e) for e in ecs]
    out["summary"] = {k: float(np.median(out[k])) for k in ("joint_s", "converts_s", "merge_s")}
    out["summary"]["converts_plus_merge_s"] = out["summary"]["converts_s"] + out["summary"]["merge_s"]
    return out


def scale_file(k, n_ec, rng):
    """A, N of scale file k: rows [0, n_ec/2) of the shared pool and n_ec/2 rows of its own, in random order."""
    half = n_ec // 2
    ids = np.concatenate([np.arange(half, dtype=np.int64), (k + 1) * half + np.arange(n_ec - half, dtype=np.int64)])
    if k == 0:
        ids = np.arange(n_ec, dtype=np.int64)
    ids = ids[rng.permutation(len(ids))]
    third = (ids % 3 == 0)
    lens = 2 + third.astype(np.int64)
    indptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
    z = int(indptr[-1])
    indices = np.empty(z, np.int32)
    starts = indptr[:-1].astype(np.int64)
    indices[starts] = ids >> 10
    indices[starts + 1] = (1 << 17) + (ids & 1023)
    indices[starts[third] + 2] = (1 << 17) + 1024 + (ids[third] % 7) * 1000
    data = np.empty(z, np.int32)
    data[starts] = 1 + (ids % 3).astype(np.int32)      # masks are a function of the row: one row is one set
    data[starts + 1] = 1 + ((ids >> 2) % 3).astype(np.int32)
    data[starts[third] + 2] = 1 + ((ids[third] >> 4) % 3).astype(np.int32)
    cnt = rng.integers(1, 50, size=n_ec).astype(np.int32)
    n = (np.array([0, n_ec], np.int32), np.arange(n_ec, dtype=np.int32), cnt)
    return (indptr, indices, data), n


def run_scale(n_files, n_ec, statement_files, tmp):
    import merge_oracle as mo
    n_targets = 1 << 18
    paths, files = [], []
    rng = np.random.default_rng(9)
    a_entries = 0
    for k in range(n_files):
        a, n = scale_file(k, n_ec, rng)
        a_entries += len(a[1])
        paths.append(os.path.join(tmp, "scale%d.bin" % k))
        bin_utils.ecsave2_arrays(paths[-1], ["A", "B"], None, None, ["s%d" % k], a, n,
                                 target_section=_targets(n_targets), n_targets=n_targets)
        if k < statement_files:
            files.append((a, n))
    t0 = time.perf_counter()
    summary, st = _merge_stats(paths, os.path.join(tmp, "scale_merged.bin"))
    wall = time.perf_counter() - t0
    entries = sum(int(os.path.getsize(p)) for p in paths)
    out = {"files": n_files, "ecs_per_file": n_ec, "merged_n_ec": summary["n_ec"], "merged_nnz_a": summary["nnz_a"],
           "wall_s": wall, "breakdown_s": summary["seconds"], "input_bytes": entries,
           "push_device_ms": st["ec_ms"], "check_device_ms": st["ec_check_ms"], "append_device_ms": st["sample_ms"],
           "finalize_device_ms": st["finalize_ms"], "ec_rows": st["ec_rows"]}
    out["push_rows_per_s"] = st["ec_rows"] / (st["ec_ms"] / 1e3)
    out["push_a_entries_per_s"] = a_entries / (st["ec_ms"] / 1e3)
    out["input_a_entries"] = a_entries
    out["new_row_entries"] = st["row_entries"]
    out["check_share_of_push"] = st["ec_check_ms"] / st["ec_ms"]
    if files:
        t0 = time.perf_counter()
        rows, n = mo.merge_statement([(mo.rows_of(a), n) for a, n in files])
        out["statement_files"] = len(files)
        out["statement_s"] = time.perf_counter() - t0
        out["statement_rows_per_s"] = sum(len(a[0]) - 1 for a, _ in files) / out["statement_s"]
    return out


def _targets(n_targets):
    import struct
    rec = [struct.pack("<i", 1) + b"t" + struct.pack("<ii", 1000, 1000)]
    return b"".join(rec * n_targets)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=8_000_000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--scale-files", type=int, default=64)
    ap.add_argument("--scale-ecs", type=int, default=4_000_000)
    ap.add_argument("--statement-files", type=int, default=8)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--ab-runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--skip", default="", help="comma-separated parts not to run (files, scale, ab)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    skip = set(filter(None, args.skip.split(",")))
    doc = {"gpu": gpu_info(0), "reads": args.reads, "files": FILES}

    def save():   # after every part, so that the parts measured so far survive an interrupted run
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(json.dumps(doc) + "\n")

    with tempfile.TemporaryDirectory(prefix="bench_ec_merge_") as tmp:
        if "files" not in skip:
            cols = synth.make_columns(args.reads, WL["n_targets"], WL["n_haps"], WL["seed"] + 1000, mode=WL["mode"])
            paths = []
            for i, p in enumerate(split(cols, FILES)):
                paths.append(os.path.join(tmp, "part%d.bam" % i))
                synth.columns_to_bam(paths[-1], p, WL["n_targets"], WL["n_haps"])
            del cols
            doc["files_run"] = run_files(paths, tmp, args.runs)
            save()
        if "scale" not in skip:
            doc["scale_run"] = run_scale(args.scale_files, args.scale_ecs, args.statement_files, tmp)
            save()
    if args.parent_lib and "ab" not in skip:
        doc["ab"] = run_ab(args.parent_lib, args.ab_runs, args.steps, args.warmup)
        save()
    print(json.dumps(doc))

if __name__ == "__main__":
    main()
