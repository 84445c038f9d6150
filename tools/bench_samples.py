"""Several samples in one EC file (bam_utils.convert_samples, ecb_sample_close, ecb_finalize_samples).

  files    bench.py's bam_e2e sample (8 M cfg2-shaped reads) split into 8 files of 1 M reads: the 8 files converted
           jointly (convert_samples) against the same 8 files converted one by one (convert), alternating, `--runs`
           passes each; wall time and alignments/s.  The joint EC file's A and row sums of N are checked against
           convert() of the whole sample.
  close    the same 8 samples pushed from host columns into one context: the device time (CUDA events) and the host
           wall time of every ecb_sample_close, the ECs it went over and its pairs; then ecb_finalize_samples against
           ecb_finalize of the same pushes without closes (finalize_ms), `--reps` times each.
  ab       bench.py's default workload (cfg2_diploid_30M, one GPU, no CPU arm) on the parent's library
           (--parent-lib) and the tree's, alternating: the ordinary path must not pay for the samples.

Prints one JSON document with the GPU's name, power limit and max SM clock (read in the same run) and writes it to
--out.

    python tools/bench_samples.py --parent-lib /path/to/parent/libecb200.so --out profiles/r8_samples.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from alntools_b200 import _native, bam_utils, bin_utils, synth  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402

WL = dict(n_targets=100_000, n_haps=2, mode="diploid", seed=2)   # bench.py's cfg2_diploid_30M
FILES = 8


def split(cols, parts):
    rg = cols["read_group"]
    n_reads = int(rg[-1]) + 1
    out = []
    for i in range(parts):
        lo, hi = np.searchsorted(rg, [n_reads * i // parts, n_reads * (i + 1) // parts])
        out.append({k: np.ascontiguousarray(cols[k][lo:hi]) for k in ("read_group", "target_idx", "hap_idx")})
    return out


def run_files(paths, whole, tmp, runs):
    joint, single = [], []
    valid = 0
    for i in range(runs):
        t0 = time.perf_counter()
        summary = bam_utils.convert_samples(paths, os.path.join(tmp, "joint.bin"))
        joint.append(time.perf_counter() - t0)
        valid = summary["n_alignments"]
        t0 = time.perf_counter()
        for j, p in enumerate(paths):
            bam_utils.convert(p, os.path.join(tmp, "one%d.bin" % j), None)
        single.append(time.perf_counter() - t0)
    bam_utils.convert(whole, os.path.join(tmp, "whole.bin"), None)
    got = bin_utils.ecload_arrays(os.path.join(tmp, "joint.bin"))
    want = bin_utils.ecload_arrays(os.path.join(tmp, "whole.bin"))
    same_a = all(np.array_equal(a, b) for a, b in zip(got["a"], want["a"]))
    sums = np.bincount(got["n"][1], weights=got["n"][2], minlength=len(got["a"][0]) - 1).astype(np.int64)
    same_n = bool(np.array_equal(sums, want["n"][2].astype(np.int64)))
    return {"alignments": int(valid), "joint_s": joint, "one_by_one_s": single,
            "joint_alignments_per_s": valid / float(np.median(joint)),
            "one_by_one_alignments_per_s": valid / float(np.median(single)),
            "joint_n_ec": int(len(got["a"][0]) - 1), "joint_nnz_n": int(len(got["n"][1])),
            "a_equals_whole_file": bool(same_a), "n_row_sums_equal_whole_file": same_n}


def run_close(parts, reps):
    out = {"close": [], "finalize_samples_ms": [], "finalize_ms": []}
    for rep in range(reps + 1):
        with _native.EcBuilder(WL["n_targets"], WL["n_haps"]) as b:
            closes = []
            for p in parts:
                b.push(p["read_group"], p["target_idx"], p["hap_idx"])
                before = b.stats()
                t0 = time.perf_counter()
                nnz = b.close_sample()
                wall = (time.perf_counter() - t0) * 1e3
                after = b.stats()
                closes.append({"n_ec": int(after["table_used"]), "pairs": nnz, "wall_ms": wall,
                               "device_ms": after["sample_ms"] - before["sample_ms"]})
            b.finalize_samples(copy=False)
            fs = b.stats()["finalize_ms"]
        with _native.EcBuilder(WL["n_targets"], WL["n_haps"]) as b:
            for p in parts:
                b.push(p["read_group"], p["target_idx"], p["hap_idx"])
            b.finalize(copy=False)
            f = b.stats()["finalize_ms"]
        if rep == 0:
            continue                                      # warm-up
        out["close"].append(closes)
        out["finalize_samples_ms"].append(fs)
        out["finalize_ms"].append(f)
    dev = [c["device_ms"] for r in out["close"] for c in r]
    wall = [c["wall_ms"] for r in out["close"] for c in r]
    out["summary"] = {"median_close_device_ms": float(np.median(dev)), "max_close_device_ms": float(max(dev)),
                      "median_close_wall_ms": float(np.median(wall)), "max_close_wall_ms": float(max(wall)),
                      "ecs_at_last_close": out["close"][0][-1]["n_ec"],
                      "median_finalize_samples_ms": float(np.median(out["finalize_samples_ms"])),
                      "median_finalize_ms": float(np.median(out["finalize_ms"]))}
    return out


def run_ab(parent_lib, runs, steps, warmup):
    out = {"parent": [], "tree": []}
    for i in range(runs):
        for side in ("parent", "tree"):
            env = dict(os.environ)
            env.pop("ECB200_LIB", None)
            if side == "parent":
                env["ECB200_LIB"] = parent_lib
            p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                                "--warmup", str(warmup), "--no-cpu-baseline"], capture_output=True, text=True, env=env,
                               cwd=ROOT, timeout=1800)
            if p.returncode != 0:
                raise SystemExit("bench.py failed (%s):\n%s" % (side, p.stderr[-3000:]))
            line = json.loads(p.stdout.strip().splitlines()[-1])
            out[side].append({"run": i, "ms_per_step": line["ms_per_step"], "alignments_per_s": line["value"],
                              "n_ec": line["config"]["n_ec"], "nnz_a": line["config"]["nnz_a"]})
    for side in ("parent", "tree"):
        ms = [r["ms_per_step"] for r in out[side]]
        out[side + "_summary"] = {"median_ms_per_step": float(np.median(ms)), "spread_ms_per_step": max(ms) - min(ms)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=8_000_000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--ab-runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    doc = {"gpu": gpu_info(0), "reads": args.reads, "files": FILES}
    cols = synth.make_columns(args.reads, WL["n_targets"], WL["n_haps"], WL["seed"] + 1000, mode=WL["mode"])
    parts = split(cols, FILES)
    with tempfile.TemporaryDirectory(prefix="bench_samples_") as tmp:
        whole = os.path.join(tmp, "whole.bam")
        synth.columns_to_bam(whole, cols, WL["n_targets"], WL["n_haps"])
        paths = []
        for i, p in enumerate(parts):
            paths.append(os.path.join(tmp, "part%d.bam" % i))
            synth.columns_to_bam(paths[-1], p, WL["n_targets"], WL["n_haps"])
        doc["files_run"] = run_files(paths, whole, tmp, args.runs)
    doc["close_run"] = run_close(parts, args.reps)
    if args.parent_lib:
        doc["ab"] = run_ab(args.parent_lib, args.ab_runs, args.steps, args.warmup)
    text = json.dumps(doc)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
