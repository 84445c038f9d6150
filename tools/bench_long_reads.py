"""Reads longer than 16384 alignments (ECB_OPT_MAX_READ): what the ordinary path pays, and what the long path costs.

  ab    bench.py's default workload (cfg2_diploid_30M, one GPU, no CPU arm) run `--runs` times on each of two libraries
        (ECB200_LIB=--parent-lib, then the tree's), alternating; the step time and group_ms of each run.
  long  `--reads` cfg2-shaped reads plus L reads of k alignments (k = 1e5, 1e6, 1e7; L = `--long`), pushed from device
        memory with max_read = 0: per push the deferred pass (long_ms), the long reads' alignments per second over it,
        the whole push and the grouping kernel, against the same reads without the long ones.  `--reps` pushes each,
        after one warm-up push.  Every result is checked against the first.
  convert  one convert() (ALNTOOLS_B200_MAX_READ=0, host decode) of a BAM file of `--convert-reads` cfg2-shaped reads
        plus L reads of 10^6 alignments; wall time.

Prints one JSON document with the GPU's name, power limit and max SM clock (read in the same run) and writes it to
--out.

    python tools/bench_long_reads.py --parent-lib /path/to/parent/libecb200.so --out profiles/r7_long_reads.json
"""
import argparse
import hashlib
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
import torch  # noqa: E402

from alntools_b200 import _native, bam_utils, synth  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402

WL = dict(n_targets=100_000, n_haps=2, mode="diploid", seed=2)   # bench.py's cfg2_diploid_30M


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
            out[side].append({"run": i, "ms_per_step": line["ms_per_step"], "group_ms": line["roofline"]["kernel_ms"],
                              "alignments_per_s": line["value"], "n_ec": line["config"]["n_ec"],
                              "nnz_a": line["config"]["nnz_a"]})
    for side in ("parent", "tree"):
        ms = [r["ms_per_step"] for r in out[side]]
        g = [r["group_ms"] for r in out[side]]
        out[side + "_summary"] = {"median_ms_per_step": float(np.median(ms)), "spread_ms_per_step": max(ms) - min(ms),
                                  "median_group_ms": float(np.median(g)), "spread_group_ms": max(g) - min(g)}
    return out


def with_long(cols, k, n_long, seed):
    """cols with n_long reads of k alignments spread between its reads (targets uniform, haplotypes uniform)."""
    rng = np.random.default_rng(seed)
    rg = cols["read_group"]
    starts = np.flatnonzero(np.r_[True, rg[1:] != rg[:-1]])
    at = np.sort(rng.choice(starts[1:], n_long, replace=False))
    parts_rg, parts_tg, parts_hp, prev, next_id = [], [], [], 0, int(rg.max()) + 1
    for a in at.tolist() + [len(rg)]:
        parts_rg.append(rg[prev:a])
        parts_tg.append(cols["target_idx"][prev:a])
        parts_hp.append(cols["hap_idx"][prev:a])
        if a < len(rg):
            parts_rg.append(np.full(k, next_id, dtype=np.int32))
            parts_tg.append(rng.integers(0, WL["n_targets"], k).astype(np.int32))
            parts_hp.append(rng.integers(0, WL["n_haps"], k).astype(np.int32))
            next_id += 1
        prev = a
    return {"read_group": np.concatenate(parts_rg), "target_idx": np.concatenate(parts_tg),
            "hap_idx": np.concatenate(parts_hp)}


def digest(res):
    h = hashlib.sha256()
    for k in ("a_indptr", "a_indices", "a_data", "n_data"):
        h.update(np.ascontiguousarray(res[k]).tobytes())
    return h.hexdigest()


def time_pushes(cols, reps):
    dev = {k: torch.from_numpy(np.ascontiguousarray(cols[k])).cuda() for k in ("read_group", "target_idx", "hap_idx")}
    n = len(cols["read_group"])
    rows, first = [], None
    for i in range(reps + 1):
        with _native.EcBuilder(WL["n_targets"], WL["n_haps"], alignments_hint=n, max_read=0) as b:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            b.push(dev["read_group"], dev["target_idx"], dev["hap_idx"])
            wall = (time.perf_counter() - t0) * 1e3
            st = b.stats()
            d = digest(b.finalize())
        if first is None:
            first = d
        elif d != first:
            raise SystemExit("results differ between pushes")
        if i:
            rows.append({"push_ms": st["push_ms"], "group_ms": st["group_ms"], "harvest_ms": st["harvest_ms"],
                         "long_ms": st["long_ms"], "long_reads": st["long_reads"], "push_wall_ms": wall})
    med = {k: float(np.median([r[k] for r in rows])) for k in rows[0]}
    med["spread_long_ms"] = max(r["long_ms"] for r in rows) - min(r["long_ms"] for r in rows)
    med["spread_push_ms"] = max(r["push_ms"] for r in rows) - min(r["push_ms"] for r in rows)
    med["sha256"] = first
    return med


def run_long(n_reads, n_long, reps):
    base = synth.make_columns(n_reads, WL["n_targets"], WL["n_haps"], WL["seed"], mode=WL["mode"])
    base = {k: base[k] for k in ("read_group", "target_idx", "hap_idx")}
    out = {"reads": n_reads, "base_alignments": len(base["read_group"]), "none": time_pushes(base, reps)}
    for k in (100_000, 1_000_000, 10_000_000):
        cols = with_long(base, k, n_long, k)
        r = time_pushes(cols, reps)
        r.update(k=k, long=n_long, long_alignments=k * n_long,
                 long_alignments_per_s=k * n_long / (r["long_ms"] * 1e-3) if r["long_ms"] else None)
        out["k%d" % k] = r
    return out


def run_convert(n_reads, n_long):
    base = synth.make_columns(n_reads, WL["n_targets"], WL["n_haps"], WL["seed"], mode=WL["mode"])
    cols = with_long({k: base[k] for k in ("read_group", "target_idx", "hap_idx")}, 1_000_000, n_long, 1)
    with tempfile.TemporaryDirectory() as d:
        bam = os.path.join(d, "long.bam")
        synth.columns_to_bam(bam, cols, WL["n_targets"], WL["n_haps"])
        os.environ["ALNTOOLS_B200_MAX_READ"] = "0"
        walls = []
        for i in range(2):
            t0 = time.perf_counter()
            summary = bam_utils.convert(bam, os.path.join(d, "out.bin"), None, sample="s")
            walls.append(time.perf_counter() - t0)
        size = os.path.getsize(bam)
    n = len(cols["read_group"])
    return {"reads": n_reads, "long": n_long, "k": 1_000_000, "alignments": n, "bam_bytes": size,
            "wall_s_first": walls[0], "wall_s": walls[1], "alignments_per_s": n / walls[1], "n_ec": summary["n_ec"],
            "n_reads": summary["n_reads"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="library of the parent commit for the A/B (none: no A/B)")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads", type=int, default=8_000_000)
    ap.add_argument("--long", type=int, default=4)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--convert-reads", type=int, default=2_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_long_reads.py needs a GPU")
    lib = os.environ.get("ECB200_LIB") or _native.LIB_PATH
    doc = {"gpu_info": gpu_info(0), "library": os.path.relpath(lib, ROOT)}
    if args.parent_lib:
        doc["ab_default_workload"] = run_ab(args.parent_lib, args.runs, args.steps, args.warmup)
    doc["long_path"] = run_long(args.reads, args.long, args.reps)
    doc["convert"] = run_convert(args.convert_reads, args.long)
    doc["gpu_info_after"] = gpu_info(0)
    text = json.dumps(doc)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
