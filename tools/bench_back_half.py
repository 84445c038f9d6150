"""The back half of a step (harvest, finalize, the push's round trips) on two libraries, alternating.

  ab      bench.py's default line (cfg2_diploid_30M, one GPU, no CPU arm) run `--runs` times on each of two
          libraries (ECB200_LIB=--parent-lib, then the tree's), alternating: ms_per_step, group_ms (the grouping
          kernel) and kernel launches per step of every run.
  parts   the same step (reset -> push -> finalize, device-resident) in a worker process per library, alternating,
          `--parts-runs` times: per run the median over `--steps` steps of push_ms, group_ms, harvest_ms, finalize_ms and
          the kernel launches of a step, from the library's own statistics.
  others  `--others` workloads (default cfg3_do8_heavy and cfg5_sweep_k16) through bench.py once per library.
  kernels one step of each library under torch.profiler: the kernels it launched, by name.

Every summary gives the median and the min-max of each figure.  Prints one JSON document with the GPU's name, power
limit and max SM clock (read in the same run) and writes it to --out.

    python tools/bench_back_half.py --parent-lib /path/to/parent/libecb200.so --out profiles/r10_back_half.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402


def summary(rows, keys):
    out = {}
    if not rows:
        return out
    for k in keys:
        v = [r[k] for r in rows]
        out[k] = {"median": float(np.median(v)), "min": float(min(v)), "max": float(max(v))}
    return out


def env_for(side, parent_lib):
    env = dict(os.environ)
    env.pop("ECB200_LIB", None)
    if side == "parent":
        env["ECB200_LIB"] = parent_lib
    return env


def run_bench(side, parent_lib, workload, steps, warmup):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                        "--warmup", str(warmup), "--no-cpu-baseline", "--workload", workload], capture_output=True,
                       text=True, env=env_for(side, parent_lib), cwd=ROOT, timeout=1800)
    if p.returncode != 0:
        raise SystemExit("bench.py failed (%s, %s):\n%s" % (side, workload, p.stderr[-3000:]))
    line = json.loads(p.stdout.strip().splitlines()[-1])
    return {"ms_per_step": line["ms_per_step"], "group_ms": line["roofline"]["kernel_ms"],
            "kernel_launches": line["gpu_launches"] / line["steps"], "alignments_per_s": line["value"],
            "n_ec": line["config"]["n_ec"], "nnz_a": line["config"]["nnz_a"]}


def run_worker(side, parent_lib, args, profile):
    cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--steps", str(args.steps), "--warmup",
           str(args.warmup)] + (["--profile"] if profile else [])
    p = subprocess.run(cmd, capture_output=True, text=True, env=env_for(side, parent_lib), cwd=ROOT, timeout=1800)
    if p.returncode != 0:
        raise SystemExit("worker failed (%s):\n%s" % (side, p.stderr[-3000:]))
    return json.loads(p.stdout.strip().splitlines()[-1])


def worker(args):
    """bench.py's default step on the library ECB200_LIB names (or the tree's)."""
    import torch
    import bench
    from alntools_b200 import synth
    from alntools_b200._native import EcBuilder

    wl = bench.WORKLOADS["cfg2_diploid_30M"]
    cols = synth.make_columns(wl["n_reads"], wl["n_targets"], wl["n_haps"], wl["seed"], mode=wl["mode"])
    dev = {k: torch.from_numpy(cols[k]).cuda() for k in ("read_group", "target_idx", "hap_idx")}
    stream = torch.cuda.current_stream()
    b = EcBuilder(wl["n_targets"], wl["n_haps"], alignments_hint=len(cols["read_group"]), result_on_device=1)
    b.set_stream(stream.cuda_stream)

    def step():
        b.reset()
        b.push(dev["read_group"], dev["target_idx"], dev["hap_idx"])
        return b.finalize_raw()

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    rows = []
    for _ in range(args.steps):
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record(stream)
        step()
        s1.record(stream)
        torch.cuda.synchronize()
        st = b.stats()
        rows.append({"step_ms": s0.elapsed_time(s1), "push_ms": st["push_ms"], "group_ms": st["group_ms"],
                     "harvest_ms": st["harvest_ms"], "finalize_ms": st["finalize_ms"],
                     "kernel_launches": st["kernel_launches"]})
    out = {k: float(np.median([r[k] for r in rows])) for k in rows[0]}
    out["step_ms_each"] = [round(r["step_ms"], 4) for r in rows]   # a slow run shows here as one slow step or many
    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        kernels = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA" and not ev.name.startswith("Memcpy") and not ev.name.startswith("Memset"):
                name = ev.name.split("<")[0].split("(")[0].replace("void ", "")
                kernels[name] = kernels.get(name, 0) + 1
        out["profiler_kernels"] = dict(sorted(kernels.items()))
        out["profiler_kernel_count"] = sum(kernels.values())
    b.close()
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="library of the parent commit")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--parts-runs", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--others", default="cfg3_do8_heavy,cfg5_sweep_k16")
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--profile", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    if not args.parent_lib:
        ap.error("--parent-lib is required")
    from bench_cells_multigpu import gpu_info
    sides = ("parent", "tree")
    doc = {"gpu_info": gpu_info(0), "parent_lib": args.parent_lib, "runs": args.runs, "steps": args.steps,
           "warmup": args.warmup}
    ab = {s: [] for s in sides}
    parts = {s: [] for s in sides}
    for i in range(args.runs):
        for s in sides:
            ab[s].append(dict(run=i, **run_bench(s, args.parent_lib, "cfg2_diploid_30M", args.steps, args.warmup)))
    for i in range(args.parts_runs):
        for s in sides:
            parts[s].append(dict(run=i, **run_worker(s, args.parent_lib, args, profile=(i == 0))))
    doc["ab_default_workload"] = {s: ab[s] for s in sides}
    doc["ab_summary"] = {s: summary(ab[s], ("ms_per_step", "group_ms", "kernel_launches")) for s in sides}
    doc["parts"] = {s: parts[s] for s in sides}
    doc["parts_summary"] = {s: summary(parts[s], ("step_ms", "push_ms", "group_ms", "harvest_ms", "finalize_ms",
                                                  "kernel_launches")) for s in sides}
    if args.runs:
        p, t = doc["ab_summary"]["parent"]["ms_per_step"], doc["ab_summary"]["tree"]["ms_per_step"]
        doc["verdict"] = {"median_gain_ms": p["median"] - t["median"], "ranges_disjoint": t["max"] < p["min"]}
    doc["others"] = {}
    for w in [x for x in args.others.split(",") if x]:
        doc["others"][w] = {s: run_bench(s, args.parent_lib, w, args.steps, args.warmup) for s in sides}
    doc["gpu_info_after"] = gpu_info(0)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    sys.exit(main())
