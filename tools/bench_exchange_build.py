"""Slice builds of the multi-GPU exchange with 2 ranks emulated on one GPU (arenas in one process instead of IPC
mappings): ecb_order_build (single-sample) and ecb_cells_order_build (per-cell) on cfg2-shaped input, `--reads` reads
per rank with bench.py's per-rank seeds (the per-cell run adds 50 000 cells and rank-major order keys).  The exchange
runs once up to the second dispatch; then, after `--warmup` builds, `--reps` builds of each rank's slice, each between
two CUDA events on the stream the owner works on.  A build ends in a synchronisation, so its host round trips are
inside the window.  The library is the one ECB200_LIB names (default: the tree's), so that two builds of it can be
compared in alternating runs.  Prints the library, the GPU's name, power limit and max SM clock, per-rank median /
p10 / p90 milliseconds and a sha256 of the slices, in one JSON line.

    ECB200_LIB=/path/to/libecb200.so python tools/bench_exchange_build.py [--reads 8000000] [--reps 200] [--warmup 20]
"""
import argparse
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from alntools_b200 import _native, synth  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402

WL = dict(n_targets=100_000, n_haps=2, mode="diploid", seed=2)   # bench.py's cfg2_diploid_30M
N_CELLS = 50_000
WORLD = 2
RANK_STRIDE = 1 << 40


def time_builds(builds, reps, warmup, stream):
    """Per rank: the milliseconds of `reps` calls of builds[r], ranks interleaved, after `warmup` rounds."""
    ms = [[] for _ in builds]
    for i in range(warmup + reps):
        for r, build in enumerate(builds):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            build()
            b.record(stream)
            b.synchronize()
            if i >= warmup:
                ms[r].append(a.elapsed_time(b))
    return {"rank%d" % r: {"median_ms": float(np.median(m)), "p10_ms": float(np.percentile(m, 10)),
                           "p90_ms": float(np.percentile(m, 90)), "mean_ms": float(np.mean(m))} for r, m in enumerate(ms)}


def digest(slices):
    h = hashlib.sha256()
    for sl in slices:
        for k in sorted(sl):
            v = sl[k]
            h.update(v.cpu().numpy().tobytes() if hasattr(v, "cpu") else str(v).encode())
    return h.hexdigest()


def single_sample(cols, args, stream):
    locals_, owners, base = [], [], 0
    for c in cols:
        n = len(c["read_group"])
        lb = _native.EcBuilder(WL["n_targets"], WL["n_haps"], alignments_hint=n)
        lb.set_stream(stream.cuda_stream)
        lb.push(c["read_group"], c["target_idx"], c["hap_idx"], order_base=base)
        base += n
        locals_.append(lb)
        owners.append(_native.EcBuilder(WL["n_targets"], WL["n_haps"], alignments_hint=n))
        owners[-1].set_stream(stream.cuda_stream)
    cap = 2 * max(lb.stats()["table_used"] for lb in locals_) + 1024      # as multi_gpu.distributed_finalize
    bases = [ob.arena_create(cap)[1] for ob in owners]
    spans = [lb.export_to_arenas(bases, cap) for lb in locals_]
    for ob in owners:
        ob.import_arena()
        ob.arena_reset()
    lo, hi = [s[0] for s in spans], [s[1] for s in spans]
    for ob in owners:
        ob.order_dispatch(bases, cap, lo, hi)
    builds = [lambda r=r: owners[r].order_build(locals_[r], lo[r], hi[r]) for r in range(WORLD)]
    out = {"timing": time_builds(builds, args.reps, args.warmup, stream)}
    slices = [b() for b in builds]
    out["n_ec"] = [sl["n_ec"] for sl in slices]
    out["nnz"] = [sl["nnz"] for sl in slices]
    out["sha256"] = digest(slices)
    for b in locals_ + owners:
        b.close()
    return out


def per_cell(cols, args, stream):
    locals_, owners = [], []
    for r, c in enumerate(cols):
        lb = _native.EcBuilder(WL["n_targets"], WL["n_haps"], with_cells=True)
        lb.set_stream(stream.cuda_stream)
        lb.push(c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"], order_base=r * RANK_STRIDE,
                drop_last_group=True)
        locals_.append(lb)
        owners.append(_native.EcBuilder(WL["n_targets"], WL["n_haps"]))
        owners[-1].set_stream(stream.cuda_stream)
    sums = [lb.cells_summary(None, N_CELLS) for lb in locals_]
    keys = torch.cat([k for k, _ in sums])
    totals = sum(t for _, t in sums)
    n_samples = [lb.cells_order(keys, totals, 1, None, WORLD) for lb in locals_][0][0]
    counts = sum(lb.cells_dispatch_counts(WORLD) for lb in locals_).tolist()
    cap_ec, cap_pairs = max(1, max(counts[:WORLD])), max(1, max(counts[WORLD:]))
    bases = [ob.cells_arena_create(cap_ec, cap_pairs)[1] for ob in owners]
    spans = [lb.cells_export_to_arenas(bases, cap_ec, cap_pairs) for lb in locals_]
    for ob in owners:
        ob.cells_import_arena()
    lo, hi = [s[0] for s in spans], [s[1] for s in spans]
    counts = sum(ob.cells_dispatch_counts(WORLD, lo, hi) for ob in owners).tolist()
    if max(counts[:WORLD]) > cap_ec or max(counts[WORLD:]) > cap_pairs:
        cap_ec, cap_pairs = max(cap_ec, max(counts[:WORLD])), max(cap_pairs, max(counts[WORLD:]))
        bases = [ob.cells_arena_create(cap_ec, cap_pairs)[1] for ob in owners]
    else:
        for ob in owners:
            ob.arena_reset()
    for ob in owners:
        ob.cells_order_dispatch(bases, cap_ec, cap_pairs, lo, hi)
    builds = [lambda r=r: owners[r].cells_order_build(locals_[r], lo[r], hi[r], n_samples) for r in range(WORLD)]
    out = {"n_samples": n_samples, "timing": time_builds(builds, args.reps, args.warmup, stream)}
    slices = [b() for b in builds]
    out["n_ec"] = [sl["n_ec"] for sl in slices]
    out["nnz"] = [sl["nnz"] for sl in slices]
    out["sha256"] = digest(slices)
    for b in locals_ + owners:
        b.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=8_000_000, help="reads per rank")
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the B200")
    torch.cuda.set_device(0)
    stream = torch.cuda.current_stream(0)
    line = {"what": "ecb_order_build and ecb_cells_order_build, %d ranks emulated on one GPU, cfg2-shaped input" % WORLD,
            "lib": os.path.realpath(os.environ.get("ECB200_LIB") or _native.LIB_PATH), "reads_per_rank": args.reads,
            "reps": args.reps, "warmup": args.warmup}
    line.update(gpu_info(0))
    cols = [synth.make_columns(args.reads, WL["n_targets"], WL["n_haps"], WL["seed"] + 7919 * r, mode=WL["mode"],
                               n_cells=N_CELLS) for r in range(WORLD)]
    line["alignments_per_rank"] = [len(c["read_group"]) for c in cols]
    line["order_build"] = single_sample(cols, args, stream)
    line["cells_order_build"] = per_cell(cols, args, stream)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
