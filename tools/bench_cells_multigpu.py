"""The per-cell (multisample) build over N GPUs, weak scaling: cfg4's workload on every GPU.

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29551 \
        tools/bench_cells_multigpu.py [--steps K] [--warmup W] [--reads R] [--no-parity]

Every rank generates 20 M reads (seed 4 + 7919 * rank, as bench.py seeds its ranks) over the same 50 000-cell
universe, cut into 4 read-aligned files, and keeps the columns on its GPU.  A step is what the device-resident
steps of bench.py time, with the per-cell exchange: reset, one push per file at rank-major order keys,
multi_gpu.distributed_finalize_cells (minimum count 1000).  Steps are timed with CUDA events on the stream the
library runs on; the step time is the slowest rank's median step.  One extra step with ECB_MGPU_TIMING phases follows the
timed ones (it synchronises after every phase, so it is not part of the step time).  Parity: rank 0 assembles
every rank's slice and compares it with the C per-cell oracle on all ranks' files, outside the timed region.
Rank 0 prints one JSON line."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WL = dict(n_reads=20_000_000, n_targets=140_000, n_haps=8, mode="diploid", seed=4, n_cells=50_000, n_files=4,
          min_count=1000)


def gpu_info(index):
    """Name, power limit and max SM clock of the GPU, read in the same run as the measurement."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        name, power, clock = [x.strip() for x in out.strip().split(",")]
        return {"gpu": name, "power_limit_w": float(power), "max_sm_clock_mhz": int(float(clock))}
    except Exception as exc:  # noqa: BLE001 - reported, not hidden
        return {"gpu": torch.cuda.get_device_name(index), "gpu_info_error": repr(exc)}


def make_rank_columns(rank, n_reads):
    from alntools_b200 import synth
    cols = synth.make_columns(n_reads, WL["n_targets"], WL["n_haps"], WL["seed"] + 7919 * rank, mode=WL["mode"],
                              n_cells=WL["n_cells"])
    n = len(cols["read_group"])
    cuts = [0]
    for k in range(1, WL["n_files"]):
        c = n * k // WL["n_files"]
        while c < n and cols["read_group"][c] == cols["read_group"][c - 1]:
            c += 1
        cuts.append(c)
    cuts.append(n)
    return cols, cuts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads", type=int, default=WL["n_reads"], help="reads per GPU")
    ap.add_argument("--no-parity", action="store_true")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist.init_process_group("nccl", device_id=dev)
    from alntools_b200 import multi_gpu
    from alntools_b200._native import EcBuilder
    from alntools_b200.bam_utils_multisample import RANK_STRIDE

    cols, cuts = make_rank_columns(rank, args.reads)
    n_aln = cuts[-1]
    d = {k: torch.from_numpy(cols[k]).to(dev) for k in ("read_group", "target_idx", "hap_idx", "cell_idx")}
    stream = torch.cuda.current_stream(dev)
    local = EcBuilder(WL["n_targets"], WL["n_haps"], with_cells=True, alignments_hint=n_aln, device=local_rank,
                      result_on_device=1)
    owner = EcBuilder(WL["n_targets"], WL["n_haps"], alignments_hint=n_aln, device=local_rank)
    local.set_stream(stream.cuda_stream)
    owner.set_stream(stream.cuda_stream)

    def step():
        local.reset()
        owner.reset()
        for a, b in zip(cuts[:-1], cuts[1:]):
            local.push(d["read_group"][a:b], d["target_idx"][a:b], d["hap_idx"][a:b], d["cell_idx"][a:b],
                       order_base=rank * RANK_STRIDE + a, drop_last_group=True)
        # the same cell universe on every rank: global cell ids are the synthetic ids (identity map)
        return multi_gpu.distributed_finalize_cells(local, lambda: owner, dev, WL["min_count"], None, WL["n_cells"])

    for _ in range(args.warmup):
        step()
    dist.barrier()
    torch.cuda.synchronize(dev)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    for i in range(args.steps):
        starts[i].record(stream)
        out = step()
        ends[i].record(stream)
    torch.cuda.synchronize(dev)
    per_step = [s.elapsed_time(e) for s, e in zip(starts, ends)]
    ms = torch.tensor([float(np.median(per_step))], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    alignments = torch.tensor([n_aln], dtype=torch.int64, device=dev)
    dist.all_reduce(alignments)
    alignments = int(alignments.item())

    # one untimed step with the per-phase wall clock
    multi_gpu._TIMING = True
    step()
    multi_gpu._TIMING = False
    phases = multi_gpu.LAST_PHASES.get("distributed_finalize_cells", [])

    parity = {"checked": False}
    if not args.no_parity:
        out = step()
        mine = {"id_base": out["id_base"], "n_ec_local": out["n_ec_local"],
                "a": [out[k].cpu().numpy() for k in ("a_indptr", "a_indices", "a_data")],
                "n": [out[k].cpu().numpy() for k in ("n_col_counts", "n_col_offset", "n_indices", "n_data")],
                "n_indptr": out["n_indptr"].cpu().numpy(), "cell_order": out["cell_order"].cpu().numpy()}
        parts = [None] * world
        dist.all_gather_object(parts, mine)
        if rank == 0:
            parity = {"checked": True, "equal": check_parity(parts, world, args.reads)}
    if rank == 0:
        line = {"metric": "cells_multigpu_step", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "reads_per_gpu": args.reads, "cells": WL["n_cells"], "files_per_gpu": WL["n_files"],
                "min_count": WL["min_count"], "step_ms": round(ms, 3), "alignments": alignments,
                "alignments_per_s": alignments / (ms / 1e3), "phases_ms": {k: round(v, 3) for k, v in phases},
                "parity": parity}
        line.update(gpu_info(local_rank))
        print(json.dumps(line), flush=True)
    local.close()
    owner.close()
    dist.destroy_process_group()


def check_parity(parts, world, n_reads):
    """Every rank's slice put together in id order against the C oracle over all ranks' files in rank order."""
    from oracle import c_oracle
    pushes = []
    for r in range(world):
        cols, cuts = make_rank_columns(r, n_reads)
        for a, b in zip(cuts[:-1], cuts[1:]):
            pushes.append(tuple(np.ascontiguousarray(cols[k][a:b]) for k in ("read_group", "target_idx", "hap_idx",
                                                                              "cell_idx")) + (True,))
        del cols
    want = c_oracle.ec_from_columns_cells(pushes, WL["min_count"])
    del pushes
    ip, n_ip = want["a_indptr"], want["n_indptr"]
    ok = np.array_equal(parts[0]["cell_order"], want["cell_order"]) and np.array_equal(parts[0]["n_indptr"], n_ip)
    ok = ok and sum(p["n_ec_local"] for p in parts) == len(ip) - 1
    ok = ok and sum(len(p["n"][2]) for p in parts) == int(n_ip[-1])
    for p in parts:
        a, b = p["id_base"], p["id_base"] + p["n_ec_local"]
        ok = ok and np.array_equal(p["a"][0], ip[a:b + 1] - ip[a]) and np.array_equal(p["a"][1], want["a_indices"][ip[a]:ip[b]]) \
            and np.array_equal(p["a"][2], want["a_data"][ip[a]:ip[b]])
        counts, offset, idx, dat = p["n"]
        starts = np.cumsum(counts) - counts
        col = np.repeat(np.arange(len(counts)), counts)
        dest = n_ip[col].astype(np.int64) + offset[col] + (np.arange(len(idx)) - starts[col])
        ok = ok and np.array_equal(want["n_indices"][dest], idx.astype(np.int64) + a) and np.array_equal(want["n_data"][dest], dat)
    return bool(ok)


if __name__ == "__main__":
    main()
