"""Collation within a device memory budget, for bench.py's bam_e2e sample (8 M cfg2-shaped reads, 16.4 M alignments)
with its alignments shuffled: convert(collate=True) unbudgeted and at budgets of about 1/4 and 1/16 of the unbudgeted
collator's device bytes (ALNTOOLS_B200_COLLATE_BUDGET), which force a spill and about 4 and 16 groups of the names
pass.  One warm-up of each, then `--passes` passes each, alternating; the best pass counts.  Every EC file must have the
sha256 of the unbudgeted one.  The collator's stats of the last pass of each budget (phase milliseconds, spills, groups,
peak device and host bytes, copies) come with it, and the GPU's name, power limit and max SM clock are read in the same
run.  Prints one JSON line.

    python tools/bench_collate_spill.py [--reads 8000000] [--passes 3]
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

import numpy as np  # noqa: E402
import torch  # noqa: E402

from alntools_b200 import bam_utils, emitter, synth  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402
from bench_collate import write  # noqa: E402

N_TARGETS, N_HAPS = 100_000, 2
ENV = "ALNTOOLS_B200_COLLATE_BUDGET"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=8_000_000)
    ap.add_argument("--passes", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the B200")
    line = {"what": "convert(collate=True) of a shuffled BAM file on one GPU, host decode (%d host threads), "
                    "unbudgeted and within device memory budgets" % os.cpu_count(), "reads": args.reads}
    line.update(gpu_info(0))
    cols = synth.make_columns(args.reads, N_TARGETS, N_HAPS, 1002, mode="diploid")   # bench.py bam_e2e: cfg2, seed + 1000
    rg, tg, hp = cols["read_group"], cols["target_idx"], cols["hap_idx"]
    n_aln = int(len(rg))
    line["alignments"] = n_aln
    perm = np.random.default_rng(5).permutation(n_aln)

    stats = []
    real = emitter.stream_collated

    def spy(*a, **kw):
        out = real(*a, **kw)
        stats.append(out[2])
        return out

    emitter.stream_collated = spy
    with tempfile.TemporaryDirectory(prefix="ecb_collate_spill_") as tmp:
        bam = os.path.join(tmp, "shuffled", "sample.bam")
        os.makedirs(os.path.dirname(bam))
        write(bam, rg[perm], tg[perm], hp[perm])
        line["file_bytes"] = os.path.getsize(bam)

        def run(name, budget):
            os.environ[ENV] = str(budget)
            out = os.path.join(tmp, name + ".bin")
            t0 = time.perf_counter()
            bam_utils.convert(bam, out, None, collate=True)
            dt = time.perf_counter() - t0
            with open(out, "rb") as fh:
                return dt, hashlib.sha256(fh.read()).hexdigest(), stats[-1]

        _, _, st = run("unbudgeted", 0)
        full = st["device_bytes"]
        budgets = {"unbudgeted": 0, "budget_quarter": full // 4, "budget_sixteenth": full // 16}
        times = {k: [] for k in budgets}
        last = {}
        for i in range(args.passes + 1):
            for name, budget in budgets.items():
                dt, digest, st = run(name, budget)
                if i > 0:
                    times[name].append(dt)
                last[name] = (digest, st)
        for name, budget in budgets.items():
            digest, st = last[name]
            st = dict(st)
            st["device_bytes_per_alignment"] = st["device_bytes"] / n_aln
            st["host_bytes_per_alignment"] = st["host_bytes"] / n_aln
            st["pcie_bytes_per_alignment"] = (st["h2d_bytes"] + st["d2h_bytes"]) / n_aln
            line[name] = {"budget_bytes": budget, "alignments_per_s": n_aln / min(times[name]), "best_s": min(times[name]),
                          "passes_s": times[name], "ec_sha256": digest, "stats": st}
        base = line["unbudgeted"]["alignments_per_s"]
        for name in ("budget_quarter", "budget_sixteenth"):
            line[name]["over_unbudgeted"] = line[name]["alignments_per_s"] / base
        line["ec_sha256_equal"] = len({line[k]["ec_sha256"] for k in budgets}) == 1
    print(json.dumps(line))


if __name__ == "__main__":
    main()
