"""Collation by read name in convert() on one GPU, for bench.py's bam_e2e sample (8 M cfg2-shaped reads, written as one
BAM file by synth.columns_to_bam): the default convert() of the grouped file, convert(collate=True) of the same file
(what collating costs when nothing needs it) and of the file with its alignments shuffled (what it is for).  One
warm-up of each, then `--passes` passes each, alternating; the best pass counts.  The EC file of the shuffled file
must have the sha256 of the default convert() of its regrouped form F', and the collated grouped file that of the
default.  One more pass through emitter.stream_collated reports the collator's own figures (CUDA-event milliseconds
per phase, device bytes).  The GPU's name, power limit and max SM clock are read in the same run.  Prints one JSON line.

    python tools/bench_collate.py [--reads 8000000] [--passes 3]
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

from alntools_b200 import bam_io, bam_utils, bamcols, emitter, synth  # noqa: E402
from alntools_b200._native import EcBuilder  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402

N_TARGETS, N_HAPS = 100_000, 2


def sha256(path):
    with open(path, "rb") as fh:
        return hashlib.sha256(fh.read()).hexdigest()


def write(path, rg, tg, hp):
    tids = tg.astype(np.int64) * N_HAPS + hp
    bam_io.write_bam_columns(path, synth.reference_names(N_TARGETS, N_HAPS), rg, np.zeros(len(tids), np.uint16), tids)


def collator_figures(bam):
    with bamcols.BamColumnReader(bam) as reader:
        tables = reader.build_tables(None)
        with EcBuilder(tables.num_targets, tables.num_haplotypes, pageable_results=1) as builder:
            t0 = time.perf_counter()
            valid, reads, st = emitter.stream_collated(reader, builder)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
    st["device_bytes_per_alignment"] = st["device_bytes"] / valid
    return {"valid": valid, "reads": reads, "decode_collate_push_s": wall, "stats": st}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=8_000_000)
    ap.add_argument("--passes", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the B200")
    line = {"what": "convert() BAM file -> EC file on one GPU, host decode (%d host threads): default vs collate=True"
                    % os.cpu_count(), "reads": args.reads}
    line.update(gpu_info(0))
    cols = synth.make_columns(args.reads, N_TARGETS, N_HAPS, 1002, mode="diploid")   # bench.py bam_e2e: cfg2, seed + 1000
    rg, tg, hp = cols["read_group"], cols["target_idx"], cols["hap_idx"]
    n_aln = int(len(rg))
    line["alignments"] = n_aln
    perm = np.random.default_rng(5).permutation(n_aln)
    srg, stg, shp = rg[perm], tg[perm], hp[perm]
    first = np.full(args.reads, n_aln, dtype=np.int64)
    np.minimum.at(first, srg, np.arange(n_aln))
    order = np.argsort(first[srg], kind="stable")
    with tempfile.TemporaryDirectory(prefix="ecb_collate_") as tmp:
        files = {"grouped": os.path.join(tmp, "sample.bam"), "shuffled": os.path.join(tmp, "shuffled", "sample.bam"),
                 "regrouped": os.path.join(tmp, "regrouped", "sample.bam")}
        for p in files.values():
            os.makedirs(os.path.dirname(p), exist_ok=True)
        write(files["grouped"], rg, tg, hp)
        write(files["shuffled"], srg, stg, shp)
        write(files["regrouped"], srg[order], stg[order], shp[order])
        runs = {"default_grouped": (files["grouped"], False), "collate_grouped": (files["grouped"], True),
                "collate_shuffled": (files["shuffled"], True)}
        times = {k: [] for k in runs}
        digests = {}
        for i in range(args.passes + 1):
            for name, (bam, collate) in runs.items():
                out = os.path.join(tmp, name + ".bin")
                t0 = time.perf_counter()
                bam_utils.convert(bam, out, None, collate=collate)
                dt = time.perf_counter() - t0
                if i > 0:
                    times[name].append(dt)
                digests[name] = sha256(out)
        out = os.path.join(tmp, "regrouped.bin")
        bam_utils.convert(files["regrouped"], out, None)
        digests["default_regrouped"] = sha256(out)
        for name in runs:
            line[name] = {"alignments_per_s": n_aln / min(times[name]), "best_s": min(times[name]), "passes_s": times[name]}
        line["collate_grouped_over_default"] = line["collate_grouped"]["alignments_per_s"] / line["default_grouped"]["alignments_per_s"]
        line["ec_sha256_equal"] = {"collate_grouped_vs_default": digests["collate_grouped"] == digests["default_grouped"],
                                   "collate_shuffled_vs_default_of_regrouped": digests["collate_shuffled"] == digests["default_regrouped"]}
        line["file_bytes"] = os.path.getsize(files["grouped"])
        line["collator_grouped"] = collator_figures(files["grouped"])
        line["collator_shuffled"] = collator_figures(files["shuffled"])
    print(json.dumps(line))


if __name__ == "__main__":
    main()
