"""Host against device BAM decode in convert() on one GPU, for bench.py's bam_e2e sample (cfg2-shaped reads written as
one BAM file) in two record shapes: names only (synth.columns_to_bam) and with a 100-bp CIGAR / SEQ / QUAL
(synth.columns_to_bam_seq).  Per shape: one warm-up of each path, then `--passes` passes each, alternating; the EC
files of both paths must have the same sha256.  One more device pass through emitter.stream_single_device reports
the decoder's own figures: compressed and inflated bytes per alignment and the stream milliseconds per phase
(CUDA events in libecb200; the hop and rules phases include their host round trips).  The GPU's name, power limit
and max SM clock are read in the same run.  Prints one JSON line.

    python tools/bench_device_decode.py [--reads 8000000] [--passes 3]
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

import torch  # noqa: E402

from alntools_b200 import bam_utils, bamcols, emitter, synth  # noqa: E402
from alntools_b200._native import EcBuilder  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402


def sha256(path):
    with open(path, "rb") as fh:
        return hashlib.sha256(fh.read()).hexdigest()


def decoder_figures(bam):
    with bamcols.BamColumnReader(bam) as reader:
        tables = reader.build_tables(None)
        with EcBuilder(tables.num_targets, tables.num_haplotypes, pageable_results=1) as builder:
            t0 = time.perf_counter()
            valid, (records, _), _, st = emitter.stream_single_device(bam, reader, builder, tables, False)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
    return {"records": records, "valid": valid, "decode_and_push_s": wall,
            "compressed_bytes_per_alignment": st["h2d_bytes"] / records,
            "inflated_bytes_per_alignment": st["inflated_bytes"] / records,
            "phase_ms": {k: st[k + "_ms"] for k in ("h2d", "inflate", "hop", "rules")},
            "inflate_GBps": st["inflated_bytes"] / (st["inflate_ms"] * 1e6) if st["inflate_ms"] else None,
            "blocks": st["blocks"], "windows": st["windows"], "hop_rounds": st["hop_rounds"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=8_000_000)
    ap.add_argument("--passes", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the B200")
    line = {"what": "convert() BAM file -> EC file, decode='host' (libbamcols, %d host threads) vs decode='device'"
                    % os.cpu_count(), "reads": args.reads}
    line.update(gpu_info(0))
    cols = synth.make_columns(args.reads, 100_000, 2, 1002, mode="diploid")   # bench.py bam_e2e: cfg2, seed + 1000
    n_aln = int(len(cols["read_group"]))
    line["alignments"] = n_aln
    with tempfile.TemporaryDirectory(prefix="ecb_decode_") as tmp:
        for shape, write in (("names", synth.columns_to_bam), ("seq100", synth.columns_to_bam_seq)):
            bam = os.path.join(tmp, shape + ".bam")
            write(bam, cols, 100_000, 2)
            res = {"file_bytes": os.path.getsize(bam)}
            times = {"host": [], "device": []}
            digests = {}
            for i in range(args.passes + 1):
                for mode in ("host", "device"):
                    out = os.path.join(tmp, "%s_%s.bin" % (shape, mode))
                    t0 = time.perf_counter()
                    bam_utils.convert(bam, out, None, decode=mode)
                    dt = time.perf_counter() - t0
                    if i > 0:
                        times[mode].append(dt)
                    digests[mode] = sha256(out)
            for mode in ("host", "device"):
                res[mode] = {"alignments_per_s": n_aln / min(times[mode]), "best_s": min(times[mode]),
                             "passes_s": times[mode]}
            res["device_over_host"] = res["device"]["alignments_per_s"] / res["host"]["alignments_per_s"]
            res["ec_sha256_equal"] = digests["host"] == digests["device"]
            res["decoder"] = decoder_figures(bam)
            line[shape] = res
            os.remove(bam)
    print(json.dumps(line))


if __name__ == "__main__":
    main()
