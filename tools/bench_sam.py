"""SAM text against BAM files on one GPU, for bench.py's bam_e2e sample (8 M cfg2-shaped reads) in two record shapes:
names only (CIGAR, SEQ and QUAL '*' in the SAM; synth.columns_to_bam) and a 100-bp CIGAR, SEQ and QUAL
(synth.columns_to_bam_seq / columns_to_sam(read_len=100)).

Per shape, after one warm-up of each, `--passes` passes each, alternating:
  bam        bam_utils.convert() of the BAM file (host decode, the default);
  sam_file   sam_utils.convert_sam() of the SAM file;
  sam_pipe   `cat x.sam | python -m alntools_b200.sam2ec - out.bin` in a fresh process (wall time of the whole command,
             with the interpreter's start and imports, which `startup_s` times alone).
The EC files must have one sha256.  One more pass through sam_utils.stream_sam_device gives the decoder's phases (stream
milliseconds between CUDA events: H2D, lines, fields, rules) and the parse rate in GB/s of text.  With --parent-tree,
bench.py's default workload runs from the parent commit's tree and this one, alternating.  The GPU's name, power limit and
max SM clock are read in the same run.  Prints one JSON document and writes it to --out.

    python tools/bench_sam.py [--reads 8000000] [--passes 3] [--parent-tree PATH] [--out FILE]
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

import torch  # noqa: E402

from alntools_b200 import bam_utils, sam_utils, synth  # noqa: E402
from alntools_b200._native import EcBuilder  # noqa: E402
from alntools_b200.header import TargetTables  # noqa: E402
from bench_cells_multigpu import gpu_info  # noqa: E402


def sha256(path):
    h = hashlib.sha256()
    with open(path, "rb") as fh:
        for block in iter(lambda: fh.read(1 << 24), b""):
            h.update(block)
    return h.hexdigest()


def run_ab(parent_tree, runs, steps, warmup):
    """bench.py's default workload from a checkout of the parent commit (its library built in place) and from this tree,
    alternating, each in a fresh process: step time and the bam_e2e line."""
    out = {"parent": [], "tree": []}
    env = dict(os.environ)
    env.pop("ECB200_LIB", None)
    for i in range(runs):
        for side, root in (("parent", parent_tree), ("tree", ROOT)):
            p = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", str(steps),
                                "--warmup", str(warmup), "--no-cpu-baseline"], capture_output=True, text=True, env=env,
                               cwd=root, timeout=1800)
            if p.returncode != 0:
                raise SystemExit("bench.py failed (%s):\n%s" % (side, p.stderr[-3000:]))
            line = json.loads(p.stdout.strip().splitlines()[-1])
            out[side].append({"run": i, "ms_per_step": line["ms_per_step"], "alignments_per_s": line["value"],
                              "bam_e2e_alignments_per_s": line.get("bam_e2e", {}).get("value")})
    for side in ("parent", "tree"):
        ms = sorted(r["ms_per_step"] for r in out[side])
        out[side + "_summary"] = {"median_ms_per_step": ms[len(ms) // 2], "spread_ms_per_step": ms[-1] - ms[0]}
    return out


def decoder_figures(sam):
    with open(sam, "rb") as fh:
        refs, lengths, n = sam_utils.read_header(fh)
        tables = TargetTables(refs, lengths)
        with EcBuilder(tables.num_targets, tables.num_haplotypes, pageable_results=1) as builder:
            t0 = time.perf_counter()
            valid, (lines, _), _, st = sam_utils.stream_sam_device(fh, sam, builder, tables, refs, n + 1, False)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
    parse_ms = st["lines_ms"] + st["fields_ms"] + st["rules_ms"]
    return {"lines": lines, "valid": valid, "calls": st["calls"], "parse_and_push_s": wall,
            "text_bytes_per_alignment": st["bytes"] / lines,
            "phase_ms": {k: st[k + "_ms"] for k in ("h2d", "lines", "fields", "rules")},
            "h2d_GBps": st["bytes"] / (st["h2d_ms"] * 1e6) if st["h2d_ms"] else None,
            "parse_GBps": st["bytes"] / (parse_ms * 1e6) if parse_ms else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=8_000_000)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--parent-tree", default=None, help="a checkout of the parent commit, its library built")
    ap.add_argument("--shapes", default="names,seq100")
    ap.add_argument("--ab-runs", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the B200")
    doc = {"what": "BAM file -> EC file (convert(), host decode on %d threads) vs SAM text -> EC file (convert_sam, "
                   "parsed on the GPU)" % os.cpu_count(), "reads": args.reads, "gpu": gpu_info(0)}

    def save():
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as fh:
                fh.write(json.dumps(doc) + "\n")

    cols = synth.make_columns(args.reads, 100_000, 2, 1002, mode="diploid")   # bench.py bam_e2e: cfg2, seed + 1000
    n_aln = int(len(cols["read_group"]))
    doc["alignments"] = n_aln
    env = dict(os.environ, PYTHONPATH=ROOT)
    t0 = time.perf_counter()
    subprocess.run([sys.executable, "-c", "import torch; torch.cuda.init(); import alntools_b200.sam_utils"], env=env,
                   check=True, cwd=ROOT)
    doc["startup_s"] = time.perf_counter() - t0
    with tempfile.TemporaryDirectory(prefix="bench_sam_") as tmp:
        for shape, read_len in (("names", 0), ("seq100", 100)):
            if shape not in args.shapes.split(","):
                continue
            bam, sam = os.path.join(tmp, shape + ".bam"), os.path.join(tmp, shape + ".sam")
            (synth.columns_to_bam if read_len == 0 else synth.columns_to_bam_seq)(bam, cols, 100_000, 2)
            synth.columns_to_sam(sam, cols, 100_000, 2, read_len=read_len)
            res = {"bam_bytes": os.path.getsize(bam), "sam_bytes": os.path.getsize(sam)}
            outs = {k: os.path.join(tmp, "%s_%s.bin" % (shape, k)) for k in ("bam", "sam_file", "sam_pipe")}
            runs = {
                "bam": lambda: bam_utils.convert(bam, outs["bam"], None, sample="s"),
                "sam_file": lambda: sam_utils.convert_sam(sam, outs["sam_file"], sample="s"),
                "sam_pipe": lambda: subprocess.run("cat %s | %s -m alntools_b200.sam2ec - %s -s s"
                                                   % (sam, sys.executable, outs["sam_pipe"]), shell=True, check=True,
                                                   env=env, cwd=ROOT),
            }
            times = {k: [] for k in runs}
            for i in range(args.passes + 1):
                for k, run in runs.items():
                    t0 = time.perf_counter()
                    run()
                    if i > 0:
                        times[k].append(time.perf_counter() - t0)
            digests = {k: sha256(p) for k, p in outs.items()}
            res["same_sha256"] = len(set(digests.values())) == 1
            for k in runs:
                best = min(times[k])
                res[k] = {"s": times[k], "best_s": best, "alignments_per_s": n_aln / best}
            res["decoder"] = decoder_figures(sam)
            doc[shape] = res
            save()
            os.remove(bam)
            os.remove(sam)
    if args.parent_tree:
        doc["ab"] = run_ab(args.parent_tree, args.ab_runs, args.steps, args.warmup)
        save()
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
