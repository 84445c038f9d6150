"""Speed of the host column emitter (libbamcols.so) in its three modes, on a synthetic 10x-style BAM with
fixed-length '|||' names written to a temporary directory:

  single  read_all()-style emit(): single-sample rules (convert())
  keys    emit_keys(): 128-bit name keys (convert(collate=True))
  cells   emit(cells=...): per-cell rules (the --multisample converter)

Every mode reads the whole file into reused buffers of `--chunk` rows, as the converters do; the time is that of
opening the reader and of the emit calls.  Per mode: alignments/s, the reader's phase seconds and the sha256 of
its columns (and, for cells, of the cell names).  `--lib` selects the libbamcols.so to load.  With `--parent-lib`
the parent's library and this tree's are run alternately, `--runs` times each, every run in a fresh process, and
the columns of both must hash alike.  Prints one JSON document with the CPU model and the thread count.

    python tools/time_emitter.py --parent-lib /path/to/parent/libbamcols.so --out profiles/r8_emitter.json
"""
import argparse
import hashlib
import json
import os
import struct
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from alntools_b200 import bam_io, bamcols, synth  # noqa: E402
from alntools_b200.header import TargetTables  # noqa: E402

T, H, CELLS = 2000, 2, 5000
MODES = ("single", "keys", "cells")


def write_bam(path, n_reads):
    """n_reads cfg-light reads of synth.make_columns as records with 10x-style names r<read>|||x...|||C<cell>."""
    cols = synth.make_columns(n_reads, T, H, seed=3, mode="light")
    rg = cols["read_group"].astype(np.int64)
    n = len(rg)
    rng = np.random.default_rng(5)
    cell_of_read = rng.integers(0, CELLS, size=int(rg.max()) + 1)
    tmpl = ("r%08d" % 0) + "|||x" * 13 + "|||C%05d" % 0
    name_len = len(tmpl) + 1
    rec_len = 36 + name_len
    raw = np.zeros((n, rec_len), dtype=np.uint8)
    raw[:, 0:4] = np.frombuffer(struct.pack("<i", 32 + name_len), dtype=np.uint8)
    core = np.zeros(n, dtype=np.dtype([("tid", "<i4"), ("pos", "<i4"), ("l_name", "u1"), ("mapq", "u1"), ("bin", "<u2"),
                                       ("ncig", "<u2"), ("flag", "<u2"), ("lseq", "<i4"), ("ntid", "<i4"), ("npos", "<i4"),
                                       ("tlen", "<i4")]))
    core["tid"] = cols["target_idx"].astype(np.int64) * H + cols["hap_idx"]
    core["l_name"] = name_len
    core["ntid"] = -1
    core["npos"] = -1
    raw[:, 4:36] = core.view(np.uint8).reshape(n, 32)
    raw[:, 36:36 + len(tmpl)] = np.frombuffer(tmpl.encode(), dtype=np.uint8)
    rem = rg.copy()
    for d in range(8, 0, -1):
        raw[:, 36 + d] = (rem % 10 + 48).astype(np.uint8)
        rem //= 10
    rem = cell_of_read[rg].copy()
    for d in range(len(tmpl) - 1, len(tmpl) - 6, -1):
        raw[:, 36 + d] = (rem % 10 + 48).astype(np.uint8)
        rem //= 10
    flat = raw.reshape(-1)
    per_block = max(1, 60000 // rec_len) * rec_len
    with open(path, "wb") as fh:
        bam_io._write_blocks(fh, bam_io.bam_header_bytes(synth.reference_names(T, H)), 60000, 1)
        for off in range(0, flat.size, per_block):
            fh.write(bam_io.bgzf_block(flat[off:off + per_block].tobytes(), 1))
        fh.write(bam_io.BGZF_EOF)
    return n


def time_mode(path, mode, chunk):
    refs = synth.reference_names(T, H)
    tables = TargetTables([r[0] for r in refs], [r[1] for r in refs], None)
    if mode == "keys":
        bufs = [np.empty(chunk, np.uint64), np.empty(chunk, np.uint64), np.empty(chunk, np.int32), np.empty(chunk, np.int32)]
    else:
        bufs = [np.empty(chunk, np.int32) for _ in range(4 if mode == "cells" else 3)]
    for b in bufs:
        b.fill(0)   # first touch outside the timed calls, as the converters' reused buffers
    hashes = [hashlib.sha256() for _ in bufs]
    cells = bamcols.CellDictionary() if mode == "cells" else None
    t0 = time.perf_counter()
    r = bamcols.BamColumnReader(path)
    r.set_tables(tables)
    seconds = time.perf_counter() - t0
    rows, done = 0, False
    while not done:
        t0 = time.perf_counter()
        if mode == "keys":
            n, done = r.emit_keys(*bufs)
        else:
            n, done = r.emit(bufs[0], bufs[1], bufs[2], bufs[3] if cells is not None else None, cells)
        seconds += time.perf_counter() - t0
        rows += n
        for h, b in zip(hashes, bufs):
            h.update(b[:n].tobytes())
    digest = hashlib.sha256(b"".join(h.digest() for h in hashes))
    if cells is not None:
        digest.update("\0".join(cells.names()).encode())
    out = {"alignments": r.all_alignments, "rows": rows, "seconds": seconds,
           "alignments_per_s": r.all_alignments / seconds, "phase_seconds": r.phase_seconds(),
           "sha256": digest.hexdigest()}
    r.close()
    return out


def one_run(path, chunk):
    return {mode: time_mode(path, mode, chunk) for mode in MODES}


def child_run(path, lib, chunk):
    p = subprocess.run([sys.executable, os.path.abspath(__file__), "--bam", path, "--lib", lib, "--chunk", str(chunk)],
                       capture_output=True, text=True, timeout=3600)
    if p.returncode != 0:
        raise SystemExit("time_emitter.py --lib %s failed:\n%s" % (lib, p.stderr[-3000:]))
    return json.loads(p.stdout.strip().splitlines()[-1])["runs"]["lib"][0]


def cpu_model():
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return None


def summary(runs):
    out = {}
    for mode in MODES:
        v = [r[mode]["alignments_per_s"] for r in runs]
        out[mode] = {"median_alignments_per_s": float(np.median(v)), "min": min(v), "max": max(v),
                     "spread": max(v) - min(v)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=2_000_000)
    ap.add_argument("--chunk", type=int, default=1 << 21, help="rows per emit call (the converters use up to 2^21)")
    ap.add_argument("--lib", default=None, help="libbamcols.so to load (default: the tree's)")
    ap.add_argument("--parent-lib", default=None, help="the parent's libbamcols.so: alternate it with --lib")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--bam", default=None, help="an existing synthetic BAM (used by the alternating runs)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lib = os.path.abspath(args.lib or bamcols.LIB_PATH)
    bamcols.LIB_PATH = lib
    doc = {"cpu_model": cpu_model(), "threads": len(os.sched_getaffinity(0)), "chunk_rows": args.chunk}
    with tempfile.TemporaryDirectory() as d:
        path = args.bam
        if path is None:
            path = os.path.join(d, "cells.bam")
            doc["reads"] = args.reads
            doc["alignments"] = write_bam(path, args.reads)
        doc["bam_bytes"] = os.path.getsize(path)
        if args.parent_lib is None:
            doc["libraries"] = {"lib": lib}
            doc["runs"] = {"lib": [one_run(path, args.chunk) for _ in range(1 if args.bam else args.runs)]}
        else:
            sides = {"parent": os.path.abspath(args.parent_lib), "tree": lib}
            doc["libraries"] = sides
            doc["runs"] = {side: [] for side in sides}
            for _ in range(args.runs):
                for side, side_lib in sides.items():
                    doc["runs"][side].append(child_run(path, side_lib, args.chunk))
    doc["summary"] = {side: summary(runs) for side, runs in doc["runs"].items()}
    doc["sha256_equal"] = {mode: len({r[mode]["sha256"] for runs in doc["runs"].values() for r in runs}) == 1
                           for mode in MODES}
    text = json.dumps(doc)
    print(text, flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(text + "\n")
    if not all(doc["sha256_equal"].values()):
        raise SystemExit("the columns differ between runs or libraries: %s" % doc["sha256_equal"])


if __name__ == "__main__":
    main()
