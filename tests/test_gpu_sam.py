"""SAM text on the GPU (ecb_sam_* in include/ecb200.h, _native.SamDecoder, sam_utils.convert_sam) against the BAM path:
SAM rendered from a BAM file converts to the bytes convert() writes for that BAM file, whatever the call size, through
a pipe as from a file; hand-made text equals the Python emitter; bad lines fail with their line number."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, golden_cases
from alntools_b200 import bam_io, bam_utils, sam_utils, synth
from sam_render import bam_to_sam, sam_text

pytestmark = pytest.mark.gpu

REFS = [("T%d_%s" % (t, h), 100 + t) for t in range(6) for h in "AB"]


@pytest.fixture(scope="module", autouse=True)
def _built(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")


def _bytes(path):
    with open(path, "rb") as fh:
        return fh.read()


def _goldens_with_outputs():
    import json
    with open(os.path.join(GOLDEN, "manifest_range.json")) as fh:
        ranged = [c for c in json.load(fh) if c["kind"] == "single"]
    return golden_cases("single") + ranged


@pytest.mark.parametrize("read_len", [0, 100])
@pytest.mark.parametrize("case", _goldens_with_outputs(), ids=lambda c: c["name"] + ("_range" if "range" in c else ""))
def test_golden_sam_gives_golden_files(case, read_len, tmp_path):
    sam, out, rng = str(tmp_path / "in.sam"), str(tmp_path / "out.bin"), str(tmp_path / "out.range.txt")
    bam_to_sam(os.path.join(GOLDEN, case["bam"]), sam, read_len)
    tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
    sam_utils.convert_sam(sam, out, range_filename=rng if "range" in case else None, sample=case["bam"],
                          target_filename=tfile)
    assert _bytes(out) == _bytes(os.path.join(GOLDEN, case["ec"]))
    if "range" in case:
        assert _bytes(rng) == _bytes(os.path.join(GOLDEN, case["range"]))


@pytest.mark.parametrize("max_bytes", [4096, 5000, 65536, 1 << 30])
def test_call_sizes_split_lines_reads_and_names(max_bytes, tmp_path):
    """Calls of a few KiB cut reads and carried names at every place; 1 GiB takes the file in one call.  A 4 KiB buffer
    is shorter than some lines (300-base SEQ and QUAL), so the buffers grow."""
    case = [c for c in golden_cases("single") if c["name"] == "synth_h8_heavy"][0]
    sam, out = str(tmp_path / "in.sam"), str(tmp_path / "out.bin")
    bam_to_sam(os.path.join(GOLDEN, case["bam"]), sam, read_len=0)
    sam_utils.convert_sam(sam, out, sample=case["bam"], max_bytes=max_bytes)
    assert _bytes(out) == _bytes(os.path.join(GOLDEN, case["ec"]))
    raw = bam_io.inflate_file(os.path.join(GOLDEN, case["bam"]))
    header = bam_io.parse_header(raw)
    recs = list(bam_io.iter_records(raw, header.records_offset))
    with open(sam, "wb") as fh:
        fh.write(sam_text(header.references, header.lengths, recs, read_len=3000))
    sam_utils.convert_sam(sam, out, sample=case["bam"], max_bytes=max_bytes)
    assert _bytes(out) == _bytes(os.path.join(GOLDEN, case["ec"]))


def test_pipe_from_standard_input(tmp_path):
    case = [c for c in golden_cases("single") if c["name"] == "synth_h2"][0]
    sam, out = str(tmp_path / "in.sam"), str(tmp_path / "out.bin")
    bam_to_sam(os.path.join(GOLDEN, case["bam"]), sam, read_len=100)
    env = dict(os.environ, PYTHONPATH=ROOT)
    cmd = "cat %s | %s -m alntools_b200.sam2ec - %s -s %s" % (sam, sys.executable, out, case["bam"])
    p = subprocess.run(cmd, shell=True, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-3000:]
    assert _bytes(out) == _bytes(os.path.join(GOLDEN, case["ec"]))


def _edge_records(rng, n=4000):
    names = ["r1", " r1", "r1 x", "r1 y", " lead", "in ner", "in ner2", "r2", "r2", "r3"]
    recs = []
    for i in range(n):
        name = names[int(rng.integers(0, len(names)))] if i % 7 else "q%04d" % (i // 5)
        flag = int(rng.choice([0, 0, 0, 4, 1 | 2, 1 | 2 | 0x80, 1, 16, 256, 1 | 2 | 0x40]))
        tid = int(rng.integers(0, len(REFS)))
        if flag & 4 and rng.random() < 0.5:
            tid = -1
        ntid = tid if rng.random() < 0.8 else int(rng.integers(-1, len(REFS)))
        recs.append((name, flag, tid, int(rng.integers(-1, 500)), ntid, int(rng.integers(-1, 300))))
    return recs


@pytest.mark.parametrize("max_bytes", [3000, 1 << 20])
def test_edge_text_equals_python_emitter_and_bam(max_bytes, tmp_path, monkeypatch):
    rng = np.random.default_rng(11)
    recs = _edge_records(rng)
    text = sam_text([r for r, _ in REFS], [l for _, l in REFS], recs, read_len=50)
    sam = str(tmp_path / "edge.sam")
    with open(sam, "wb") as fh:
        fh.write(text.rstrip(b"\n"))                    # the last line without its '\n'
    out = {}
    for emitter in ("native", "python"):
        monkeypatch.setenv("ALNTOOLS_B200_EMITTER", emitter)
        out[emitter] = str(tmp_path / (emitter + ".bin"))
        sam_utils.convert_sam(sam, out[emitter], sample="s", max_bytes=max_bytes)
    monkeypatch.delenv("ALNTOOLS_B200_EMITTER")
    bam = str(tmp_path / "edge.bam")
    with open(sam, "rb") as fh:
        refs, lengths, n = sam_utils.read_header(fh)
        statement = list(sam_utils.iter_records(fh, refs, n + 1))
    assert statement == recs
    bam_io.write_bam(bam, list(zip(refs, lengths)), statement)
    bam_utils.convert(bam, str(tmp_path / "bam.bin"), None, sample="s")
    rng_sam, rng_bam = str(tmp_path / "s.range"), str(tmp_path / "b.range")
    sam_utils.convert_sam(sam, str(tmp_path / "r.bin"), range_filename=rng_sam, sample="s", max_bytes=max_bytes)
    bam_utils.convert(bam, str(tmp_path / "rb.bin"), None, sample="s", range_filename=rng_bam)
    assert _bytes(out["native"]) == _bytes(out["python"]) == _bytes(str(tmp_path / "bam.bin"))
    assert _bytes(rng_sam) == _bytes(rng_bam)


@pytest.mark.parametrize("mode,n_haps", [("diploid", 2), ("heavy", 8)])
def test_large_synthetic_sam_equals_bam(mode, n_haps, tmp_path):
    cols = synth.make_columns(1_500_000, 20_000, n_haps, 77, mode=mode)
    bam, sam = str(tmp_path / "x.bam"), str(tmp_path / "x.sam")
    synth.columns_to_bam(bam, cols, 20_000, n_haps)
    synth.columns_to_sam(sam, cols, 20_000, n_haps, read_len=100 if mode == "diploid" else 0)
    del cols
    bam_utils.convert(bam, str(tmp_path / "b.bin"), None, sample="s")
    sam_utils.convert_sam(sam, str(tmp_path / "s.bin"), sample="s", max_bytes=64 << 20)
    assert hashlib.sha256(_bytes(str(tmp_path / "b.bin"))).digest() == hashlib.sha256(_bytes(str(tmp_path / "s.bin"))).digest()


def test_a_million_sq_names(tmp_path):
    refs = [("ENST%09d_%s" % (t, "AB"[h]), 500 + t % 1000) for t in range(500_000) for h in range(2)]
    rng = np.random.default_rng(3)
    tids = rng.integers(0, len(refs), 200_000)
    recs = [("r%06d" % (i // 3), 0, int(t), 10, -1, -1) for i, t in enumerate(tids)]
    sam, bam = str(tmp_path / "m.sam"), str(tmp_path / "m.bam")
    with open(sam, "wb") as fh:
        fh.write(sam_text([r for r, _ in refs], [l for _, l in refs], recs, header_extra=False))
    bam_io.write_bam(bam, refs, recs)
    sam_utils.convert_sam(sam, str(tmp_path / "s.bin"), sample="s")
    bam_utils.convert(bam, str(tmp_path / "b.bin"), None, sample="s")
    assert _bytes(str(tmp_path / "s.bin")) == _bytes(str(tmp_path / "b.bin"))


def test_long_read_with_max_read_unlimited(tmp_path, monkeypatch):
    rng = np.random.default_rng(5)
    recs = [("s%d" % i, 0, i % len(REFS), 1, -1, -1) for i in range(20)]
    recs += [("huge", 0, int(t), 1, -1, -1) for t in rng.integers(0, len(REFS), 100_000)]
    recs += [("t%d" % i, 0, i % len(REFS), 1, -1, -1) for i in range(20)]
    sam, bam = str(tmp_path / "l.sam"), str(tmp_path / "l.bam")
    with open(sam, "wb") as fh:
        fh.write(sam_text([r for r, _ in REFS], [l for _, l in REFS], recs))
    bam_io.write_bam(bam, REFS, recs)
    with pytest.raises(Exception, match="16384"):
        sam_utils.convert_sam(sam, str(tmp_path / "x.bin"), sample="s")
    monkeypatch.setenv("ALNTOOLS_B200_MAX_READ", "0")
    sam_utils.convert_sam(sam, str(tmp_path / "s.bin"), sample="s", max_bytes=1 << 20)
    bam_utils.convert(bam, str(tmp_path / "b.bin"), None, sample="s")
    assert _bytes(str(tmp_path / "s.bin")) == _bytes(str(tmp_path / "b.bin"))


def test_header_only_and_all_filtered_raise_like_convert(tmp_path):
    sam = str(tmp_path / "h.sam")
    for body in (b"", b"u\t4\t*\t0\t0\t*\t*\t0\t0\t*\t*\n"):
        with open(sam, "wb") as fh:
            fh.write(sam_text([r for r, _ in REFS], [l for _, l in REFS], []) + body)
        with pytest.raises(RuntimeError, match="three positive integers"):
            sam_utils.convert_sam(sam, str(tmp_path / "o.bin"))
        assert not os.path.exists(str(tmp_path / "o.bin"))


BAD = [
    (b"@CO\tlate", "a header line (starting with '@') after the first alignment line"),
    (b"", "fewer than 11 tab-separated fields"),
    (b"a\t0\tT0_A\t1\t0\t*\t*\t0\t0\t*", "fewer than 11 tab-separated fields"),
    (b"\t0\tT0_A\t1\t0\t*\t*\t0\t0\t*\t*", "QNAME empty or longer than 254 bytes"),
    (b"q" * 255 + b"\t0\tT0_A\t1\t0\t*\t*\t0\t0\t*\t*", "QNAME empty or longer than 254 bytes"),
    (b"a\t65536\tT0_A\t1\t0\t*\t*\t0\t0\t*\t*", "FLAG not a decimal integer in [0, 65535]"),
    (b"a\t+1\tT0_A\t1\t0\t*\t*\t0\t0\t*\t*", "FLAG not a decimal integer in [0, 65535]"),
    (b"a\t0\tT0_AB\t1\t0\t*\t*\t0\t0\t*\t*", "RNAME not '*' and not an @SQ name"),
    (b"a\t0\tT0_A\t99999999999\t0\t*\t*\t0\t0\t*\t*", "POS not a decimal integer in [0, 2147483647]"),
    (b"a\t0\tT0_A\t1\t0\t*\tT0\t0\t0\t*\t*", "RNEXT not '*', '=' or an @SQ name"),
    (b"a\t0\tT0_A\t1\t0\t*\t*\t1x\t0\t*\t*", "PNEXT not a decimal integer in [0, 2147483647]"),
    (b"a\t0\t*\t1\t0\t*\t*\t0\t0\t*\t*", "alignment with reference id -1 outside the header's 12 references"),
]


@pytest.mark.parametrize("line,what", BAD, ids=[str(i) for i in range(len(BAD))])
def test_bad_line_in_the_second_call(line, what, tmp_path):
    good = [("g%04d" % (i // 2), 0, i % len(REFS), 5, -1, -1) for i in range(400)]
    text = sam_text([r for r, _ in REFS], [l for _, l in REFS], good)
    n_head = len(REFS) + 2
    body_lines = text.split(b"\n")[n_head:-1]
    bad_at = 300
    body_lines[bad_at] = line
    sam, out = str(tmp_path / "bad.sam"), str(tmp_path / "o.bin")
    with open(sam, "wb") as fh:
        fh.write(b"\n".join(text.split(b"\n")[:n_head] + body_lines) + b"\n")
    with pytest.raises(ValueError) as err:
        sam_utils.convert_sam(sam, out, max_bytes=8192)     # the first call ends near line 250
    assert str(err.value) == "%s: line %d: %s" % (sam, n_head + bad_at + 1, what)
    assert not os.path.exists(out)


def test_decoder_stats_and_counters(tmp_path):
    from alntools_b200._native import EcBuilder, SamDecoder
    from alntools_b200.header import TargetTables
    recs = [("c%03d" % (i // 3), 4 if i % 5 == 0 else 0, i % len(REFS), 9, -1, -1) for i in range(900)]
    text = sam_text([r for r, _ in REFS], [l for _, l in REFS], recs, header_extra=False)
    body = text[text.index(b"c000"):]
    tables = TargetTables([r for r, _ in REFS], [l for _, l in REFS])
    half = body.index(b"\n", len(body) // 2) + 1
    with EcBuilder(tables.num_targets, tables.num_haplotypes) as builder:
        with SamDecoder(builder, [r for r, _ in REFS], tables.tid_target, tables.tid_hap, len(REFS) + 1, True) as dec:
            rows = [x.cpu().numpy() for x in dec.parse(np.frombuffer(body[:half], np.uint8).copy())]
            rest = [x.cpu().numpy() for x in dec.parse(np.frombuffer(body[half:], np.uint8).copy(), last=True)]
            with pytest.raises(Exception):          # a decoder that had its last call refuses more
                dec.parse(np.zeros(0, np.uint8), last=True)
            st = dec.stats()
            assert dec.counters() == (900, 300)
            lo, hi = dec.ranges()
    assert st["bytes"] == len(body) and st["lines"] == 900 and st["calls"] == 2
    assert all(st[k] >= 0 for k in ("h2d_ms", "lines_ms", "fields_ms", "rules_ms"))
    from alntools_b200 import emitter
    want = emitter.emit_single(recs, tables)
    for i, k in enumerate(("read_group", "target_idx", "hap_idx")):
        assert np.array_equal(np.concatenate([rows[i], rest[i]]), getattr(want, k)), k
    assert (lo == 9).all() and (hi == 9).all()
