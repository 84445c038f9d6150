"""Device BAM decode (ecb_bam_* in include/ecb200.h, _native.BamDecoder, convert(decode="device")) against the host
reader libbamcols: the device rows, concatenated over all calls, must equal BamColumnReader.read_all() element for
element, with the same counters and --rangefile ranges; the EC and range files of convert() must equal the goldens.
Records, reads and blocks are made to span windows (ECB_OPT_BAM_WINDOW) and calls."""
import hashlib
import os
import struct
import zlib

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases
from alntools_b200 import bam_io, bamcols, synth

pytestmark = pytest.mark.gpu

REFS = [("T%d_%s" % (t, h), 100 + t) for t in range(6) for h in "AB"]
WINDOWS = (4096, 65536, 0)


@pytest.fixture(scope="module", autouse=True)
def _built(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a B200")


def _host(path):
    with bamcols.BamColumnReader(path) as r:
        r.build_tables(None)
        r.track_ranges(True)
        cols = r.read_all()
        return cols, (r.all_alignments, r.n_groups), r.ranges()


def _device(path, window=0, max_bytes=32 << 20, builder=None):
    """Columns of `path` from the device decoder: calls of up to max_bytes compressed bytes."""
    from alntools_b200._native import BamDecoder, EcBuilder
    with bamcols.BamColumnReader(path) as reader:
        tables = reader.build_tables(None)
        own = builder is None
        b = EcBuilder(max(1, tables.num_targets), max(1, tables.num_haplotypes)) if own else builder
        try:
            b.set_option("bam_window", window)
            parts = []
            with open(path, "rb") as fh:
                data = fh.read()
            with BamDecoder(b, tables.tid_target, tables.tid_hap, True) as dec:
                first = reader.plan_shards(1)[0]
                c, skip = first >> 16, first & 0xFFFF
                while True:
                    off, length, isize, end = reader.blocks(c, max_bytes)
                    if len(off) == 0:
                        break
                    got = dec.decode(np.frombuffer(data[c:end], dtype=np.uint8).copy(), off, length, isize, skip=skip)
                    parts.append([x.cpu().numpy() for x in got])
                    skip, c = 0, end
                got = dec.decode(np.zeros(0, np.uint8), [], [], [], last=True)
                parts.append([x.cpu().numpy() for x in got])
                cols = {k: np.concatenate([p[i] for p in parts]) for i, k in enumerate(("read_group", "target_idx", "hap_idx"))}
                return cols, dec.counters(), dec.ranges(), dec.stats()
        finally:
            if own:
                b.close()


def _same(path, windows=WINDOWS, call_bytes=(32 << 20, 3000)):
    want, counters, (lo, hi) = _host(path)
    for window in windows:
        for max_bytes in call_bytes:
            got, got_counters, (glo, ghi), _ = _device(path, window, max_bytes)
            for k in ("read_group", "target_idx", "hap_idx"):
                assert np.array_equal(got[k], want[k]), (path, window, max_bytes, k)
            assert got_counters == counters, (path, window, max_bytes)
            assert np.array_equal(glo, lo) and np.array_equal(ghi, hi), (path, window, max_bytes)
    return want


def _single_goldens():
    return sorted({c["bam"] for c in golden_cases("single")})


@pytest.mark.parametrize("bam", _single_goldens())
def test_golden_bams(bam):
    _same(os.path.join(GOLDEN, bam))


def _record(name, tid, flag=0, pos=7, ntid=-1, npos=-1, tail=b"", n_cigar=0, l_seq=0):
    nm = name.encode() + b"\x00"
    core = struct.pack("<iiBBHHHiiii", tid, pos, len(nm), 30, 4680, n_cigar, flag, l_seq, ntid, npos, 0) + nm + tail
    return struct.pack("<i", len(core)) + core


def _write_raw(path, raw, cut, compress=None):
    with open(path, "wb") as fh:
        for i, off in enumerate(range(0, len(raw), cut)):
            fh.write(compress(raw[off:off + cut], i) if compress else bam_io.bgzf_block(raw[off:off + cut]))
        fh.write(bam_io.BGZF_EOF)
    return path


def test_filters_names_and_tiny_blocks(tmp_path):
    """Unmapped / read2 / improper / mate-elsewhere alignments, names with leading and inner blanks, 70-byte blocks."""
    rng = np.random.default_rng(5)
    names = ["r1", " r1", "r1 x", "r1 y", " lead", "in ner", "in ner2", "r2", "r2", "r3"]
    alns = []
    for i in range(3000):
        name = names[int(rng.integers(0, len(names)))] if i % 7 else "q%04d" % (i // 5)
        flag = int(rng.choice([0, 0, 0, 4, 1 | 2, 1 | 2 | 0x80, 1, 16, 256]))
        tid = int(rng.integers(0, len(REFS)))
        ntid = tid if rng.random() < 0.8 else int(rng.integers(-1, len(REFS)))
        alns.append((name, flag, tid, int(rng.integers(0, 500)), ntid, int(rng.integers(-1, 300))))
    path = str(tmp_path / "filters.bam")
    bam_io.write_bam(path, REFS, alns, block_payload=70)
    _same(path)


def test_records_with_cigar_sequence_and_tags(tmp_path):
    rng = np.random.default_rng(31)
    recs = []
    for i in range(700):
        n_cig, l_seq = int(rng.integers(0, 4)), int(rng.integers(0, 200))
        tail = rng.integers(0, 256, 4 * n_cig + (l_seq + 1) // 2 + l_seq + int(rng.integers(0, 40)), dtype=np.uint8).tobytes()
        recs.append(_record("frag%04d" % (i // 3), int(rng.integers(0, len(REFS))), int(rng.choice([0, 16, 4, 256])),
                            int(rng.integers(0, 1000)), tail=tail, n_cigar=n_cig, l_seq=l_seq))
    raw = bam_io.bam_header_bytes(REFS) + b"".join(recs)
    _same(_write_raw(str(tmp_path / "full.bam"), raw, 777))


def test_parallel_hop_rejects_decoys(tmp_path):
    """Tag areas that hold byte-exact copies of small records: a segment that guesses one is hopped again."""
    rng = np.random.default_rng(77)
    decoy = _record("decoyA", 1) + _record("decoyB", 2)
    recs = []
    for i in range(3000):
        filler = rng.integers(0, 256, int(rng.integers(0, 90)), dtype=np.uint8).tobytes()
        tail = filler
        if i % 3 == 0:
            tail = filler + decoy + decoy if i % 2 else filler + decoy + rng.integers(0, 256, 60, dtype=np.uint8).tobytes()
        recs.append(_record("frag%04d" % (i // 2), int(rng.integers(0, len(REFS))), tail=tail))
    raw = bam_io.bam_header_bytes(REFS) + b"".join(recs)
    _same(_write_raw(str(tmp_path / "decoy.bam"), raw, 3000))


def test_long_read_and_long_records(tmp_path):
    """A read of 60 000 alignments, and records longer than a hop segment and than a 4 KiB window."""
    rng = np.random.default_rng(9)
    recs = [_record("short%d" % i, i % len(REFS)) for i in range(50)]
    recs += [_record("huge", int(t)) for t in rng.integers(0, len(REFS), 60000)]
    recs += [_record("long%d" % i, 3, tail=rng.integers(0, 256, 5000 * (i % 4), dtype=np.uint8).tobytes()) for i in range(40)]
    raw = bam_io.bam_header_bytes(REFS) + b"".join(recs)
    _same(_write_raw(str(tmp_path / "long.bam"), raw, 60000))


def test_stored_fixed_dynamic_and_empty_blocks(tmp_path):
    rng = np.random.default_rng(3)
    recs = [_record("m%05d" % (i // 2), int(rng.integers(0, len(REFS))), tail=b"ACGT" * int(rng.integers(0, 9)))
            for i in range(4000)]
    raw = bam_io.bam_header_bytes(REFS) + b"".join(recs)

    def compress(payload, i):
        level, strategy = [(0, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FIXED), (6, zlib.Z_DEFAULT_STRATEGY),
                           (1, zlib.Z_HUFFMAN_ONLY)][i % 4]
        comp = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        body = comp.compress(payload) + comp.flush()
        block = (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(body) + 25) + body
                 + struct.pack("<II", zlib.crc32(payload) & 0xFFFFFFFF, len(payload)))
        return block + (bam_io.bgzf_block(b"") if i % 3 == 1 else b"")
    _same(_write_raw(str(tmp_path / "mixed.bam"), raw, 2500, compress))


def _goldens_with_outputs():
    import json
    with open(os.path.join(GOLDEN, "manifest_range.json")) as fh:
        ranged = [c for c in json.load(fh) if c["kind"] == "single"]
    return golden_cases("single") + ranged


@pytest.mark.parametrize("case", _goldens_with_outputs(), ids=lambda c: c["name"] + ("_range" if "range" in c else ""))
def test_convert_device_reproduces_golden_files(case, tmp_path):
    from alntools_b200 import bam_utils
    out, rng = str(tmp_path / "out.bin"), str(tmp_path / "out.range.txt")
    tfile = os.path.join(GOLDEN, case["targets"]) if case["targets"] else None
    bam_utils.convert(os.path.join(GOLDEN, case["bam"]), out, None, num_chunks=1, number_processes=1,
                      target_filename=tfile, range_filename=rng if "range" in case else None, decode="device")
    with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
        assert a.read() == b.read()
    if "range" in case:
        with open(rng) as a, open(os.path.join(GOLDEN, case["range"])) as b:
            assert a.read() == b.read()


@pytest.mark.parametrize("shape", ["names", "seq100"])
def test_cfg2_shaped_8m_reads_host_equals_device(shape, tmp_path):
    from alntools_b200 import bam_utils
    cols = synth.make_columns(8_000_000, 100_000, 2, 1002, mode="diploid")
    bam = str(tmp_path / "cfg2.bam")
    if shape == "names":
        synth.columns_to_bam(bam, cols, 100_000, 2)
    else:
        synth.columns_to_bam_seq(bam, cols, 100_000, 2)
    del cols
    digests = {}
    for mode in ("host", "device"):
        out = str(tmp_path / (mode + ".bin"))
        bam_utils.convert(bam, out, None, decode=mode)
        with open(out, "rb") as fh:
            digests[mode] = hashlib.sha256(fh.read()).hexdigest()
    assert digests["host"] == digests["device"]


def _good_file(tmp_path):
    raw = bam_io.bam_header_bytes(REFS) + b"".join(_record("g%03d" % (i // 2), i % len(REFS)) for i in range(500))
    return _write_raw(str(tmp_path / "good.bam"), raw, 1000)


def test_corrupt_block_fails_in_the_device_inflate_and_a_fresh_decoder_recovers(tmp_path):
    """A damaged block far behind the header (the host reader inflates only the first blocks when it opens the file):
    the device inflate rejects it, reports it as ECB_ERR_FORMAT -> ValueError naming the block, as the host reader
    raises ValueError for the same file; a fresh decoder on the same builder then decodes the good bytes."""
    from alntools_b200._native import BamDecoder, EcBuilder
    raw = bam_io.bam_header_bytes(REFS) + b"".join(_record("c%04d" % (i // 2), i % len(REFS)) for i in range(3000))
    good = _write_raw(str(tmp_path / "good.bam"), raw, 1000)
    want = _host(good)[0]
    with bamcols.BamColumnReader(good) as reader:
        tables = reader.build_tables(None)
        first = reader.plan_shards(1)[0]
        c, skip = first >> 16, first & 0xFFFF
        off, length, isize, end = reader.blocks(c, 1 << 30)
    assert len(off) > 40
    with open(good, "rb") as fh:
        data = fh.read()[c:end]
    j = 37                                           # block index in the call
    damaged = bytearray(data)
    for k in range(int(length[j])):                  # first damage zlib rejects
        trial = bytearray(damaged)
        trial[int(off[j]) + k] ^= 0xFF
        d = zlib.decompressobj(-15)
        try:
            out = d.decompress(bytes(trial[int(off[j]):int(off[j]) + int(length[j])]), int(isize[j]) + 1)
            ok = d.eof and len(out) == int(isize[j])
        except zlib.error:
            ok = False
        if not ok:
            damaged = trial
            break
    assert damaged != bytearray(data)
    bad = str(tmp_path / "corrupt.bam")
    with open(good, "rb") as fh:
        head = fh.read()[:c]
    with open(bad, "wb") as fh:
        fh.write(head + bytes(damaged) + bam_io.BGZF_EOF)
    with pytest.raises(ValueError) as host_err:
        _host(bad)
    assert "inflate failed" in str(host_err.value)
    with EcBuilder(max(1, tables.num_targets), max(1, tables.num_haplotypes)) as builder:
        with BamDecoder(builder, tables.tid_target, tables.tid_hap) as dec:
            with pytest.raises(ValueError) as dev_err:
                dec.decode(np.frombuffer(bytes(damaged), dtype=np.uint8).copy(), off, length, isize, skip=skip)
            assert "block %d of this call" % j in str(dev_err.value)
            with pytest.raises(Exception):           # a failed decoder refuses further calls
                dec.decode(np.zeros(0, np.uint8), [], [], [], last=True)
        builder.reset()
        got = _device(good, builder=builder)[0]
        for k in ("read_group", "target_idx", "hap_idx"):
            assert np.array_equal(got[k], want[k]), k


def test_rows_live_on_the_builders_gpu(tmp_path):
    """convert(device=N) with torch's current device elsewhere: the rows are views on GPU N and the EC file is right."""
    import torch
    from alntools_b200 import bam_utils
    from alntools_b200._native import BamDecoder, EcBuilder
    last = torch.cuda.device_count() - 1
    if last < 1:
        pytest.skip("needs a second GPU")
    assert torch.cuda.current_device() != last
    case = golden_cases("single")[0]
    path = os.path.join(GOLDEN, case["bam"])
    with bamcols.BamColumnReader(path) as reader:
        tables = reader.build_tables(None)
        first = reader.plan_shards(1)[0]
        off, length, isize, end = reader.blocks(first >> 16, 1 << 30)
        with open(path, "rb") as fh:
            data = fh.read()[first >> 16:end]
    with EcBuilder(tables.num_targets, tables.num_haplotypes, device=last) as builder:
        with BamDecoder(builder, tables.tid_target, tables.tid_hap) as dec:
            rg, tg, hp = dec.decode(np.frombuffer(data, dtype=np.uint8).copy(), off, length, isize, skip=first & 0xFFFF,
                                    last=True)
            assert rg.device == tg.device == hp.device == torch.device("cuda", last)
    out = str(tmp_path / "out.bin")
    bam_utils.convert(path, out, None, num_chunks=1, number_processes=1, device=last, decode="device")
    with open(out, "rb") as a, open(os.path.join(GOLDEN, case["ec"]), "rb") as b:
        assert a.read() == b.read()


def test_errors_raise_the_host_exception_and_a_fresh_decoder_recovers(tmp_path):
    from alntools_b200._native import EcBuilder
    header = bam_io.bam_header_bytes(REFS)
    body = b"".join(_record("e%03d" % i, i % len(REFS)) for i in range(300))
    bad = {}
    bad["truncated"] = bam_io.bgzf_block(header + body + _record("t", 1)[:-5]) + bam_io.BGZF_EOF
    bad["block_size"] = bam_io.bgzf_block(header + body + struct.pack("<i", 5) + b"x" * 64) + bam_io.BGZF_EOF
    bad["tid"] = bam_io.bgzf_block(header + body + _record("z", len(REFS) + 3)) + bam_io.BGZF_EOF
    good = _good_file(tmp_path)
    want = _host(good)[0]
    with EcBuilder(6, 2) as builder:
        for name, blob in bad.items():
            path = str(tmp_path / (name + ".bam"))
            with open(path, "wb") as fh:
                fh.write(blob)
            with pytest.raises(Exception) as host_err:
                _host(path)
            with pytest.raises(Exception) as dev_err:
                _device(path, builder=builder)
            assert type(dev_err.value) is type(host_err.value), (name, host_err.value, dev_err.value)
            builder.reset()
            got = _device(good, builder=builder)[0]
            for k in ("read_group", "target_idx", "hap_idx"):
                assert np.array_equal(got[k], want[k]), (name, k)


def test_no_valid_alignment_raises_like_the_host_path(tmp_path):
    from alntools_b200 import bam_utils
    path = str(tmp_path / "unmapped.bam")
    bam_io.write_bam(path, REFS, [("u%d" % i, 4, 0) for i in range(50)])
    errors = []
    for mode in ("host", "device"):
        with pytest.raises(RuntimeError) as err:
            bam_utils.convert(path, str(tmp_path / "x.bin"), None, decode=mode)
        errors.append(str(err.value))
    assert errors[0] == errors[1]
