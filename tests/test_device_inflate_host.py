"""The device BGZF block decoder (alntools_b200/csrc/ecb_inflate.cuh) built for the host by g++ with AddressSanitizer and
UBSan (through tests/inflate_host_shim.cpp) and compared with zlib: every case must get zlib's accept/reject decision
(accepted iff the stream ends and exactly ISIZE bytes come out; ISIZE 0 is accepted unread) and, when accepted, the
same bytes, with no sanitizer report.  Also the BGZF block table of BamColumnReader.blocks() and the argument checks
of convert(decode=...), which run before any GPU work.  No GPU involved."""
import os
import shutil
import subprocess
import sys
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


# ---------------------------------------------------------------- cases (run in a sanitized child process)
def zlib_decision(src, isize):
    if isize == 0:
        return b""
    d = zlib.decompressobj(-15)
    try:
        out = d.decompress(src, isize + 1)
    except zlib.error:
        return None
    return out if d.eof and len(out) == isize else None


class BitWriter(object):
    def __init__(self):
        self.bits = []

    def put(self, value, n):                 # LSB first (header fields, extra bits)
        self.bits += [(value >> i) & 1 for i in range(n)]

    def code(self, code, n):                 # Huffman codes go MSB first
        self.bits += [(code >> (n - 1 - i)) & 1 for i in range(n)]

    def align(self):
        while len(self.bits) % 8:
            self.bits.append(0)

    def raw(self, data):
        self.align()
        for byte in data:
            self.put(byte, 8)

    def bytes(self):
        self.align()
        return bytes(sum(b << i for i, b in enumerate(self.bits[k:k + 8])) for k in range(0, len(self.bits), 8))


def fixed_lit(w, sym):
    if sym < 144:
        w.code(0x30 + sym, 8)
    elif sym < 256:
        w.code(0x190 + sym - 144, 9)
    elif sym < 280:
        w.code(sym - 256, 7)
    else:
        w.code(0xC0 + sym - 280, 8)


def canonical(lengths):
    codes, code, count = {}, 0, [0] * 16
    for l in lengths:
        count[l] += 1
    count[0] = 0
    nxt = [0] * 16
    for bits in range(1, 16):
        code = (code + count[bits - 1]) << 1
        nxt[bits] = code
    for s, l in enumerate(lengths):
        if l:
            codes[s] = (nxt[l], l)
            nxt[l] += 1
    return codes


def dynamic_block(lit_lens, dist_lens, symbols, cl_lens=None, final=1):
    """A dynamic block whose code lengths are sent with a code-length code of 16 four-bit codes (symbols 0-15)."""
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    cl = cl_lens if cl_lens is not None else [4] * 16 + [0, 0, 0]
    w = BitWriter()
    w.put(final, 1)
    w.put(2, 2)
    w.put(len(lit_lens) - 257, 5)
    w.put(len(dist_lens) - 1, 5)
    w.put(19 - 4, 4)
    for s in order:
        w.put(cl[s], 3)
    for l in list(lit_lens) + list(dist_lens):
        w.code(l, 4)                         # canonical code of symbol l when 0-15 all have 4 bits
    lc, dc = canonical(lit_lens), canonical(dist_lens)
    for kind, s in symbols:
        c, n = (lc if kind == "l" else dc)[s]
        w.code(c, n)
    return w.bytes()


def hand_built_cases():
    cases = []
    # distance 32 768 / length 258 / symbol 285 after a 32 768-byte stored block
    first = bytes(range(256)) * 128
    w = BitWriter()
    w.put(0, 1), w.put(0, 2)
    w.align()
    w.put(len(first), 16), w.put(len(first) ^ 0xFFFF, 16)
    w.raw(first)
    w.put(1, 1), w.put(1, 2)
    fixed_lit(w, 285)
    w.code(29, 5), w.put(32768 - 24577, 13)   # distance symbol 29 + 13 extra bits = 32 768
    fixed_lit(w, 256)
    far = w.bytes()
    whole = first + (first[:258])
    cases += [("far_match", far, len(whole)), ("far_match_short", far, len(whole) - 1), ("far_match_long", far, len(whole) + 1)]
    # a distance one byte too far
    w = BitWriter()
    w.put(1, 1), w.put(1, 2)
    fixed_lit(w, 65)
    fixed_lit(w, 257)
    w.code(1, 5)                              # distance 2 with one byte of output
    fixed_lit(w, 256)
    cases.append(("too_far", w.bytes(), 4))
    # stored LEN != ~NLEN
    cases.append(("stored_nlen", b"\x01\x05\x00\xfa\xff" + b"hello", 5))
    cases.append(("stored_nlen_bad", b"\x01\x05\x00\xfb\xff" + b"hello", 5))
    cases.append(("stored_short_input", b"\x01\x05\x00\xfa\xff" + b"hel", 5))
    # fixed symbols 286/287 and distances 30/31
    for sym in (286, 287):
        w = BitWriter()
        w.put(1, 1), w.put(1, 2)
        fixed_lit(w, 65)
        fixed_lit(w, sym)
        fixed_lit(w, 256)
        cases.append(("fixed_sym%d" % sym, w.bytes(), 4))
    for dist in (30, 31):
        w = BitWriter()
        w.put(1, 1), w.put(1, 2)
        fixed_lit(w, 65)
        fixed_lit(w, 257)
        w.code(dist, 5)
        fixed_lit(w, 256)
        cases.append(("fixed_dist%d" % dist, w.bytes(), 4))
    # missing end-of-block code: literals, then the input ends
    w = BitWriter()
    w.put(1, 1), w.put(1, 2)
    for ch in b"abc":
        fixed_lit(w, ch)
    cases.append(("no_eob", w.bytes(), 3))
    # dynamic headers
    lit = [0] * 257
    lit[65], lit[256] = 1, 1
    cases.append(("single_dist_code", dynamic_block(lit, [1], [("l", 65), ("l", 65), ("l", 256)]), 2))
    cases.append(("no_dist_code", dynamic_block(lit, [0], [("l", 65), ("l", 256)]), 1))
    cases.append(("cl_oversubscribed", dynamic_block(lit, [1], [("l", 256)], cl_lens=[1] * 19), 0 + 1))
    cases.append(("cl_incomplete", dynamic_block(lit, [1], [("l", 256)], cl_lens=[4] * 15 + [0] * 4), 1))
    lit2 = [0] * 257
    lit2[65], lit2[66], lit2[256] = 2, 2, 2
    cases.append(("lit_incomplete", dynamic_block(lit2, [1], [("l", 65), ("l", 256)]), 1))
    lit3 = [0] * 257
    lit3[65], lit3[66], lit3[256] = 1, 1, 1
    cases.append(("lit_oversubscribed", dynamic_block(lit3, [1], [("l", 65)]) + b"\x00" * 4, 1))
    lit4 = [0] * 257
    lit4[65], lit4[66] = 1, 1
    cases.append(("lit_no_eob_code", dynamic_block(lit4, [1], [("l", 65), ("l", 66)]) + b"\x00" * 4, 2))
    dist_inc = [2, 2, 0]
    lit5 = [0] * 258
    lit5[65], lit5[256], lit5[257] = 1, 2, 2
    cases.append(("dist_incomplete", dynamic_block(lit5, dist_inc, [("l", 65), ("l", 256)]), 1))
    # trailing bytes after the final block; ISIZE 0 with garbage
    good = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = good.compress(b"trailing test " * 20) + good.flush()
    cases.append(("trailing", body + b"garbage after the end", 280))
    cases.append(("isize0_garbage", b"\xff\xfe\xfd", 0))
    cases.append(("isize0_empty", b"", 0))
    cases.append(("empty_input", b"", 5))
    return cases


def payloads():
    from alntools_b200 import bam_io
    rng = np.random.default_rng(2)
    raw = bam_io.inflate_file(os.path.join(HERE, "golden", "synth_h8_heavy.bam"))
    return [("records", raw[:60000]), ("records_small", raw[1000:1700]), ("random", rng.bytes(3000)),
            ("runs", b"".join(bytes([int(c)]) * int(n) for c, n in zip(rng.integers(0, 4, 400), rng.integers(1, 300, 400)))[:65536]),
            ("zeros", bytes(65536)), ("full", (raw * 2)[:65536]), ("random_full", rng.bytes(65536))]


def compressed_cases():
    cases = []
    for pname, data in payloads():
        for level in range(10):
            for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED):
                c = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
                cases.append(("%s_l%d_s%d" % (pname, level, strategy), c.compress(data) + c.flush(), len(data)))
        for flush in (zlib.Z_SYNC_FLUSH, zlib.Z_FULL_FLUSH):
            c = zlib.compressobj(6, zlib.DEFLATED, -15)
            parts = [c.compress(data[k:k + 997]) + c.flush(flush) for k in range(0, len(data), 997)]
            cases.append(("%s_flush%d" % (pname, flush), b"".join(parts) + c.flush(), len(data)))
    return cases


def mutated_cases(n, seed=11):
    rng = np.random.default_rng(seed)
    base = [c for c in compressed_cases() if len(c[1]) < 4000 and c[2] < 8000]
    out = []
    for k in range(n):
        name, src, isize = base[int(rng.integers(0, len(base)))]
        b = bytearray(src)
        kind = k % 3
        if kind == 0 and b:
            for _ in range(int(rng.integers(1, 4))):
                i = int(rng.integers(0, len(b)))
                b[i] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1 and b:
            b = b[:int(rng.integers(0, len(b)))]
        elif b:
            i = int(rng.integers(0, len(b)))
            b[i] = int(rng.integers(0, 256))
            isize += int(rng.integers(-2, 3)) if rng.random() < 0.3 else 0
        out.append(("mut%d_%s" % (k, name), bytes(b), max(0, isize)))
    return out


def run_cases(lib_path, n_mutations):
    import ctypes
    lib = ctypes.CDLL(lib_path)
    lib.shim_inflate.argtypes = [ctypes.c_char_p, ctypes.c_int64, ctypes.c_char_p, ctypes.c_int64]
    lib.shim_inflate.restype = ctypes.c_int
    counts = {"accepted": 0, "rejected": 0}
    required = {"far_match": True, "single_dist_code": True, "no_dist_code": True, "trailing": True, "isize0_garbage": True,
                "stored_nlen": True, "stored_nlen_bad": False, "cl_oversubscribed": False, "cl_incomplete": False,
                "lit_incomplete": False, "lit_oversubscribed": False, "lit_no_eob_code": False, "fixed_sym286": False,
                "fixed_sym287": False, "fixed_dist30": False, "fixed_dist31": False, "no_eob": False, "too_far": False,
                "far_match_short": False, "far_match_long": False, "dist_incomplete": False}
    for name, src, isize in hand_built_cases() + compressed_cases() + mutated_cases(n_mutations):
        want = zlib_decision(src, isize)
        # exact-size buffers, so that ASan sees any access outside them
        s = ctypes.create_string_buffer(src, len(src)) if src else None
        d = ctypes.create_string_buffer(isize) if isize else None
        got = lib.shim_inflate(s, len(src), d, isize)
        assert got == (want is not None), (name, got, want is not None)
        if got:
            assert (d.raw if isize else b"") == want, name
            counts["accepted"] += 1
        else:
            counts["rejected"] += 1
        if name in required:
            assert (want is not None) == required[name], (name, "zlib decided", want is not None)
    print("OK %d accepted %d rejected" % (counts["accepted"], counts["rejected"]))


# ---------------------------------------------------------------- tests
def _sanitized_shim(tmp_path):
    so = str(tmp_path / "inflate_shim.so")
    errors = []
    # $CXX may be a compiler without the sanitizer runtimes; the system g++ has them
    for cxx in dict.fromkeys(filter(None, [shutil.which(os.environ.get("CXX", "g++")), shutil.which("g++")])):
        proc = subprocess.run([cxx, "-O1", "-g", "-std=c++17", "-fPIC", "-shared", "-fsanitize=address,undefined",
                               "-fno-sanitize-recover=all", "-fno-omit-frame-pointer",
                               os.path.join(HERE, "inflate_host_shim.cpp"), "-o", so], capture_output=True, text=True)
        if proc.returncode == 0:
            asan = subprocess.check_output([cxx, "-print-file-name=libasan.so"], text=True).strip()
            return so, asan
        errors.append(cxx + ": " + proc.stderr[-500:])
    pytest.fail("no C++ compiler builds the sanitized shim:\n" + "\n".join(errors))


def test_device_inflate_equals_zlib_under_sanitizers(tmp_path):
    so, asan = _sanitized_shim(tmp_path)
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="halt_on_error=1:print_stacktrace=1")
    proc = subprocess.run([sys.executable, os.path.abspath(__file__), so, "10000"], env=env, capture_output=True, text=True,
                          timeout=1800)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-6000:]
    assert "OK " in proc.stdout and "runtime error" not in proc.stderr and "AddressSanitizer" not in proc.stderr


def test_block_table_equals_the_python_walk(tmp_path):
    from alntools_b200 import bam_io, bamcols
    path = str(tmp_path / "t.bam")
    refs = [("T%d_A" % t, 100) for t in range(5)]
    bam_io.write_bam(path, refs, [("r%04d" % (i // 3), 0, i % 5) for i in range(5000)], block_payload=900)
    with open(path, "rb") as fh:
        want = list(bam_io.iter_bgzf_blocks(fh))
    with bamcols.BamColumnReader(path) as r:
        for max_bytes in (1, 5000, 1 << 30):
            got, c = [], 0
            while True:
                off, length, isize, end = r.blocks(c, max_bytes)
                if len(off) == 0:
                    assert end == c == os.path.getsize(path)
                    break
                assert len(off) == 1 or end - c <= max_bytes
                start = c
                for o, l, s in zip(off.tolist(), length.tolist(), isize.tolist()):
                    got.append((start, 18 + l + 8, s))
                    assert o == start - c + 18
                    start += 18 + l + 8
                assert start == end
                c = end
            assert got == want
        # a damaged block header: the reader's own error
        with open(path, "rb") as fh:
            data = bytearray(fh.read())
    data[want[30][0]] = 0
    bad = str(tmp_path / "bad.bam")
    with open(bad, "wb") as fh:
        fh.write(bytes(data))
    with bamcols.BamColumnReader(bad) as r:
        with pytest.raises(ValueError) as err:
            r.blocks(0, 1 << 30)
    assert "not a BGZF block at offset %d" % want[30][0] in str(err.value)


def test_device_decode_refuses_what_it_does_not_cover(tmp_path, monkeypatch):
    """These checks come before any file is opened or any GPU is touched."""
    from alntools_b200 import bam_utils, bam_utils_multisample
    missing = str(tmp_path / "missing.bam")
    with pytest.raises(NotImplementedError):
        bam_utils.convert(missing, None, None, devices=2, decode="device")
    with monkeypatch.context() as m:
        m.setenv("WORLD_SIZE", "2")
        m.setenv("RANK", "0")
        with pytest.raises(NotImplementedError):
            bam_utils.convert(missing, None, None, decode="device")
    with monkeypatch.context() as m:
        m.setenv("ALNTOOLS_B200_EMITTER", "python")
        with pytest.raises(NotImplementedError):
            bam_utils.convert(missing, None, None, decode="device")
    with monkeypatch.context() as m:
        m.setenv("ALNTOOLS_B200_DECODE", "device")
        with pytest.raises(NotImplementedError):
            bam_utils_multisample.convert_files([missing], None, None, 1)
        with pytest.raises(NotImplementedError):
            bam_utils.convert(missing, None, None, devices=2)
    with monkeypatch.context() as m:
        m.setenv("ALNTOOLS_B200_DECODE", "gpu")
        with pytest.raises(ValueError):
            bam_utils.convert(missing, None, None)
    with pytest.raises(ValueError):
        bam_utils.convert(missing, None, None, decode="elsewhere")


if __name__ == "__main__":
    run_cases(sys.argv[1], int(sys.argv[2]))
