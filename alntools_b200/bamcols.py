"""ctypes binding of libbamcols.so (include/bamcols.h): the native host column emitter.

BAM file -> int32 columns (read_group, target_idx, hap_idx[, cell_idx]) with the reference's filters
and read-name grouping (alntools/bam_utils.py:253-306, bam_utils_multisample.py:209-300), decoded by
a pool of inflate threads instead of one pysam object per alignment.  `emitter.py` holds the
record-level Python statement of the same rules; tests/test_bamcols.py keeps the two identical.
"""
import ctypes
import os

import numpy as np

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libbamcols.so")
_lib = None

_I32P = ctypes.POINTER(ctypes.c_int32)
SIGNATURES = {
    "bamcols_open": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_char_p, ctypes.c_int]),
    "bamcols_close": (None, [ctypes.c_void_p]),
    "bamcols_last_error": (ctypes.c_char_p, [ctypes.c_void_p]),
    "bamcols_n_references": (ctypes.c_int, [ctypes.c_void_p]),
    "bamcols_reference_name": (ctypes.c_char_p, [ctypes.c_void_p, ctypes.c_int]),
    "bamcols_reference_length": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "bamcols_reference_blob": (ctypes.c_int64, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p),
                                                ctypes.POINTER(ctypes.c_void_p)]),
    "bamcols_set_tables": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]),
    "bamcols_build_tables": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_int64]),
    "bamcols_tables": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32),
                                      ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64),
                                      ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64),
                                      ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                      ctypes.POINTER(ctypes.c_void_p)]),
    "bamcols_cells_create": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p)]),
    "bamcols_cells_destroy": (None, [ctypes.c_void_p]),
    "bamcols_cells_count": (ctypes.c_int64, [ctypes.c_void_p]),
    "bamcols_cells_name": (ctypes.c_char_p, [ctypes.c_void_p, ctypes.c_int64]),
    "bamcols_emit": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                      ctypes.POINTER(ctypes.c_int)]),
    "bamcols_emit_keys": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                           ctypes.c_void_p, ctypes.c_int64, ctypes.POINTER(ctypes.c_int)]),
    "bamcols_all_alignments": (ctypes.c_int64, [ctypes.c_void_p]),
    "bamcols_n_groups": (ctypes.c_int64, [ctypes.c_void_p]),
    "bamcols_plan_shards": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int64)]),
    "bamcols_set_range": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64]),
    "bamcols_track_ranges": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int]),
    "bamcols_ranges": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p)]),
    "bamcols_phase_seconds": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]),
    "bamcols_target_section": (ctypes.c_int64, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]),
    "bamcols_blocks": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    "bamcols_inflate_raw": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int]),
}

BAMCOLS_ERR_IO, BAMCOLS_ERR_FORMAT, BAMCOLS_ERR_INVALID, BAMCOLS_ERR_CELL_FIELD, BAMCOLS_ERR_TID = -1, -2, -3, -4, -5


def load_library(path=None):
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.isfile(p):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'`" % p)
    lib = ctypes.CDLL(p)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    if path is None:
        _lib = lib
    return lib


def inflate_raw(data, out_len, mode=0):
    """Inflate a raw DEFLATE stream of known inflated size with the reader's block decoder.
    mode 0: as the reader does (whole-buffer decoder, zlib for what it declines), 1: zlib only,
    2: whole-buffer decoder only.  Returns the bytes, or None if the decoder said no."""
    lib = load_library()
    buf = ctypes.create_string_buffer(max(1, int(out_len)))
    rc = lib.bamcols_inflate_raw(bytes(data), len(data), buf, int(out_len), int(mode))
    if rc < 0:
        raise ValueError("bamcols_inflate_raw: bad arguments")
    return buf.raw[:out_len] if rc == 1 else None


def _raise(code, msg):
    if code == BAMCOLS_ERR_CELL_FIELD:
        raise IndexError(msg)                      # what the reference raises (bam_utils_multisample.py:273)
    if code == BAMCOLS_ERR_IO:
        raise IOError(msg)
    raise ValueError(msg)


class CellDictionary(object):
    """Cell names of one per-cell job, dense ids in order of first appearance (shared by all files)."""

    def __init__(self):
        self._lib = load_library()
        h = ctypes.c_void_p()
        self._lib.bamcols_cells_create(ctypes.byref(h))
        self._h = h

    def __len__(self):
        return int(self._lib.bamcols_cells_count(self._h))

    def names(self):
        return [self._lib.bamcols_cells_name(self._h, i).decode() for i in range(len(self))]

    def close(self):
        if self._h:
            self._lib.bamcols_cells_destroy(self._h)
            self._h = None

    def __del__(self):
        self.close()


class BamColumnReader(object):
    """One BAM file.  `references` / `lengths` as pysam's; set_tables() then emit()/read_all()."""

    def __init__(self, filename, n_threads=0):
        self._h = None
        self._lib = load_library()
        h = ctypes.c_void_p()
        rc = self._lib.bamcols_open(ctypes.byref(h), os.fsencode(filename), int(n_threads))
        if rc != 0:
            _raise(rc, self._lib.bamcols_last_error(None).decode())
        self._h = h
        self.n_references = int(self._lib.bamcols_n_references(h))
        self._references = self._lengths = None

    def _load_references(self):
        # 200 000 Python strings cost more than decoding a few million alignments: built on first use only
        n = self.n_references
        names, lens = ctypes.c_void_p(), ctypes.c_void_p()
        nbytes = self._lib.bamcols_reference_blob(self._h, ctypes.byref(names), ctypes.byref(lens))
        self._references = tuple(ctypes.string_at(names, nbytes).decode().split("\0")[:n]) if n else ()
        self._lengths = tuple((ctypes.c_int32 * n).from_address(lens.value)) if n else ()

    @property
    def references(self):
        """@SQ names in tid order, as pysam's .references."""
        if self._references is None:
            self._load_references()
        return self._references

    @property
    def lengths(self):
        """@SQ lengths in tid order, as pysam's .lengths."""
        if self._lengths is None:
            self._load_references()
        return self._lengths

    def set_tables(self, tables):
        tt = np.ascontiguousarray(tables.tid_target, dtype=np.int32)
        th = np.ascontiguousarray(tables.tid_hap, dtype=np.int32)
        rc = self._lib.bamcols_set_tables(self._h, tt.ctypes.data, th.ctypes.data, len(tt))
        if rc != 0:
            _raise(rc, self._lib.bamcols_last_error(self._h).decode())

    def build_tables(self, target_filename=None):
        """Header -> TargetTables-compatible object, built natively and installed in this reader."""
        from . import utils
        first = b""
        if target_filename:
            ids = utils.parse_targets(target_filename)
            if len(ids) == 0:                                   # bam_utils.py:577-579
                utils.get_logger().error("Unable to parse target file")
                raise SystemExit(-1)
            first = b"".join(t.encode() + b"\0" for t in ids)
        rc = self._lib.bamcols_build_tables(self._h, first, len(first))
        if rc != 0:
            _raise(rc, self._lib.bamcols_last_error(self._h).decode())
        nt, nh = ctypes.c_int32(), ctypes.c_int32()
        tp, hp_, a, b, c = (ctypes.c_void_p() for _ in range(5))
        tl, hl = ctypes.c_int64(), ctypes.c_int64()
        self._lib.bamcols_tables(self._h, ctypes.byref(nt), ctypes.byref(nh), ctypes.byref(tp), ctypes.byref(tl),
                                 ctypes.byref(hp_), ctypes.byref(hl), ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
        n_ref = self.n_references

        names_blob = ctypes.string_at(tp, tl.value)
        n_targets = nt.value

        class _Tables(object):
            """TargetTables-compatible view of the native tables; the 100 000-entry name structures are only
            built when something asks for them (convert() writes the EC file from target_section())."""
            _main_targets = None

            @property
            def main_targets(self):
                if self._main_targets is None:
                    names = names_blob.decode().split("\0")[:n_targets] if n_targets else []
                    self._main_targets = dict(zip(names, range(len(names))))   # insertion-ordered
                return self._main_targets
        t = _Tables()
        reader = self

        def target_section():
            if reader._h is None:                      # the reader is gone: the caller uses the name list
                return None
            p = ctypes.c_void_p()
            nbytes = reader._lib.bamcols_target_section(reader._h, ctypes.byref(p))
            if nbytes < 0:
                _raise(int(nbytes), reader._lib.bamcols_last_error(reader._h).decode())
            return ctypes.string_at(p, nbytes) if nbytes > 0 else None    # None: non-ASCII names, use the name list
        t.target_section = target_section
        t.haplotypes = ctypes.string_at(hp_, hl.value).decode().split("\0")[:nh.value] if nh.value else []
        t.tid_target = np.array((ctypes.c_int32 * n_ref).from_address(a.value), dtype=np.int32) if n_ref else np.zeros(0, np.int32)
        t.tid_hap = np.array((ctypes.c_int32 * n_ref).from_address(b.value), dtype=np.int32) if n_ref else np.zeros(0, np.int32)
        cells_ = nt.value * nh.value
        t.lengths = (np.array((ctypes.c_int32 * cells_).from_address(c.value), dtype=np.int32).reshape(nt.value, nh.value)
                     if cells_ else np.zeros((nt.value, nh.value), np.int32))
        t.num_targets, t.num_haplotypes = nt.value, nh.value
        return t

    def emit(self, read_group, target_idx, hap_idx, cell_idx=None, cells=None):
        """Fill the given int32 arrays (numpy or pinned torch tensors) with the next whole reads.
        Returns (rows, done)."""
        cap = int(read_group.shape[0])
        done = ctypes.c_int(0)
        ptr = lambda a: None if a is None else (a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr())
        n = self._lib.bamcols_emit(self._h, cells._h if cells is not None else None, ptr(read_group),
                                   ptr(target_idx), ptr(hap_idx), ptr(cell_idx), cap, ctypes.byref(done))
        if n < 0:
            _raise(int(n), self._lib.bamcols_last_error(self._h).decode())
        return int(n), bool(done.value)

    def read_all(self, cells=None, chunk=1 << 20):
        """The whole file as numpy columns: dict(read_group, target_idx, hap_idx[, cell_idx])."""
        parts = []
        while True:
            bufs = [np.empty(chunk, dtype=np.int32) for _ in range(4 if cells is not None else 3)]
            try:
                n, done = self.emit(bufs[0], bufs[1], bufs[2], bufs[3] if cells is not None else None, cells)
            except ValueError as exc:
                if "buffers hold" in str(exc) and chunk < (1 << 28):   # a read longer than the chunk
                    chunk *= 4
                    continue
                raise
            parts.append([b[:n] for b in bufs])
            if done:
                break
        cols = [np.concatenate([p[i] for p in parts]) if len(parts) > 1 else parts[0][i]
                for i in range(len(parts[0]))]
        out = {"read_group": cols[0], "target_idx": cols[1], "hap_idx": cols[2]}
        if cells is not None:
            out["cell_idx"] = cols[3]
        return out

    def emit_keys(self, key_lo, key_hi, target_idx, hap_idx):
        """Fill the given arrays (uint64 / int32 numpy arrays or pinned torch tensors of int64 / int32) with the next
        valid alignments as (name key, target, haplotype) rows, for collation.  Returns (rows, done)."""
        cap = int(key_lo.shape[0])
        done = ctypes.c_int(0)
        ptr = lambda a: a.ctypes.data if isinstance(a, np.ndarray) else a.data_ptr()
        n = self._lib.bamcols_emit_keys(self._h, ptr(key_lo), ptr(key_hi), ptr(target_idx), ptr(hap_idx), cap,
                                        ctypes.byref(done))
        if n < 0:
            _raise(int(n), self._lib.bamcols_last_error(self._h).decode())
        return int(n), bool(done.value)

    def read_all_keys(self, chunk=1 << 20):
        """The whole file as numpy columns: dict(key_lo, key_hi (uint64), target_idx, hap_idx (int32))."""
        parts = []
        while True:
            bufs = [np.empty(chunk, dtype=np.uint64), np.empty(chunk, dtype=np.uint64),
                    np.empty(chunk, dtype=np.int32), np.empty(chunk, dtype=np.int32)]
            n, done = self.emit_keys(*bufs)
            parts.append([b[:n] for b in bufs])
            if done:
                break
        return {k: np.concatenate([p[i] for p in parts]) for i, k in enumerate(("key_lo", "key_hi", "target_idx", "hap_idx"))}

    @property
    def all_alignments(self):
        return int(self._lib.bamcols_all_alignments(self._h))

    def plan_shards(self, n_shards):
        """n_shards + 1 BGZF virtual offsets: shard k holds the records of [v[k], v[k + 1]); every shard starts
        at a read boundary, v[0] is the first record of the file, -1 stands for the end of the file.  What the
        reference's calculate_chunks (bam_utils.py:1174-1304) plans - without the temporary BAM files."""
        v = (ctypes.c_int64 * (int(n_shards) + 1))()
        rc = self._lib.bamcols_plan_shards(self._h, int(n_shards), v)
        if rc != 0:
            _raise(rc, self._lib.bamcols_last_error(self._h).decode())
        return [int(x) for x in v]

    def set_range(self, vbegin, vend=-1):
        """Confine this reader to the records of [vbegin, vend) (virtual offsets of plan_shards); before the
        first emit()."""
        rc = self._lib.bamcols_set_range(self._h, int(vbegin), int(vend))
        if rc != 0:
            _raise(rc, self._lib.bamcols_last_error(self._h).decode())

    def blocks(self, c_begin, max_bytes, max_blocks=1 << 16):
        """The BGZF blocks from compressed offset c_begin on, without inflating them: at most max_blocks blocks whose
        compressed bytes fit in max_bytes (at least one while any is left).  -> (payload_off int64 [counted from
        c_begin], payload_len int32, isize int32, c_end); no blocks at the end of the file."""
        off = np.empty(int(max_blocks), dtype=np.int64)
        length = np.empty(int(max_blocks), dtype=np.int32)
        isize = np.empty(int(max_blocks), dtype=np.int32)
        end = ctypes.c_int64()
        n = self._lib.bamcols_blocks(self._h, int(c_begin), int(max_bytes), int(max_blocks), off.ctypes.data,
                                     length.ctypes.data, isize.ctypes.data, ctypes.byref(end))
        if n < 0:
            _raise(int(n), self._lib.bamcols_last_error(self._h).decode())
        return off[:n], length[:n], isize[:n], int(end.value)

    def track_ranges(self, enable=True):
        rc = self._lib.bamcols_track_ranges(self._h, 1 if enable else 0)
        if rc != 0:
            _raise(rc, self._lib.bamcols_last_error(self._h).decode())

    def ranges(self):
        """(min_pos, max_pos) int32 arrays per reference; min > max where no valid alignment was seen."""
        lo, hi = ctypes.c_void_p(), ctypes.c_void_p()
        n = self._lib.bamcols_ranges(self._h, ctypes.byref(lo), ctypes.byref(hi))
        if n < 0:
            raise ValueError("ranges were not tracked")
        if n == 0:
            return np.zeros(0, np.int32), np.zeros(0, np.int32)
        return (np.array((ctypes.c_int32 * n).from_address(lo.value), dtype=np.int32),
                np.array((ctypes.c_int32 * n).from_address(hi.value), dtype=np.int32))

    def phase_seconds(self):
        """dict phase -> wall-clock seconds so far (single-sample path)."""
        out = (ctypes.c_double * 6)()
        self._lib.bamcols_phase_seconds(self._h, out)
        return dict(zip(("inflate", "record_hop", "validity", "read_starts", "rows", "copy_out"), list(out)))

    @property
    def n_groups(self):
        return int(self._lib.bamcols_n_groups(self._h))

    def close(self):
        if self._h:
            self._lib.bamcols_close(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        self.close()
