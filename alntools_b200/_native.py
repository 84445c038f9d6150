"""ctypes binding of libecb200.so (C ABI declared in include/ecb200.h).

The library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is no CPU
implementation behind this module: if the shared object is missing or no B200 is visible the
constructors raise.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libecb200.so")

ECB_OPT_RESULT_ON_DEVICE = 1
ECB_OPT_TABLE_SLOTS = 2
ECB_OPT_PAIR_SLOTS = 3
ECB_OPT_GRID_CTAS = 4
ECB_OPT_HOT_CACHE = 5
ECB_OPT_VERIFY_KEYS = 6
ECB_OPT_CHUNK_LEN = 7
ECB_OPT_PAGEABLE_RESULTS = 8
ECB_OPT_BAM_WINDOW = 9
ECB_OPT_COLLATE_SLOTS = 10
ECB_OPT_COLLATE_PIECE = 11
ECB_OPT_COLLATE_BUDGET = 12
ECB_OPT_MAX_READ = 13

ECB_ERR_LIMIT = -4
ECB_ERR_EMPTY = -5
ECB_ERR_STATE = -6
ECB_ERR_FORMAT = -7

_i32p = ctypes.POINTER(ctypes.c_int32)


class EcbResult(ctypes.Structure):
    _fields_ = [
        ("n_ec", ctypes.c_int64), ("nnz_a", ctypes.c_int64),
        ("a_indptr", _i32p), ("a_indices", _i32p), ("a_data", _i32p),
        ("n_samples", ctypes.c_int64), ("nnz_n", ctypes.c_int64),
        ("n_indptr", _i32p), ("n_indices", _i32p), ("n_data", _i32p),
        ("cell_order", _i32p),
        ("n_reads", ctypes.c_int64), ("n_alignments", ctypes.c_int64),
    ]


class EcbStats(ctypes.Structure):
    _fields_ = [
        ("group_ms", ctypes.c_double), ("harvest_ms", ctypes.c_double),
        ("push_ms", ctypes.c_double), ("finalize_ms", ctypes.c_double),
        ("kernel_launches", ctypes.c_int64), ("table_slots", ctypes.c_int64),
        ("table_used", ctypes.c_int64), ("table_grows", ctypes.c_int64),
        ("overflow_reads", ctypes.c_int64), ("h2d_bytes", ctypes.c_int64),
        ("d2h_bytes", ctypes.c_int64), ("row_entries", ctypes.c_int64),
        ("long_reads", ctypes.c_int64), ("long_ms", ctypes.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for cls in reversed(type(self).__mro__)
                for name, _ in cls.__dict__.get("_fields_", ())}


class EcbStatsSamples(EcbStats):
    """ecb_stats since version 2006: EcbStats (the layout up to version 2005), then the fields of the samples
    (ecb_sample_close).  ecb_get_stats writes the whole of it."""
    _fields_ = [("samples", ctypes.c_int64), ("sample_pairs", ctypes.c_int64), ("sample_ms", ctypes.c_double)]


class EcbStatsEcRows(EcbStatsSamples):
    """ecb_stats since version 2007: EcbStatsSamples, then the fields of the EC-row pushes (ecb_push_ecs)."""
    _fields_ = [("ec_pushes", ctypes.c_int64), ("ec_rows", ctypes.c_int64), ("ec_claimed", ctypes.c_int64),
                ("ec_ms", ctypes.c_double), ("ec_check_ms", ctypes.c_double)]


class EcbSlice(ctypes.Structure):
    _i32p = ctypes.POINTER(ctypes.c_int32)
    _fields_ = [("id_base", ctypes.c_int64), ("n_ec", ctypes.c_int64), ("nnz", ctypes.c_int64),
                ("a_indptr", _i32p), ("a_indices", _i32p), ("a_data", _i32p), ("n_data", _i32p)]


class EcbCellsSlice(ctypes.Structure):
    _i32p = ctypes.POINTER(ctypes.c_int32)
    _fields_ = [("n_ec", ctypes.c_int64), ("nnz", ctypes.c_int64),
                ("a_indptr", _i32p), ("a_indices", _i32p), ("a_data", _i32p),
                ("n_samples", ctypes.c_int64), ("nnz_n", ctypes.c_int64),
                ("n_col_counts", _i32p), ("n_indices", _i32p), ("n_data", _i32p)]


class EcbBamStats(ctypes.Structure):
    _fields_ = [
        ("h2d_bytes", ctypes.c_int64), ("inflated_bytes", ctypes.c_int64), ("blocks", ctypes.c_int64),
        ("windows", ctypes.c_int64), ("hop_rounds", ctypes.c_int64), ("records", ctypes.c_int64),
        ("h2d_ms", ctypes.c_double), ("inflate_ms", ctypes.c_double), ("hop_ms", ctypes.c_double),
        ("rules_ms", ctypes.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class EcbSamStats(ctypes.Structure):
    _fields_ = [
        ("bytes", ctypes.c_int64), ("lines", ctypes.c_int64), ("calls", ctypes.c_int64),
        ("h2d_ms", ctypes.c_double), ("lines_ms", ctypes.c_double), ("fields_ms", ctypes.c_double),
        ("rules_ms", ctypes.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class EcbCollateStats(ctypes.Structure):
    _fields_ = [
        ("alignments", ctypes.c_int64), ("reads", ctypes.c_int64), ("table_slots", ctypes.c_int64),
        ("table_grows", ctypes.c_int64), ("pieces", ctypes.c_int64), ("device_bytes", ctypes.c_int64),
        ("h2d_bytes", ctypes.c_int64), ("add_ms", ctypes.c_double), ("table_ms", ctypes.c_double),
        ("order_ms", ctypes.c_double), ("layout_ms", ctypes.c_double), ("push_ms", ctypes.c_double),
        ("spills", ctypes.c_int64), ("groups", ctypes.c_int64), ("host_bytes", ctypes.c_int64),
        ("d2h_bytes", ctypes.c_int64), ("spill_ms", ctypes.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


# every symbol include/ecb200.h declares, with its ctypes signature
SIGNATURES = {
    "ecb_version": (ctypes.c_int, []),
    "ecb_create": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                  ctypes.c_int, ctypes.c_int64]),
    "ecb_set_option": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int64]),
    "ecb_set_stream": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "ecb_arena_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_char_p, ctypes.POINTER(ctypes.c_void_p)]),
    "ecb_arena_open_peer": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]),
    "ecb_arena_reset": (ctypes.c_int, [ctypes.c_void_p]),
    "ecb_rebase": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64]),
    "ecb_order_dispatch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p), ctypes.c_int64,
                                          ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_order_build": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(EcbSlice)]),
    "ecb_export_to_arenas": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p), ctypes.c_int64,
                                            ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_import_arena": (ctypes.c_int, [ctypes.c_void_p]),
    "ecb_cells_summary": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
                                         ctypes.c_void_p]),
    "ecb_cells_order": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                       ctypes.c_int64, ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64),
                                       ctypes.POINTER(ctypes.c_void_p)]),
    "ecb_cells_dispatch_counts": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_int64),
                                                 ctypes.POINTER(ctypes.c_int64), ctypes.c_void_p]),
    "ecb_cells_arena_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_char_p,
                                              ctypes.POINTER(ctypes.c_void_p)]),
    "ecb_cells_export_to_arenas": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p), ctypes.c_int64,
                                                  ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_cells_import_arena": (ctypes.c_int, [ctypes.c_void_p]),
    "ecb_cells_order_dispatch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p), ctypes.c_int64,
                                                ctypes.c_int64, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_cells_order_build": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                             ctypes.POINTER(EcbCellsSlice)]),
    "ecb_push": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.c_int]),
    "ecb_finalize": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.POINTER(EcbResult)]),
    "ecb_sample_close": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    "ecb_finalize_samples": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(EcbResult)]),
    "ecb_push_ecs": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                    ctypes.c_int64, ctypes.c_int64, ctypes.c_int]),
    "ecb_sample_append": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_int64, ctypes.c_int64, ctypes.c_int, ctypes.POINTER(ctypes.c_int64)]),
    "ecb_reset": (ctypes.c_int, [ctypes.c_void_p]),
    "ecb_get_stats": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(EcbStats)]),
    "ecb_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ecb_last_error": (ctypes.c_char_p, [ctypes.c_void_p]),
    "ecb_bam_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_void_p)]),
    "ecb_bam_decode": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                      ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_bam_counters": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_bam_ranges": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ecb_bam_get_stats": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(EcbBamStats)]),
    "ecb_bam_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ecb_sam_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "ecb_sam_parse": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                     ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_void_p),
                                     ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_sam_counters": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "ecb_sam_ranges": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "ecb_sam_get_stats": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(EcbSamStats)]),
    "ecb_sam_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "ecb_collate_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_void_p)]),
    "ecb_collate_add": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_int64, ctypes.c_int]),
    "ecb_collate_push": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    "ecb_collate_get_stats": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(EcbCollateStats)]),
    "ecb_collate_destroy": (ctypes.c_int, [ctypes.c_void_p]),
}

_lib = None


class EcbError(RuntimeError):
    def __init__(self, code, message):
        RuntimeError.__init__(self, "libecb200 error %d: %s" % (code, message))
        self.code = code


def load_library(path=None):
    """dlopen libecb200.so and attach signatures.  Raises if the extension has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or os.environ.get("ECB200_LIB") or LIB_PATH
    if not os.path.isfile(p):
        raise ImportError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback for the EC build)" % p)
    lib = ctypes.CDLL(p)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    if path is None:
        _lib = lib
    return lib


def _ptr(x):
    """Address of a numpy array / torch tensor / raw int; keeps nothing alive."""
    if x is None:
        return None
    if isinstance(x, int):
        return x
    if isinstance(x, np.ndarray):
        if x.dtype != np.int32 or not x.flags["C_CONTIGUOUS"]:
            raise TypeError("columns must be C-contiguous int32 arrays")
        return x.ctypes.data
    if hasattr(x, "data_ptr"):  # torch tensor (host pinned or device); plumbing only
        import torch
        if x.dtype != torch.int32 or not x.is_contiguous():
            raise TypeError("columns must be contiguous int32 tensors")
        return x.data_ptr()
    raise TypeError("unsupported column type %r" % type(x))


class _CudaArray(object):
    """Zero-copy hand-off of library-owned device memory to torch (CUDA array interface)."""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (ptr, False), "version": 2}


def _device_view(ptr, shape, typestr, dtype, device):
    import torch
    if shape[0] == 0 or not ptr:
        return torch.empty(shape, dtype=dtype, device=device)
    return torch.as_tensor(_CudaArray(ptr, shape, typestr), device=device)


def _on_device(x):
    return bool(getattr(x, "is_cuda", False))


class EcBuilder(object):
    """One context = one GPU.  push() columns, finalize() -> dict of numpy int32 arrays.

    Options are the ECB_OPT_* of include/ecb200.h by their names in _OPTIONS.  max_read (ECB_OPT_MAX_READ) is the
    longest read a push accepts: 16384 alignments by default, 0 for the push limit (2^31 - 8192).  Reads longer than
    16384 then take a sort-based pass of their own on the GPU, with the same result as the reference.  The default
    stays at 16384 because in a file grouped by read name a read that long is more often a broken input than a real
    one, and the error says so early."""

    def __init__(self, n_targets, n_haps, with_cells=False, alignments_hint=0, device=0, **options):
        self._lib = load_library()
        self._ctx = ctypes.c_void_p()
        rc = self._lib.ecb_create(ctypes.byref(self._ctx), device, int(n_targets), int(n_haps),
                                  1 if with_cells else 0, int(alignments_hint))
        if rc != 0:
            raise EcbError(rc, self._lib.ecb_last_error(None).decode())
        self.with_cells = bool(with_cells)
        self.device = int(device)               # the CUDA device of this context (not necessarily torch's current one)
        self._result_on_device = False
        for key, value in options.items():
            self.set_option(key, value)

    _OPTIONS = {"result_on_device": ECB_OPT_RESULT_ON_DEVICE, "table_slots": ECB_OPT_TABLE_SLOTS,
                "pair_slots": ECB_OPT_PAIR_SLOTS, "grid_ctas": ECB_OPT_GRID_CTAS,
                "hot_cache": ECB_OPT_HOT_CACHE, "verify_keys": ECB_OPT_VERIFY_KEYS,
                "chunk_len": ECB_OPT_CHUNK_LEN, "pageable_results": ECB_OPT_PAGEABLE_RESULTS,
                "bam_window": ECB_OPT_BAM_WINDOW, "collate_slots": ECB_OPT_COLLATE_SLOTS,
                "collate_piece": ECB_OPT_COLLATE_PIECE, "collate_budget": ECB_OPT_COLLATE_BUDGET,
                "max_read": ECB_OPT_MAX_READ}

    def _check(self, rc):
        if rc != 0:
            raise EcbError(rc, self._lib.ecb_last_error(self._ctx).decode())

    def set_option(self, name, value):
        self._check(self._lib.ecb_set_option(self._ctx, self._OPTIONS[name], int(value)))
        if name == "result_on_device":
            self._result_on_device = bool(value)

    def set_stream(self, cuda_stream):
        """cuda_stream: a cudaStream_t as int (e.g. torch.cuda.current_stream().cuda_stream), or None for
        the library's own stream.  torch reports its default stream as handle 0, which the C ABI reads
        as "own stream"; it is passed as cudaStreamLegacy (0x1), the explicit name of the same stream."""
        if cuda_stream is not None and int(cuda_stream) == 0:
            cuda_stream = 1
        self._check(self._lib.ecb_set_stream(self._ctx, cuda_stream))

    def push(self, read_group, target_idx, hap_idx, cell_idx=None, order_base=0, drop_last_group=False,
             n=None):
        if n is None:
            n = int(read_group.shape[0])
        dev = _on_device(read_group)
        self._check(self._lib.ecb_push(self._ctx, _ptr(read_group), _ptr(target_idx), _ptr(hap_idx),
                                       _ptr(cell_idx), n, int(order_base), 1 if drop_last_group else 0,
                                       1 if dev else 0))

    def finalize_raw(self, min_cell_count=0):
        res = EcbResult()
        self._check(self._lib.ecb_finalize(self._ctx, int(min_cell_count), ctypes.byref(res)))
        return res

    def finalize(self, min_cell_count=0, copy=True):
        """Returns dict(a_indptr, a_indices, a_data, n_indptr, n_indices, n_data[, cell_order]) as
        numpy int32 arrays plus scalar sizes.  copy=False returns VIEWS of the library's result buffers
        (valid until the next finalize / reset / close): the EC file can be written straight from them."""
        if self._result_on_device:
            raise RuntimeError("finalize() needs host results; use finalize_raw() with result_on_device")
        return self._host_result(self.finalize_raw(min_cell_count), copy)

    def close_sample(self):
        """Close the current sample: the alignments pushed since the previous close (or since create / reset) are
        one column of N.  Later pushes take order_base from 0 again (see ecb_sample_close).  -> the sample's
        non-zero entries."""
        nnz = ctypes.c_int64()
        self._check(self._lib.ecb_sample_close(self._ctx, ctypes.byref(nnz)))
        return int(nnz.value)

    def push_ecs(self, a_indptr, a_indices, a_data, order_base=0):
        """The rows of one EC file's A matrix (CSR, int32: indptr, target indices, haplotype masks) as ECs of this
        context, first occurrences at order_base + row (see ecb_push_ecs).  No read is counted.  numpy arrays or
        torch tensors, all on the host or all on this builder's GPU."""
        n_ec = int(a_indptr.shape[0]) - 1
        if n_ec < 0:
            raise ValueError("a_indptr needs at least one entry")
        self._check(self._lib.ecb_push_ecs(self._ctx, _ptr(a_indptr), _ptr(a_indices), _ptr(a_data), n_ec,
                                           int(a_indices.shape[0]), int(order_base), 1 if _on_device(a_indptr) else 0))

    def append_samples(self, n_indptr, n_indices, n_data):
        """Columns of counts (CSC, int32) over the rows of the last push_ecs, closed as samples at once (see
        ecb_sample_append).  -> the non-zero entries added."""
        n_samples = int(n_indptr.shape[0]) - 1
        if n_samples < 0:
            raise ValueError("n_indptr needs at least one entry")
        nnz = ctypes.c_int64()
        self._check(self._lib.ecb_sample_append(self._ctx, _ptr(n_indptr), _ptr(n_indices), _ptr(n_data), n_samples,
                                                int(n_indices.shape[0]), 1 if _on_device(n_indptr) else 0,
                                                ctypes.byref(nnz)))
        return int(nnz.value)

    def finalize_samples_raw(self):
        res = EcbResult()
        self._check(self._lib.ecb_finalize_samples(self._ctx, ctypes.byref(res)))
        return res

    def finalize_samples(self, copy=True):
        """As finalize(), with N holding one column per closed sample (ecb_finalize_samples)."""
        if self._result_on_device:
            raise RuntimeError("finalize_samples() needs host results; use finalize_samples_raw() with "
                               "result_on_device")
        return self._host_result(self.finalize_samples_raw(), copy)

    def _host_result(self, res, copy):
        def arr(ptr, n):
            if n == 0:
                return np.zeros(0, dtype=np.int32)
            view = np.ctypeslib.as_array(ptr, shape=(n,))
            return view.copy() if copy else view

        out = {
            "n_ec": res.n_ec, "nnz_a": res.nnz_a, "n_samples": res.n_samples, "nnz_n": res.nnz_n,
            "n_reads": res.n_reads, "n_alignments": res.n_alignments,
            "a_indptr": arr(res.a_indptr, res.n_ec + 1),
            "a_indices": arr(res.a_indices, res.nnz_a),
            "a_data": arr(res.a_data, res.nnz_a),
            "n_indptr": arr(res.n_indptr, res.n_samples + 1),
            "n_indices": arr(res.n_indices, res.nnz_n),
            "n_data": arr(res.n_data, res.nnz_n),
        }
        if self.with_cells:
            out["cell_order"] = arr(res.cell_order, res.n_samples)
        return out

    def reset(self):
        self._check(self._lib.ecb_reset(self._ctx))

    # ---- multi-GPU exchange: CUDA IPC arenas (see include/ecb200.h and multi_gpu.py) ---------------
    def arena_create(self, cap_records):
        """-> (64-byte IPC handle, base address) of this OWNER context's arena (cap_records records of 32 bytes)."""
        handle = ctypes.create_string_buffer(64)
        base = ctypes.c_void_p()
        self._check(self._lib.ecb_arena_create(self._ctx, int(cap_records), handle, ctypes.byref(base)))
        return handle.raw, int(base.value)

    def arena_open_peer(self, handle):
        base = ctypes.c_void_p()
        self._check(self._lib.ecb_arena_open_peer(self._ctx, ctypes.create_string_buffer(handle, 64), ctypes.byref(base)))
        return int(base.value)

    def arena_reset(self):
        self._check(self._lib.ecb_arena_reset(self._ctx))

    def rebase(self, delta):
        """Shift the order key of everything pushed so far by `delta` (see ecb_rebase in include/ecb200.h)."""
        self._check(self._lib.ecb_rebase(self._ctx, int(delta)))

    def export_to_arenas(self, bases, cap_records):
        """Dispatch 1: every EC of this LOCAL context as {key, first, count} into the arena of its owner rank.
        -> (min_base, max_end) of the positions pushed here."""
        arr = (ctypes.c_void_p * len(bases))(*bases)
        lo, hi = ctypes.c_int64(), ctypes.c_int64()
        self._check(self._lib.ecb_export_to_arenas(self._ctx, len(bases), arr, int(cap_records), ctypes.byref(lo), ctypes.byref(hi)))
        return int(lo.value), int(hi.value)

    def import_arena(self):
        self._check(self._lib.ecb_import_arena(self._ctx))

    def order_dispatch(self, bases, cap_records, shard_lo, shard_hi):
        """Dispatch 2: every merged EC of this OWNER context as {key, position inside its shard, count} to the rank
        whose shard of the read order holds its first occurrence (shard_lo / shard_hi: one entry per rank)."""
        arr = (ctypes.c_void_p * len(bases))(*bases)
        lo = (ctypes.c_int64 * len(bases))(*[int(x) for x in shard_lo])
        hi = (ctypes.c_int64 * len(bases))(*[int(x) for x in shard_hi])
        self._check(self._lib.ecb_order_dispatch(self._ctx, len(bases), arr, int(cap_records), lo, hi))

    def order_build(self, local, shard_lo, shard_hi):
        """-> dict(n_ec, nnz, a_indptr, a_indices, a_data, n_data): the ECs whose first occurrence lies in this
        rank's shard, in id order, rows taken from `local` (the builder that holds this rank's reads), as torch
        views of library memory (valid until the next call on this context)."""
        import torch
        sl = EcbSlice()
        self._check(self._lib.ecb_order_build(self._ctx, local._ctx, int(shard_lo), int(shard_hi), ctypes.byref(sl)))
        dev = torch.device("cuda", torch.cuda.current_device())
        view = lambda p, n: _device_view(ctypes.cast(p, ctypes.c_void_p).value, (n,), "<i4", torch.int32, dev)
        return {"n_ec": int(sl.n_ec), "nnz": int(sl.nnz), "a_indptr": view(sl.a_indptr, sl.n_ec + 1),
                "a_indices": view(sl.a_indices, max(sl.nnz, 1))[:sl.nnz], "a_data": view(sl.a_data, max(sl.nnz, 1))[:sl.nnz],
                "n_data": view(sl.n_data, max(sl.n_ec, 1))[:sl.n_ec]}

    # ---- per-cell exchange (see include/ecb200.h and multi_gpu.distributed_finalize_cells) ------------------
    def cells_summary(self, cell_map, n_cells):
        """-> (cell_key, cell_total): int64 device tensors [n_cells] (uint64 bit patterns) indexed by GLOBAL cell id:
        this LOCAL context's sort key of every cell (-1 = ~0 when absent) and its reads here.  cell_map: int32
        device tensor local id -> global id, or None (identity)."""
        import torch
        dev = torch.device("cuda", torch.cuda.current_device())
        key = torch.empty(int(n_cells), dtype=torch.int64, device=dev)
        total = torch.empty(int(n_cells), dtype=torch.int64, device=dev)
        self._check(self._lib.ecb_cells_summary(self._ctx, _ptr(cell_map), 0 if cell_map is None else int(cell_map.numel()),
                                                int(n_cells), key.data_ptr(), total.data_ptr()))
        return key, total

    def cells_order(self, cell_keys, cell_totals, min_cell_count, cell_map, world):
        """The cell decision from the gathered keys [world * n_cells] and summed totals [n_cells] (int64 device
        tensors).  -> (n_samples, cell_order: int32 device view [n_samples] of global cell ids)."""
        import torch
        n_samples, order = ctypes.c_int64(), ctypes.c_void_p()
        self._check(self._lib.ecb_cells_order(self._ctx, int(world), cell_keys.data_ptr(), cell_totals.data_ptr(),
                                              int(cell_totals.numel()), int(min_cell_count), _ptr(cell_map),
                                              ctypes.byref(n_samples), ctypes.byref(order)))
        dev = torch.device("cuda", torch.cuda.current_device())
        return int(n_samples.value), _device_view(order.value, (int(n_samples.value),), "<i4", torch.int32, dev)

    def cells_dispatch_counts(self, world, shard_lo=None, shard_hi=None):
        """-> int64 device tensor [2 * world]: records of the next dispatch per destination rank (ECs, then pairs).
        Without shards: dispatch 1 of this LOCAL context; with them: dispatch 2 of this OWNER context."""
        import torch
        counts = torch.empty(2 * int(world), dtype=torch.int64, device=torch.device("cuda", torch.cuda.current_device()))
        lo = hi = None
        if shard_lo is not None:
            lo = (ctypes.c_int64 * world)(*[int(x) for x in shard_lo])
            hi = (ctypes.c_int64 * world)(*[int(x) for x in shard_hi])
        self._check(self._lib.ecb_cells_dispatch_counts(self._ctx, int(world), lo, hi, counts.data_ptr()))
        return counts

    def cells_arena_create(self, cap_ec, cap_pairs):
        """-> (64-byte IPC handle, base address) of this OWNER context's per-cell arena; replaces an earlier one."""
        handle = ctypes.create_string_buffer(64)
        base = ctypes.c_void_p()
        self._check(self._lib.ecb_cells_arena_create(self._ctx, int(cap_ec), int(cap_pairs), handle, ctypes.byref(base)))
        return handle.raw, int(base.value)

    def cells_export_to_arenas(self, bases, cap_ec, cap_pairs):
        """Dispatch 1 of the per-cell exchange.  -> (min_base, max_end) of the positions pushed here."""
        arr = (ctypes.c_void_p * len(bases))(*bases)
        lo, hi = ctypes.c_int64(), ctypes.c_int64()
        self._check(self._lib.ecb_cells_export_to_arenas(self._ctx, len(bases), arr, int(cap_ec), int(cap_pairs),
                                                         ctypes.byref(lo), ctypes.byref(hi)))
        return int(lo.value), int(hi.value)

    def cells_import_arena(self):
        self._check(self._lib.ecb_cells_import_arena(self._ctx))

    def cells_order_dispatch(self, bases, cap_ec, cap_pairs, shard_lo, shard_hi):
        arr = (ctypes.c_void_p * len(bases))(*bases)
        lo = (ctypes.c_int64 * len(bases))(*[int(x) for x in shard_lo])
        hi = (ctypes.c_int64 * len(bases))(*[int(x) for x in shard_hi])
        self._check(self._lib.ecb_cells_order_dispatch(self._ctx, len(bases), arr, int(cap_ec), int(cap_pairs), lo, hi))

    def cells_order_build(self, local, shard_lo, shard_hi, n_samples):
        """-> dict(n_ec, nnz, a_indptr, a_indices, a_data, nnz_n, n_col_counts, n_indices, n_data): this rank's slice
        as torch views of library memory (valid until the next call on this context); n_indices are local to
        the slice."""
        import torch
        sl = EcbCellsSlice()
        self._check(self._lib.ecb_cells_order_build(self._ctx, local._ctx, int(shard_lo), int(shard_hi), int(n_samples),
                                                    ctypes.byref(sl)))
        dev = torch.device("cuda", torch.cuda.current_device())
        view = lambda p, n: _device_view(ctypes.cast(p, ctypes.c_void_p).value, (max(n, 1),), "<i4", torch.int32, dev)[:n]
        return {"n_ec": int(sl.n_ec), "nnz": int(sl.nnz), "a_indptr": view(sl.a_indptr, sl.n_ec + 1),
                "a_indices": view(sl.a_indices, sl.nnz), "a_data": view(sl.a_data, sl.nnz), "nnz_n": int(sl.nnz_n),
                "n_col_counts": view(sl.n_col_counts, sl.n_samples), "n_indices": view(sl.n_indices, sl.nnz_n),
                "n_data": view(sl.n_data, sl.nnz_n)}

    def stats(self):
        st = EcbStatsEcRows()
        self._check(self._lib.ecb_get_stats(self._ctx, ctypes.byref(st)))
        return st.as_dict()

    def close(self):
        if self._ctx:
            self._lib.ecb_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class BamDecoder(object):
    """Device decode of one single-sample BAM file on `builder`'s context (ecb_bam_* in include/ecb200.h): BGZF
    blocks in, the columns bamcols_emit produces out, in device memory.  Malformed input raises ValueError, as the
    host reader (bamcols) does for the same file."""

    def __init__(self, builder, tid_target, tid_hap, track_ranges=False):
        self._lib = builder._lib
        self._builder = builder                   # the decoder lives in the builder's context: keep it alive
        self._h = ctypes.c_void_p()
        self.n_references = len(tid_target)
        tt = np.ascontiguousarray(tid_target, dtype=np.int32)
        th = np.ascontiguousarray(tid_hap, dtype=np.int32)
        self._check(self._lib.ecb_bam_create(builder._ctx, tt.ctypes.data, th.ctypes.data, len(tt),
                                             1 if track_ranges else 0, ctypes.byref(self._h)))

    def _check(self, rc):
        if rc == 0:
            return
        msg = self._lib.ecb_last_error(self._builder._ctx).decode()
        if rc == ECB_ERR_FORMAT:
            raise ValueError(msg)
        raise EcbError(rc, msg)

    def decode(self, data, payload_off, payload_len, isize, skip=0, last=False, n_bytes=None):
        """data: compressed bytes (pinned uint8 tensor preferred, or a numpy array / bytes); the block table as from
        BamColumnReader.blocks().  -> (read_group, target_idx, hap_idx): int32 torch views of the device rows of
        every read closed so far, valid until the next call."""
        import torch
        if isinstance(data, (bytes, bytearray)):
            data = np.frombuffer(data, dtype=np.uint8)
        ptr = data.data_ptr() if hasattr(data, "data_ptr") else data.ctypes.data
        n_bytes = int(data.shape[0]) if n_bytes is None else int(n_bytes)
        off = np.ascontiguousarray(payload_off, dtype=np.int64)
        length = np.ascontiguousarray(payload_len, dtype=np.int32)
        size = np.ascontiguousarray(isize, dtype=np.int32)
        rg, tg, hp = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        rows = ctypes.c_int64()
        self._check(self._lib.ecb_bam_decode(self._h, ptr, n_bytes, off.ctypes.data, length.ctypes.data, size.ctypes.data,
                                             len(off), int(skip), 1 if last else 0, ctypes.byref(rg), ctypes.byref(tg),
                                             ctypes.byref(hp), ctypes.byref(rows)))
        n = int(rows.value)
        dev = torch.device("cuda", self._builder.device)   # the rows live on the builder's GPU
        return tuple(_device_view(p.value, (n,), "<i4", torch.int32, dev) for p in (rg, tg, hp))

    def counters(self):
        """-> (all_alignments, n_groups): records seen so far and reads started."""
        a, g = ctypes.c_int64(), ctypes.c_int64()
        self._check(self._lib.ecb_bam_counters(self._h, ctypes.byref(a), ctypes.byref(g)))
        return int(a.value), int(g.value)

    def ranges(self):
        """(min_pos, max_pos) int32 arrays per reference, as BamColumnReader.ranges()."""
        lo = np.empty(self.n_references, dtype=np.int32)
        hi = np.empty(self.n_references, dtype=np.int32)
        self._check(self._lib.ecb_bam_ranges(self._h, lo.ctypes.data, hi.ctypes.data))
        return lo, hi

    def stats(self):
        st = EcbBamStats()
        self._check(self._lib.ecb_bam_get_stats(self._h, ctypes.byref(st)))
        return st.as_dict()

    def close(self):
        if self._h:
            self._lib.ecb_bam_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SamDecoder(object):
    """Device parse of single-sample SAM text on `builder`'s context (ecb_sam_* in include/ecb200.h): whole alignment
    lines in, the columns BamDecoder gives for the same alignments as BAM out, in device memory.  references: the @SQ
    names in header order (str); first_line: the line number of the first byte of the first call.  A bad line raises
    ValueError with "line N: <what>"."""

    def __init__(self, builder, references, tid_target, tid_hap, first_line=1, track_ranges=False):
        self._lib = builder._lib
        self._builder = builder                   # the decoder lives in the builder's context: keep it alive
        self._h = ctypes.c_void_p()
        self.n_references = len(tid_target)
        names = [r.encode() for r in references]
        blob = b"".join(names)
        off = np.zeros(len(names) + 1, dtype=np.int64)
        np.cumsum([len(n) for n in names], out=off[1:])
        tt = np.ascontiguousarray(tid_target, dtype=np.int32)
        th = np.ascontiguousarray(tid_hap, dtype=np.int32)
        self._check(self._lib.ecb_sam_create(builder._ctx, blob, off.ctypes.data, len(tt), tt.ctypes.data, th.ctypes.data,
                                             int(first_line), 1 if track_ranges else 0, ctypes.byref(self._h)))

    def _check(self, rc):
        if rc == 0:
            return
        msg = self._lib.ecb_last_error(self._builder._ctx).decode()
        if rc == ECB_ERR_FORMAT:
            raise ValueError(msg)
        raise EcbError(rc, msg)

    def parse(self, data, n_bytes=None, last=False):
        """data: text bytes (pinned uint8 tensor preferred, or a numpy array / bytes), its first n_bytes whole lines.
        -> (read_group, target_idx, hap_idx): int32 torch views of the device rows of every read closed so far, valid
        until the next call."""
        import torch
        if isinstance(data, (bytes, bytearray)):
            data = np.frombuffer(data, dtype=np.uint8)
        ptr = data.data_ptr() if hasattr(data, "data_ptr") else data.ctypes.data
        n_bytes = int(data.shape[0]) if n_bytes is None else int(n_bytes)
        rg, tg, hp = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        rows = ctypes.c_int64()
        self._check(self._lib.ecb_sam_parse(self._h, ptr if n_bytes else None, n_bytes, 1 if last else 0,
                                            ctypes.byref(rg), ctypes.byref(tg), ctypes.byref(hp), ctypes.byref(rows)))
        n = int(rows.value)
        dev = torch.device("cuda", self._builder.device)
        return tuple(_device_view(p.value, (n,), "<i4", torch.int32, dev) for p in (rg, tg, hp))

    def counters(self):
        """-> (all_alignments, n_groups): alignment lines seen so far and reads started."""
        a, g = ctypes.c_int64(), ctypes.c_int64()
        self._check(self._lib.ecb_sam_counters(self._h, ctypes.byref(a), ctypes.byref(g)))
        return int(a.value), int(g.value)

    def ranges(self):
        """(min_pos, max_pos) int32 arrays per reference, as BamDecoder.ranges()."""
        lo = np.empty(self.n_references, dtype=np.int32)
        hi = np.empty(self.n_references, dtype=np.int32)
        self._check(self._lib.ecb_sam_ranges(self._h, lo.ctypes.data, hi.ctypes.data))
        return lo, hi

    def stats(self):
        st = EcbSamStats()
        self._check(self._lib.ecb_sam_get_stats(self._h, ctypes.byref(st)))
        return st.as_dict()

    def close(self):
        if self._h:
            self._lib.ecb_sam_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _column_ptr(x, dtypes):
    """Address of a contiguous numpy array or torch tensor (host or device) of one of `dtypes` (numpy dtype names)."""
    if isinstance(x, np.ndarray):
        if x.dtype.name not in dtypes or not x.flags["C_CONTIGUOUS"]:
            raise TypeError("expected a C-contiguous array of %s, got %s" % ("/".join(dtypes), x.dtype))
        return x.ctypes.data
    if hasattr(x, "data_ptr"):
        if str(x.dtype).replace("torch.", "") not in dtypes or not x.is_contiguous():
            raise TypeError("expected a contiguous tensor of %s, got %s" % ("/".join(dtypes), x.dtype))
        return x.data_ptr()
    raise TypeError("unsupported column type %r" % type(x))


class Collator(object):
    """Collation by read name on `builder`'s context (ecb_collate_* in include/ecb200.h): add() the rows of
    BamColumnReader.emit_keys in file order, then push() regroups them on the GPU and pushes them into the builder as
    name-grouped reads."""

    def __init__(self, builder):
        self._lib = builder._lib
        self._builder = builder                   # the collator lives in the builder's context: keep it alive
        self._h = ctypes.c_void_p()
        self._check(self._lib.ecb_collate_create(builder._ctx, ctypes.byref(self._h)))

    def _check(self, rc):
        if rc != 0:
            raise EcbError(rc, self._lib.ecb_last_error(self._builder._ctx).decode())

    def add(self, key_lo, key_hi, target_idx, hap_idx, n=None):
        """key_lo / key_hi: uint64 (numpy) or int64 / uint64 (torch) columns; target_idx / hap_idx: int32.  numpy
        arrays, pinned host tensors or device tensors on the builder's GPU; the first n rows (default: all)."""
        if n is None:
            n = int(key_lo.shape[0])
        wide = ("uint64", "int64")
        self._check(self._lib.ecb_collate_add(self._h, _column_ptr(key_lo, wide), _column_ptr(key_hi, wide),
                                              _column_ptr(target_idx, ("int32",)), _column_ptr(hap_idx, ("int32",)),
                                              int(n), 1 if _on_device(key_lo) else 0))

    def push(self):
        """Regroup everything added and push it into the builder; -> number of reads."""
        n_reads = ctypes.c_int64()
        self._check(self._lib.ecb_collate_push(self._h, ctypes.byref(n_reads)))
        return int(n_reads.value)

    def stats(self):
        st = EcbCollateStats()
        self._check(self._lib.ecb_collate_get_stats(self._h, ctypes.byref(st)))
        return st.as_dict()

    def close(self):
        if self._h:
            self._lib.ecb_collate_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
