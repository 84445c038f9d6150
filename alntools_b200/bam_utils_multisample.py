"""Per-cell (multisample) bam2ec / bam2emase converter: same signature as
alntools/bam_utils_multisample.convert (bam_utils_multisample.py:357).  One BAM file per task, the
cell id is field 14 of the '|||'-split read name, the last read of every file is dropped (:306-308),
cells below the minimum count and ECs left without cells are removed (:595-636).  On several GPUs
(devices=N, ALNTOOLS_GPUS=N or torchrun) every rank takes a contiguous run of the files and the ranks merge
through multi_gpu.distributed_finalize_cells; the EC file is the same bytes.
"""
import glob
import os
import time

import numpy as np

from . import bamcols, bin_utils, emase, emitter, utils
from ._native import EcBuilder
from .header import TargetTables

LOG = utils.get_logger()


class _DecodeAhead(object):
    """A worker thread that decodes the files in order, one ahead of the consumer (a queue of one item): next()
    gives (read_group, target_idx, hap_idx, cell_idx) of the next file, None after the last.  Cell ids come from
    `cells`.  The target tables are built from the first file unless `tables` is given (state["tables"])."""

    def __init__(self, bam_files, cells, target_filename, range_filename, tables=None, n_threads=0):
        import queue
        import threading
        self._queue = queue
        self.state = {"tables": tables, "section": None, "references": None, "lo": None, "hi": None}
        self.ready = queue.Queue(maxsize=1)
        self._stop = threading.Event()
        self.first_tables = threading.Event()
        if tables is not None:
            self.first_tables.set()
        state, ready, stop, first_tables = self.state, self.ready, self._stop, self.first_tables

        def decode():
            try:
                for bam_file in bam_files:
                    if stop.is_set():
                        return
                    with bamcols.BamColumnReader(bam_file, n_threads=n_threads) as reader:
                        if state["tables"] is None:              # tables from the first file only (:399)
                            state["tables"] = reader.build_tables(target_filename)
                            state["section"] = state["tables"].target_section()   # while the reader lives
                            if range_filename is not None:
                                state["references"] = reader.references
                            first_tables.set()
                        else:
                            reader.set_tables(state["tables"])
                        if range_filename is not None:
                            reader.track_ranges(True)
                        c = reader.read_all(cells=cells, chunk=1 << 23)
                        if range_filename is not None:            # merged over the files (:568-576)
                            lo, hi = reader.ranges()
                            state["lo"] = lo if state["lo"] is None else np.minimum(state["lo"], lo)
                            state["hi"] = hi if state["hi"] is None else np.maximum(state["hi"], hi)
                    item = (c["read_group"], c["target_idx"], c["hap_idx"], c["cell_idx"])
                    while not stop.is_set():
                        try:
                            ready.put(item, timeout=0.05)
                            break
                        except queue.Full:
                            continue
                ready.put(None)
            except BaseException as exc:                          # re-raised by the consumer
                first_tables.set()
                ready.put(exc)

        self.worker = threading.Thread(target=decode, daemon=True)
        self.worker.start()

    def first(self):
        """The first item, once the tables exist."""
        self.first_tables.wait()
        return self.next()

    def next(self):
        item = self.ready.get()
        if isinstance(item, BaseException):
            raise item
        return item

    def stop(self):
        # whatever happened, the decode thread has left the native library before the dictionary is closed
        self._stop.set()
        while self.worker.is_alive():
            try:
                self.ready.get_nowait()
            except self._queue.Empty:
                pass
            self.worker.join(timeout=0.05)


def _push_files(builder, ahead, item, base):
    """One push per file (drop_last_group), at order keys from `base` on.  -> alignments pushed."""
    start = base
    while item is not None:
        rg, tg, hp, cell = item
        builder.push(rg, tg, hp, cell, order_base=base, drop_last_group=True)
        base += len(rg)
        item = ahead.next()
    return base - start


def partition_files(sizes, world):
    """Contiguous runs of the file list for `world` ranks, balanced by (compressed) file size: rank r gets files
    [cuts[r], cuts[r + 1]).  A rank may get no file (more ranks than files).  -> world + 1 cuts."""
    n = len(sizes)
    cum = np.concatenate([[0], np.cumsum(np.asarray(sizes, dtype=np.float64))])
    cuts = [0]
    for k in range(1, world):
        target = cum[-1] * k / world
        j = int(np.searchsorted(cum, target))                 # first cut at or beyond the target
        if 0 < j <= n and target - cum[j - 1] < cum[j] - target:
            j -= 1
        cuts.append(min(n, max(cuts[-1], j)))
    cuts.append(n)
    return cuts


def merge_cell_names(name_lists):
    """Global cell ids from the ranks' cell-name lists, taken in rank order: a cell's id is its first appearance
    (the id one CellDictionary over all files in order gives).  -> (global names, per-list int32 maps local id ->
    global id)."""
    ids, names, maps = {}, [], []
    for lst in name_lists:
        m = np.empty(len(lst), dtype=np.int32)
        for i, name in enumerate(lst):
            g = ids.get(name)
            if g is None:
                g = ids[name] = len(names)
                names.append(name)
            m[i] = g
        maps.append(m)
    return names, maps


RANK_STRIDE = 1 << 40      # order keys are rank-major: rank r pushes from r * 2^40 on (see include/ecb200.h)


def convert_files_rank(bam_files, ec_filename, emase_filename, minimum_count, target_filename=None,
                       range_filename=None):
    """One rank of the multi-GPU per-cell convert (one process per GPU; RANK / WORLD_SIZE / LOCAL_RANK / MASTER_*
    in the environment, as torchrun sets them).  The rank decodes its contiguous run of the file list
    (partition_files) with a decode-ahead thread and pushes one file at a time at rank-major order keys; the
    ranks agree on global cell ids (merge_cell_names over all-gathered name lists), merge through
    multi_gpu.distributed_finalize_cells, and every rank writes its byte ranges of the EC file.  Output as the
    one-GPU convert_files.  Returns the totals on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from . import multi_gpu
    start_time = time.time()
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    utils.bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    own_group = not dist.is_initialized()
    if own_group:
        dist.init_process_group("nccl", device_id=device)
    try:
        cuts = partition_files([os.path.getsize(f) for f in bam_files], world)
        mine = bam_files[cuts[rank]:cuts[rank + 1]]
        n_threads = max(1, (os.cpu_count() or 1) // world)      # the host threads are shared by the ranks
        with bamcols.BamColumnReader(bam_files[0], n_threads=1) as reader:   # tables from the first file only (:399)
            tables = reader.build_tables(target_filename)
            section = tables.target_section()
            references = reader.references
        cells = bamcols.CellDictionary()
        ahead = _DecodeAhead(mine, cells, target_filename, range_filename, tables=tables, n_threads=n_threads)
        opts = dict(alignments_hint=0, device=local_rank, result_on_device=1)
        try:
            with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=True, **opts) as builder, \
                    EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=False, **opts) as owner:
                valid = _push_files(builder, ahead, ahead.first(), rank * RANK_STRIDE)
                ahead.stop()
                lists = [None] * world
                dist.all_gather_object(lists, cells.names())
                names, maps = merge_cell_names(lists)
                cell_map = torch.from_numpy(maps[rank]).to(device) if len(maps[rank]) else None
                out = multi_gpu.distributed_finalize_cells(builder, lambda: owner, device, minimum_count, cell_map,
                                                           max(1, len(names)))
                n_ec, id_base = int(out["n_ec"]), int(out["id_base"])
                n_local, nnz_local = int(out["n_ec_local"]), int(out["nnz_local"])
                if n_ec + 1 > 0x7FFFFFFF or out["nnz_a"] > 0x7FFFFFFF or out["nnz_n"] > 0x7FFFFFFF:
                    raise RuntimeError("the EC file's int32 fields cannot hold %d ECs, %d A and %d N non-zeros"
                                       % (n_ec, out["nnz_a"], out["nnz_n"]))
                sizes = [torch.empty(2, dtype=torch.int64, device=device) for _ in range(world)]
                dist.all_gather(sizes, torch.tensor([valid, nnz_local], dtype=torch.int64, device=device))
                sizes = torch.stack(sizes).tolist()
                lo_hi = [torch.empty(2, dtype=torch.int64, device=device) for _ in range(world)]
                dist.all_gather(lo_hi, torch.tensor([id_base, n_local], dtype=torch.int64, device=device))
                lo_hi = torch.stack(lo_hi).tolist()
                nnz_base = sum(sizes[r][1] for r in range(world) if lo_hi[r][1] and lo_hi[r][0] < id_base)
                host = lambda t: t.cpu().numpy()
                a = (host(out["a_indptr"][:n_local + 1]), host(out["a_indices"]), host(out["a_data"]))
                npieces = (host(out["n_indptr"]), host(out["n_col_counts"]), host(out["n_col_offset"]),
                           host(out["n_indices"]), host(out["n_data"]))
                sample_names = [names[c] for c in out["cell_order"].tolist()]
        finally:
            ahead.stop()
            cells.close()
        total_valid = sum(r[0] for r in sizes)
        target_names = list(tables.main_targets.keys()) if (emase_filename or section is None) else None
        if ec_filename:
            header = bin_utils.ec_header_bytes(tables.haplotypes, target_names, tables.lengths, sample_names,
                                               target_section=section, n_targets=tables.num_targets)
            args = (ec_filename, header, n_ec, out["nnz_a"], id_base, nnz_base) + a + npieces
            if rank == 0:
                try:
                    os.remove(ec_filename)
                except OSError:
                    pass
                bin_utils.ecsave2_cells_slice(*args, create=True)
            dist.barrier()                                    # the file is laid out
            if rank != 0:
                bin_utils.ecsave2_cells_slice(*args, create=False)
            dist.barrier()
        if emase_filename:                                    # one writer: the slices travel to rank 0
            parts = [None] * world
            dist.all_gather_object(parts, (id_base, a, npieces))
            if rank == 0:
                a_csr, n_csc = _assemble(parts, n_ec)
                try:
                    os.remove(emase_filename)
                except OSError:
                    pass
                emase.save_emase(emase_filename, "Multisample APM", (tables.num_targets, tables.num_haplotypes, n_ec),
                                 tables.haplotypes, target_names, tables.lengths, sample_names, a_csr, n_csc,
                                 incidence_only=False)
        if range_filename is not None:                        # :638-668, over all ranks' files
            lo, hi = ahead.state["lo"], ahead.state["hi"]
            n_t = len(references)
            lo_t = torch.from_numpy(lo.copy()).to(device) if lo is not None else None
            hi_t = torch.from_numpy(hi.copy()).to(device) if hi is not None else None
            if lo_t is None:                                  # a rank without files: neutral elements
                info = np.iinfo(np.int64)
                lo_t = torch.full((n_t,), info.max, dtype=torch.int64, device=device)
                hi_t = torch.full((n_t,), info.min, dtype=torch.int64, device=device)
            dtype = lo_t.dtype
            lo_t, hi_t = lo_t.to(torch.int64), hi_t.to(torch.int64)
            dist.all_reduce(lo_t, op=dist.ReduceOp.MIN)
            dist.all_reduce(hi_t, op=dist.ReduceOp.MAX)
            if rank == 0:
                utils.write_range_file(range_filename, list(tables.main_targets.keys()), tables.haplotypes,
                                       references, lo_t.to(dtype).cpu().numpy(), hi_t.to(dtype).cpu().numpy())
        if rank != 0:
            return None
        LOG.info("Number of alignments: {:,}".format(total_valid))
        LOG.info("Number of main targets: {:,}".format(tables.num_targets))
        LOG.info("Number of haplotypes: {:,}".format(tables.num_haplotypes))
        LOG.info("Number of ECs after filtering : {:,}".format(n_ec))
        LOG.info("Number of cells after filtering: {:,}".format(len(sample_names)))
        LOG.info("{} GPUs, total time: {}".format(world, utils.format_time(start_time, time.time())))
        return {"n_ec": n_ec, "nnz_a": int(out["nnz_a"]), "n_samples": len(sample_names), "nnz_n": int(out["nnz_n"]),
                "n_alignments": total_valid, "n_gpus": world, "files_per_gpu": [cuts[r + 1] - cuts[r] for r in range(world)]}
    finally:
        if own_group and dist.is_initialized():
            dist.destroy_process_group()


def _assemble(parts, n_ec):
    """The whole matrices from every rank's (id_base, A pieces, N pieces), in id order (EMASE output)."""
    parts = sorted((p for p in parts if len(p[1][0]) > 1), key=lambda p: p[0])
    indptr, at = [np.zeros(1, dtype=np.int64)], 0
    for _, (ip, ix, _d), _n in parts:
        indptr.append(ip[1:].astype(np.int64) + at)
        at += len(ix)
    a_csr = (np.concatenate(indptr).astype(np.int32), np.concatenate([p[1][1] for p in parts]).astype(np.int32),
             np.concatenate([p[1][2] for p in parts]).astype(np.int32))
    n_indptr = parts[0][2][0] if parts else np.zeros(1, dtype=np.int32)
    nnz = int(n_indptr[-1])
    idx, dat = np.empty(nnz, dtype=np.int32), np.empty(nnz, dtype=np.int32)
    for id_base, _a, (ptr, counts, offset, ix, d) in parts:
        counts = counts.astype(np.int64)
        starts = np.cumsum(counts) - counts
        col = np.repeat(np.arange(len(counts)), counts)
        dest = ptr[col].astype(np.int64) + offset[col] + (np.arange(len(ix)) - starts[col])
        idx[dest] = ix + id_base
        dat[dest] = d
    return a_csr, (n_indptr.astype(np.int32), idx, dat)


def _refuse_collation():
    if emitter.collate_mode():
        raise NotImplementedError("the per-cell (--multisample) conversion has no collation by read name: its rules "
                                  "depend on consecutive records (unset ALNTOOLS_B200_COLLATE)")


def convert_files(bam_files, ec_filename, emase_filename, minimum_count, target_filename=None, device=0,
                  range_filename=None, devices=None):
    """The reference's convert() after its glob: files are merged in the given order
    (bam_utils_multisample.py:503-560).  devices=N (or the environment variable ALNTOOLS_GPUS=N) spreads the
    files over N GPUs of this machine, one worker process per GPU (convert_files_rank); the same happens without
    either inside a one-process-per-GPU job (torchrun).  The EC file does not depend on the number of GPUs."""
    if emitter.decode_mode() == "device":
        raise NotImplementedError("the per-cell (--multisample) conversion has no device BAM decode yet: it needs a GPU "
                                  "cell-name dictionary (unset ALNTOOLS_B200_DECODE)")
    _refuse_collation()
    job = dict(bam_files=list(bam_files), ec_filename=ec_filename, emase_filename=emase_filename,
               minimum_count=minimum_count, target_filename=target_filename, range_filename=range_filename)
    if utils.under_launcher() or utils.requested_gpus(devices) > 1:
        if emitter.use_python_emitter():
            raise NotImplementedError("the multi-GPU path needs the native emitter (unset ALNTOOLS_B200_EMITTER)")
        if utils.under_launcher():
            return convert_files_rank(**job)
        return utils.spawn_ranks(utils.requested_gpus(devices), job, body="cells")
    start_time = time.time()
    per_file = []
    total_valid = 0
    if emitter.use_python_emitter():
        header, _ = emitter.read_bam(bam_files[0])            # tables from the first file only (:399)
        tables = TargetTables(header.references, header.lengths, target_filename)
        cell_ids = {}
        for bam_file in bam_files:
            _, records = emitter.read_bam(bam_file)
            cols = emitter.emit_multisample(records, tables, cell_ids)
            per_file.append((cols.read_group, cols.target_idx, cols.hap_idx, cols.cell_idx))
            total_valid += cols.valid_alignments
        cell_names = [None] * len(cell_ids)
        for name, idx in cell_ids.items():
            cell_names[idx] = name
        with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=True,
                       alignments_hint=total_valid, device=device) as builder:
            base = 0
            for rg, tg, hp, cell in per_file:
                builder.push(rg, tg, hp, cell, order_base=base, drop_last_group=True)
                base += len(rg)
            res = builder.finalize(minimum_count)
    else:
        # native emitter: a worker thread decodes file i + 1 while file i is pushed (one push = one file: the file
        # is part of the (file, EC, cell) key and its last read is dropped); at most two files are in host memory
        cells = bamcols.CellDictionary()
        ahead = _DecodeAhead(bam_files, cells, target_filename, range_filename)
        try:
            first = ahead.first()
            tables, section = ahead.state["tables"], ahead.state["section"]
            with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=True,
                           alignments_hint=0, device=device) as builder:
                total_valid = _push_files(builder, ahead, first, 0)
                res = builder.finalize(minimum_count)
        finally:
            ahead.stop()
        state = ahead.state
        cell_names = cells.names()
        cells.close()
        if range_filename is not None:                        # :638-668
            utils.write_range_file(range_filename, list(tables.main_targets.keys()), tables.haplotypes,
                                   state["references"], state["lo"], state["hi"])

    LOG.info("Number of alignments: {:,}".format(total_valid))
    LOG.info("Number of main targets: {:,}".format(tables.num_targets))
    LOG.info("Number of haplotypes: {:,}".format(tables.num_haplotypes))
    LOG.info("Number of ECs after filtering : {:,}".format(res["n_ec"]))
    LOG.info("Number of cells after filtering: {:,}".format(res["n_samples"]))
    sample_names = [cell_names[c] for c in res["cell_order"].tolist()]
    a_csr = (res["a_indptr"], res["a_indices"], res["a_data"])
    n_csc = (res["n_indptr"], res["n_indices"], res["n_data"])
    if emitter.use_python_emitter():
        section = None
    target_names = list(tables.main_targets.keys()) if (emase_filename or section is None) else None
    if emase_filename:
        try:
            os.remove(emase_filename)
        except OSError:
            pass
        emase.save_emase(emase_filename, "Multisample APM",
                         (tables.num_targets, tables.num_haplotypes, res["n_ec"]), tables.haplotypes,
                         target_names, tables.lengths, sample_names, a_csr, n_csc, incidence_only=False)
    if ec_filename:
        try:
            os.remove(ec_filename)
        except OSError:
            pass
        bin_utils.ecsave2_arrays(ec_filename, tables.haplotypes, target_names, tables.lengths, sample_names,
                                 a_csr, n_csc, target_section=section, n_targets=tables.num_targets)
        LOG.info("{} created, total time: {}".format(ec_filename, utils.format_time(start_time, time.time())))
    return res


def convert(bam_filename, ec_filename, emase_filename, num_chunks, minimum_count, number_processes, temp_dir,
            range_filename, target_filename, device=0, devices=None):
    """The reference's per-cell convert: every *.bam of the directory, in filesystem order.  devices /
    ALNTOOLS_GPUS: as convert_files."""
    _refuse_collation()
    if os.path.isfile(bam_filename):                          # :375-377
        LOG.error('bam file must be a directory')
        return None
    bam_files = glob.glob(os.path.join(bam_filename, "*.bam"))  # :379 (filesystem order, as the reference)
    if len(bam_files) == 0:
        LOG.error('No bam files found in directory: {}'.format(bam_filename))
        return None
    if range_filename is not None and emitter.use_python_emitter():
        raise NotImplementedError("--rangefile needs the native emitter (unset ALNTOOLS_B200_EMITTER)")
    return convert_files(bam_files, ec_filename, emase_filename, minimum_count, target_filename, device,
                         range_filename, devices)
