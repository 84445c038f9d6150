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

from . import bamcols, bin_utils, emitter, utils
from ._native import EcBuilder
from .header import TargetTables

LOG = utils.get_logger()


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


def _tables(bam_file, target_filename, with_references):
    """The job's target tables, built from the first file only (:399), with their targets section and, if asked
    for, the header's reference names: both are read while the file's reader is open."""
    with bamcols.BamColumnReader(bam_file, n_threads=1) as reader:
        tables = reader.build_tables(target_filename)
        return tables, tables.target_section(), reader.references if with_references else None


def convert_files_rank(bam_files, ec_filename, emase_filename, minimum_count, target_filename=None,
                       range_filename=None):
    """One rank of the multi-GPU per-cell convert (one process per GPU; RANK / WORLD_SIZE / LOCAL_RANK / MASTER_*
    in the environment, as torchrun sets them).  The rank decodes its contiguous run of the file list
    (partition_files) with emitter.stream_files and pushes one file at a time at rank-major order keys; the
    ranks agree on global cell ids (merge_cell_names over all-gathered name lists), merge through
    multi_gpu.distributed_finalize_cells, and every rank writes its byte ranges of the EC file
    (multi_gpu.save_rank_outputs).  Output as the one-GPU convert_files.  Returns the totals on rank 0, None
    elsewhere."""
    import torch
    import torch.distributed as dist
    from . import multi_gpu
    start_time = time.time()
    limit = emitter.max_read()
    with multi_gpu.rank_process() as (rank, world, device):
        cuts = partition_files([os.path.getsize(f) for f in bam_files], world)
        n_threads = max(1, (os.cpu_count() or 1) // world)      # the host threads are shared by the ranks
        tables, section, references = _tables(bam_files[0], target_filename, range_filename is not None)
        cells = bamcols.CellDictionary()
        opts = dict(alignments_hint=0, device=device.index, result_on_device=1)
        try:
            with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=True, max_read=limit, **opts) as builder, \
                    EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=False, **opts) as owner:
                valid, ranges = emitter.stream_files(bam_files[cuts[rank]:cuts[rank + 1]], tables, cells, builder,
                                                     rank * RANK_STRIDE, n_threads, range_filename is not None)
                total_valid = torch.tensor([valid], dtype=torch.int64, device=device)
                dist.all_reduce(total_valid)
                lists = [None] * world
                dist.all_gather_object(lists, cells.names())
                names, maps = merge_cell_names(lists)
                cell_map = torch.from_numpy(maps[rank]).to(device) if len(maps[rank]) else None
                out = multi_gpu.distributed_finalize_cells(builder, lambda: owner, device, minimum_count, cell_map,
                                                           max(1, len(names)))
                sample_names = [names[c] for c in out["cell_order"].tolist()]
                multi_gpu.save_rank_outputs(out, tables, section, sample_names, ec_filename, emase_filename,
                                            range_filename, references, ranges)
        finally:
            cells.close()
        if rank != 0:
            return None
        n_ec, total_valid = int(out["n_ec"]), int(total_valid.item())
        LOG.info("Number of alignments: {:,}".format(total_valid))
        LOG.info("Number of main targets: {:,}".format(tables.num_targets))
        LOG.info("Number of haplotypes: {:,}".format(tables.num_haplotypes))
        LOG.info("Number of ECs after filtering : {:,}".format(n_ec))
        LOG.info("Number of cells after filtering: {:,}".format(len(sample_names)))
        LOG.info("{} GPUs, total time: {}".format(world, utils.format_time(start_time, time.time())))
        return {"n_ec": n_ec, "nnz_a": int(out["nnz_a"]), "n_samples": len(sample_names), "nnz_n": int(out["nnz_n"]),
                "n_alignments": total_valid, "n_gpus": world, "files_per_gpu": [cuts[r + 1] - cuts[r] for r in range(world)]}


def convert_files(bam_files, ec_filename, emase_filename, minimum_count, target_filename=None, device=0,
                  range_filename=None, devices=None):
    """The reference's convert() after its glob: files are merged in the given order
    (bam_utils_multisample.py:503-560).  devices=N (or the environment variable ALNTOOLS_GPUS=N) spreads the
    files over N GPUs of this machine, one worker process per GPU (convert_files_rank); the same happens without
    either inside a one-process-per-GPU job (torchrun).  The EC file does not depend on the number of GPUs.
    ALNTOOLS_B200_MAX_READ: the longest read accepted, as for the single-sample convert (emitter.max_read)."""
    mode = emitter.resolve_mode(True, devices, range_file=range_filename is not None)
    limit = emitter.max_read()
    bam_files = list(bam_files)
    if not bam_files:
        raise ValueError("convert_files needs at least one BAM file")
    job = dict(bam_files=bam_files, ec_filename=ec_filename, emase_filename=emase_filename,
               minimum_count=minimum_count, target_filename=target_filename, range_filename=range_filename)
    if mode.launcher:
        return convert_files_rank(**job)
    if mode.gpus > 1:
        return utils.spawn_ranks(mode.gpus, job, body="cells")
    start_time = time.time()
    references = ranges = None
    if mode.python:
        header, _ = emitter.read_bam(bam_files[0])            # tables from the first file only (:399)
        tables = TargetTables(header.references, header.lengths, target_filename)
        section = tables.target_section()
        per_file = []
        cell_ids = {}
        for bam_file in bam_files:
            _, records = emitter.read_bam(bam_file)
            per_file.append(emitter.emit_multisample(records, tables, cell_ids))
        total_valid = sum(cols.valid_alignments for cols in per_file)
        cell_names = [None] * len(cell_ids)
        for name, idx in cell_ids.items():
            cell_names[idx] = name
        with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=True,
                       alignments_hint=total_valid, device=device, max_read=limit) as builder:
            base = 0
            for cols in per_file:
                builder.push(cols.read_group, cols.target_idx, cols.hap_idx, cols.cell_idx, order_base=base,
                             drop_last_group=True)
                base += len(cols.read_group)
            res = builder.finalize(minimum_count)
    else:
        # native emitter: file i + 1 is decoded while file i is pushed
        tables, section, references = _tables(bam_files[0], target_filename, range_filename is not None)
        cells = bamcols.CellDictionary()
        try:
            with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=True,
                           alignments_hint=0, device=device, max_read=limit) as builder:
                total_valid, ranges = emitter.stream_files(bam_files, tables, cells, builder,
                                                           track_ranges=range_filename is not None)
                res = builder.finalize(minimum_count)
            cell_names = cells.names()
        finally:
            cells.close()

    LOG.info("Number of alignments: {:,}".format(total_valid))
    LOG.info("Number of main targets: {:,}".format(tables.num_targets))
    LOG.info("Number of haplotypes: {:,}".format(tables.num_haplotypes))
    LOG.info("Number of ECs after filtering : {:,}".format(res["n_ec"]))
    LOG.info("Number of cells after filtering: {:,}".format(res["n_samples"]))
    bin_utils.save_outputs(tables, section, [cell_names[c] for c in res["cell_order"].tolist()],
                           (res["a_indptr"], res["a_indices"], res["a_data"]),
                           (res["n_indptr"], res["n_indices"], res["n_data"]), True, ec_filename, emase_filename,
                           range_filename, references, ranges)
    if ec_filename:
        LOG.info("{} created, total time: {}".format(ec_filename, utils.format_time(start_time, time.time())))
    return res


def convert(bam_filename, ec_filename, emase_filename, num_chunks, minimum_count, number_processes, temp_dir,
            range_filename, target_filename, device=0, devices=None):
    """The reference's per-cell convert: every *.bam of the directory, in filesystem order.  devices /
    ALNTOOLS_GPUS: as convert_files."""
    emitter.resolve_mode(True, devices, range_file=range_filename is not None)   # refusals before the directory is read
    emitter.max_read()
    if os.path.isfile(bam_filename):                          # :375-377
        LOG.error('bam file must be a directory')
        return None
    bam_files = glob.glob(os.path.join(bam_filename, "*.bam"))  # :379 (filesystem order, as the reference)
    if len(bam_files) == 0:
        LOG.error('No bam files found in directory: {}'.format(bam_filename))
        return None
    return convert_files(bam_files, ec_filename, emase_filename, minimum_count, target_filename, device,
                         range_filename, devices)
