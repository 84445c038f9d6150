"""Single-sample bam2ec / bam2emase converter: same signature as alntools/bam_utils.convert
(bam_utils.py:512), with the grouping, counting, ordering and matrix build on the GPU.

Call stack: convert -> header tables (host) -> column emitter (host decode + filters + name compare)
-> EcBuilder.push (H2D + sm_100a kernels) -> EcBuilder.finalize (CSR A, CSC N) -> EC file writer.
"""
import multiprocessing
import collections
import os
import time

import numpy as np

from . import bam_io, bamcols, bin_utils, emitter, utils
from ._native import EcBuilder
from .header import TargetTables

LOG = utils.get_logger()


# ---- the reference's chunk-worker interface (bam_utils.py:30-62, 157-195, 198-363, 490-498) -------------
# convert() below does not use it - it decodes the file once and streams it to the GPU - but code that drives
# the reference's workers directly (a ConvertParams per process, wrapper_convert through Pool.imap, results
# merged in chunk order) finds the same names, fields and results here.
ParseRecord = collections.namedtuple("ParseRecord", ["header_size", "begin_read_offset", "begin_read_size",
                                                     "file_offset", "file_bytes", "end_read_offset", "end_read_size"])


class ConvertParams(object):
    slots = ['input_file', 'temp_dir', 'process_id', 'track_ranges', 'data']

    def __init__(self):
        self.input_file = None
        self.temp_dir = None
        self.process_id = None
        self.track_ranges = False
        self.data = []                      # tuples of (idx, ParseRecord)

    def __str__(self):
        return "Input: {}\nProcess ID: {}\nData: {}".format(self.input_file, self.process_id, self.data)


class ConvertResults(object):
    slots = ['valid_alignments', 'all_alignments', 'ec', 'unique_reads', 'init', 'tid_ranges']

    def __init__(self):
        self.valid_alignments = None
        self.all_alignments = None
        self.ec = None
        self.unique_reads = None
        self.init = False
        self.tid_ranges = None


def chunk_bam_file(bam_filename, new_filename, parse_rec):
    """A BAM file holding one chunk of `bam_filename` (bam_utils.py:157-195): the header blocks, the tail of
    the block the chunk starts in, the whole blocks in between, the head of the block it ends in, EOF."""
    from . import bam_io
    with open(bam_filename, "rb") as src, open(new_filename, "wb") as out:
        out.write(src.read(parse_rec.header_size))
        if parse_rec.begin_read_offset > 0:
            data = bam_io.read_virtual(bam_filename, parse_rec.begin_read_offset, parse_rec.begin_read_size)
            for off in range(0, len(data), 60000):
                out.write(bam_io.bgzf_block(data[off:off + 60000]))
        src.seek(parse_rec.file_offset)
        out.write(src.read(parse_rec.file_bytes))
        if parse_rec.end_read_offset > 0:
            data = bam_io.read_virtual(bam_filename, parse_rec.end_read_offset, parse_rec.end_read_size)
            for off in range(0, len(data), 60000):
                out.write(bam_io.bgzf_block(data[off:off + 60000]))
        out.write(bam_io.BGZF_EOF)


def process_convert_bam(cp, device=0):
    """One worker of the reference (bam_utils.py:198-363): the chunks of cp.data, in order, through the GPU
    EC build; returns ConvertResults with `ec` = OrderedDict 'tid,tid,...' (tids as strings, sorted as
    strings, :306) -> number of reads, in first-occurrence order, exactly as the reference's worker.
    unique_reads (log-only in the reference, every read name of the chunk) is left empty.  As in the
    reference, a chunk without a valid alignment ends the worker with what it has (:336-349)."""
    from collections import OrderedDict
    ret = ConvertResults()
    ret.valid_alignments = 0
    ret.all_alignments = 0
    ret.ec = OrderedDict()
    ret.unique_reads = {}
    ret.tid_ranges = {}
    builder = tables = None
    pushed = 0
    try:
        for idx, parse_record in cp.data:
            temp_file = os.path.join(cp.temp_dir, "_bam2ec.{}.bam".format(idx))
            utils.delete_file(temp_file)
            chunk_bam_file(cp.input_file, temp_file, parse_record)
            try:
                with bamcols.BamColumnReader(temp_file) as reader:
                    if tables is None:
                        tables = reader.build_tables(None)
                    else:
                        reader.set_tables(tables)
                    if cp.track_ranges:
                        reader.track_ranges(True)
                    cols = reader.read_all(chunk=1 << 23)
                    ret.all_alignments += reader.all_alignments
                    if cp.track_ranges:
                        lo, hi = reader.ranges()
                        for tid in np.flatnonzero(lo <= hi).tolist():        # bam_utils.py:272-286: keys are str(tid)
                            n, x = ret.tid_ranges.get(str(tid), (int(lo[tid]), int(hi[tid])))
                            ret.tid_ranges[str(tid)] = (min(n, int(lo[tid])), max(x, int(hi[tid])))
            finally:
                utils.delete_file(temp_file)
            n = len(cols["read_group"])
            if n == 0:
                LOG.error("Error: sequence item 0: expected str instance, NoneType found")   # what :348 logs
                break
            if builder is None:
                builder = EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=False, alignments_hint=0,
                                    device=device, max_read=emitter.max_read())
            builder.push(cols["read_group"], cols["target_idx"], cols["hap_idx"], order_base=pushed)
            pushed += n
            ret.valid_alignments += n
        if builder is not None and pushed:
            res = builder.finalize()
            # EC row (main target, haplotype mask) -> the tids of the reference's key
            tid_of = np.full((tables.num_targets, max(1, tables.num_haplotypes)), -1, dtype=np.int64)
            tid_of[tables.tid_target, tables.tid_hap] = np.arange(len(tables.tid_target))
            indptr, indices, data, counts = res["a_indptr"], res["a_indices"], res["a_data"], res["n_data"]
            for e in range(int(res["n_ec"])):
                tids = []
                for j in range(int(indptr[e]), int(indptr[e + 1])):
                    mask = int(data[j])
                    for h in range(tables.num_haplotypes):
                        if (mask >> h) & 1:
                            tids.append(str(int(tid_of[indices[j], h])))
                ret.ec[",".join(sorted(tids))] = int(counts[e])
    finally:
        if builder is not None:
            builder.close()
    return ret


def wrapper_convert(args):
    """As the reference's (bam_utils.py:490-498): unpack the argument tuple Pool.imap delivers."""
    return process_convert_bam(*args)


def _job_plan(num_chunks, number_processes):
    """bam_utils.py:530-544."""
    num_processes = multiprocessing.cpu_count() if number_processes <= 0 else number_processes
    if num_chunks <= 0:
        num_chunks = num_processes
    elif num_chunks > 1000:
        LOG.info("Modifying number of chunks from {} to 1000".format(num_chunks))
        num_chunks = 1000
    return num_chunks, min(num_processes, num_chunks)


def _convert_python_emitter(bam_filename, target_filename, device, start_time, collate=False, max_read=16384):
    """The same build fed by the record-level Python emitter (ALNTOOLS_B200_EMITTER=python); collate: reads by name
    over the whole file (emitter.emit_collated); max_read: as emitter.max_read."""
    temp_time = time.time()
    header, records = emitter.read_bam(bam_filename)
    tables = TargetTables(header.references, header.lengths, target_filename)
    LOG.info("File parsed in {}, total time: {}".format(utils.format_time(temp_time, time.time()),
                                                        utils.format_time(start_time, time.time())))
    cols = emitter.emit_collated(records, tables) if collate else emitter.emit_single(records, tables)
    if cols.valid_alignments == 0:
        raise RuntimeError("The shape must be a tuple of three positive integers.")
    with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=False,
                   alignments_hint=cols.valid_alignments, device=device, max_read=max_read) as builder:
        builder.push(cols.read_group, cols.target_idx, cols.hap_idx, order_base=0)
        res = builder.finalize()
    return res, tables, cols.valid_alignments


def convert_rank(bam_filename, ec_filename, emase_filename, num_chunks=0, number_processes=-1, temp_dir=None,
                 range_filename=None, sample=None, target_filename=None):
    """One rank of the multi-GPU convert (one process per GPU; RANK / WORLD_SIZE / LOCAL_RANK / MASTER_* in
    the environment, as torchrun sets them).  What the reference does with a process pool over chunk BAMs
    merged in chunk order (alntools/bam_utils.py:642-724) happens here as: every rank plans the same shards of
    the ONE file (virtual offsets at read boundaries, no temporary BAMs: bamcols_plan_shards), decodes and
    groups its own on its GPU, is moved to its global position in read order (ecb_rebase: the position is
    known once every rank has counted its alignments), and the ranks merge through the exchange of
    multi_gpu.distributed_finalize.  The final matrices stay partitioned by EC-id range; every rank writes its
    byte ranges of the EC file (multi_gpu.save_rank_outputs).  Returns the totals on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from . import multi_gpu
    start_time = time.time()
    limit = emitter.max_read()
    with multi_gpu.rank_process() as (rank, world, device):
        _, num_processes = _job_plan(num_chunks, number_processes)
        num_processes = max(1, num_processes // world)          # the host threads are shared by the ranks
        if sample is None:
            sample = os.path.basename(bam_filename)
        with bamcols.BamColumnReader(bam_filename, n_threads=num_processes) as reader:
            tables = reader.build_tables(target_filename)
            plan = reader.plan_shards(world)
            reader.set_range(plan[rank], plan[rank + 1])
            if range_filename is not None:
                reader.track_ranges(True)
            opts = dict(with_cells=False, alignments_hint=0, device=device.index, result_on_device=1)
            with EcBuilder(tables.num_targets, tables.num_haplotypes, max_read=limit, **opts) as builder, \
                    EcBuilder(tables.num_targets, tables.num_haplotypes, **opts) as owner:
                chunk_rows = int(min(1 << 21, max(1 << 16, os.path.getsize(bam_filename) // 2)))   # 24 MB of columns per piece
                valid = emitter.stream_single(reader, builder, chunk_rows=chunk_rows, pinned=True)
                mine = torch.tensor([valid, reader.all_alignments], dtype=torch.int64, device=device)
                every = [torch.empty_like(mine) for _ in range(world)]
                dist.all_gather(every, mine)
                every = torch.stack(every).tolist()
                total_valid = sum(r[0] for r in every)
                if total_valid == 0:                              # as the single-GPU path (Sparse3DMatrix.py:45-46)
                    raise RuntimeError("The shape must be a tuple of three positive integers.")
                builder.rebase(sum(r[0] for r in every[:rank]))
                out = multi_gpu.distributed_finalize(builder, lambda: owner, device, result_on="slices")
                reads = out["n_data"][:int(out["n_ec_local"])].to(torch.int64).sum().reshape(1)
                dist.all_reduce(reads)
                track = range_filename is not None
                nnz_a = multi_gpu.save_rank_outputs(out, tables, tables.target_section(), [sample], ec_filename,
                                                    emase_filename, range_filename, reader.references if track else None,
                                                    reader.ranges() if track else None)
        if rank != 0:
            return None
        n_ec = int(out["n_ec"])
        LOG.info("# Valid Alignments: {:,}".format(total_valid))
        LOG.info("# Main Targets: {:,}".format(tables.num_targets))
        LOG.info("# Haplotypes: {:,}".format(tables.num_haplotypes))
        LOG.info("# Equivalence Classes: {:,}".format(n_ec))
        LOG.info("# Unique Reads: {:,}".format(int(reads.item())))
        LOG.info("{} GPUs, total time: {}".format(world, utils.format_time(start_time, time.time())))
        return {"n_ec": n_ec, "nnz_a": nnz_a, "n_samples": 1, "nnz_n": n_ec, "n_reads": int(reads.item()),
                "n_alignments": total_valid, "n_gpus": world,
                "alignments_per_gpu": [r[0] for r in every]}


def convert(bam_filename, ec_filename, emase_filename, num_chunks=0, number_processes=-1, temp_dir=None,
            range_filename=None, sample=None, target_filename=None, device=0, devices=None, decode=None, collate=None):
    """Convert a name-grouped BAM file into an EC binary file and/or an EMASE file.

    Arguments keep the reference's meaning.  num_chunks / number_processes only shape the host decode
    (the EC file does not depend on them, as in the reference); temp_dir is unused because no
    temporary BAM is written.  `device` selects the GPU.  devices=N (or the environment variable
    ALNTOOLS_GPUS=N) shards the file over N GPUs of this machine, one worker process per GPU (convert_rank);
    the same happens without either when the call is made inside a one-process-per-GPU job (torchrun).
    The EC file does not depend on the number of GPUs.  decode="device" (or ALNTOOLS_B200_DECODE=device) inflates
    and decodes the BAM file on the GPU (one GPU, native emitter); "host" (the default) decodes it on the CPU.
    The outputs do not depend on it.
    collate=True (or ALNTOOLS_B200_COLLATE=1) takes a file that is not grouped by read name: a read is every valid
    alignment with one trimmed name, wherever it lies, and reads are ordered by their first alignment (one GPU, host
    decode).  The outputs are those of the default convert() of the file regrouped that way; for a grouped file they
    are the default's.  ALNTOOLS_B200_COLLATE_BUDGET caps the device bytes of the collation (emitter.collate_budget);
    a file whose rows do not fit is collated in passes through host memory, with the same outputs.
    ALNTOOLS_B200_MAX_READ raises the longest read accepted from 16384 alignments (emitter.max_read; 0: the push limit),
    in every mode; longer reads take a sort-based pass on the GPU.  The default stays, because in a file grouped by
    name a read that long more often means a broken input.
    """
    start_time = time.time()
    mode = emitter.resolve_mode(False, devices, decode, collate, range_filename is not None)
    budget = emitter.collate_budget() if mode.collate else 0
    limit = emitter.max_read()
    job = dict(bam_filename=bam_filename, ec_filename=ec_filename, emase_filename=emase_filename, num_chunks=num_chunks,
               number_processes=number_processes, temp_dir=temp_dir, range_filename=range_filename, sample=sample,
               target_filename=target_filename)
    if mode.launcher:
        return convert_rank(**job)
    if mode.gpus > 1:
        return utils.spawn_ranks(mode.gpus, job)
    num_chunks, num_processes = _job_plan(num_chunks, number_processes)
    if sample is None:                                        # bam_utils.py:552-554
        sample = os.path.basename(bam_filename)
        LOG.info("Sample not supplied, using filename: {}".format(sample))

    def save(res, tables, valid, temp_time, references=None, ranges=None):
        """Log the totals and write the outputs from the result arrays (bam_utils.py:726-876)."""
        LOG.info("All results combined in {}, total time: {}".format(utils.format_time(temp_time, time.time()),
                                                                     utils.format_time(start_time, time.time())))
        LOG.info("# Valid Alignments: {:,}".format(valid))
        LOG.info("# Main Targets: {:,}".format(tables.num_targets))
        LOG.info("# Haplotypes: {:,}".format(tables.num_haplotypes))
        LOG.info("# Equivalence Classes: {:,}".format(res["n_ec"]))
        LOG.info("# Unique Reads: {:,}".format(res["n_reads"]))
        for name in (emase_filename, ec_filename):
            if name:
                LOG.info("Saving to {}...".format(name))
        temp_time = time.time()
        bin_utils.save_outputs(tables, tables.target_section(), [sample], (res["a_indptr"], res["a_indices"], res["a_data"]),
                               (res["n_indptr"], res["n_indices"], res["n_data"]), False, ec_filename, emase_filename,
                               range_filename, references, ranges)
        if ec_filename:
            LOG.info("{} created in {}, total time: {}".format(ec_filename,
                                                               utils.format_time(temp_time, time.time()),
                                                               utils.format_time(start_time, time.time())))
        return {k: v for k, v in res.items() if not hasattr(v, "shape")}   # the scalar totals

    LOG.info("Parsing file information ...")
    temp_time = time.time()
    if mode.python:
        res, tables, valid = _convert_python_emitter(bam_filename, target_filename, device, start_time, mode.collate,
                                                     limit)
        return save(res, tables, valid, temp_time)
    # native emitter: inflate threads + one record pass, streamed to the GPU in read-aligned chunks
    import torch
    with bamcols.BamColumnReader(bam_filename, n_threads=num_processes) as reader:
        tables = reader.build_tables(target_filename)       # native statement of header.TargetTables
        if range_filename is not None and mode.decode == "host":
            reader.track_ranges(True)
        LOG.info("File parsed in {}, total time: {}".format(utils.format_time(temp_time, time.time()),
                                                            utils.format_time(start_time, time.time())))
        temp_time = time.time()
        # no alignment count is known up front: the library sizes its table from the first chunk and
        # grows it ahead of later ones; one finalize per context, so results skip the pinning cost
        with EcBuilder(tables.num_targets, tables.num_haplotypes, with_cells=False, alignments_hint=0,
                       device=device, pageable_results=1, collate_budget=budget, max_read=limit) as builder:
            chunk_rows = int(min(1 << 21, max(1 << 16, os.path.getsize(bam_filename) // 2)))   # 24 MB of columns per piece
            if mode.decode == "device":
                valid, _, ranges, _ = emitter.stream_single_device(bam_filename, reader, builder, tables,
                                                                range_filename is not None)
            elif mode.collate:
                valid, _, _ = emitter.stream_collated(reader, builder, chunk_rows=chunk_rows, pinned=torch.cuda.is_available())
                ranges = reader.ranges() if range_filename is not None else None
            else:
                valid = emitter.stream_single(reader, builder, chunk_rows=chunk_rows, pinned=torch.cuda.is_available())
                ranges = reader.ranges() if range_filename is not None else None
            if valid == 0:
                # the reference ends up with zero ECs and APM() raises (Sparse3DMatrix.py:45-46)
                raise RuntimeError("The shape must be a tuple of three positive integers.")
            # the files are written straight from the library's result buffers (no intermediate copies)
            return save(builder.finalize(copy=False), tables, valid, temp_time,
                        reader.references if range_filename is not None else None, ranges)


def convert_samples(bam_files, ec_filename, sample_names=None, target_filename=None, range_filename=None, device=0,
                    decode=None, collate=None, devices=None):
    """Convert several BAM files, one per sample, into one EC file whose N matrix has one column per file.

    Every file is read with the rules of the single-sample convert() (filters, name trimming, a new read at each
    change of trimmed name; with collate=True each file is collated on its own), and a read never spans two files.
    The ECs, their ids and the A matrix are those of convert() over the files' valid alignments back to back, in the
    given order: an EC id is the rank of its first occurrence over the first file, then the second, and so on.  Entry
    (e, s) of N is the number of reads of file s in EC e; a file without a valid alignment is an empty column.  So
    files converted together share one EC index, which separately converted files do not.  With one file the EC
    file is the bytes convert() writes.

    sample_names: one name per file (default: each file's base name, as convert() names its sample).  Every file must
    have the @SQ list (names and lengths) of the first; the targets and target_filename apply as in convert().
    range_filename: the smallest and largest position per reference over all files.  decode / collate and the
    environment variables ALNTOOLS_B200_DECODE, ALNTOOLS_B200_COLLATE, ALNTOOLS_B200_COLLATE_BUDGET,
    ALNTOOLS_B200_MAX_READ and ALNTOOLS_B200_EMITTER=python work as for convert().  One GPU (`device`): more than one
    GPU (devices, ALNTOOLS_GPUS or a launcher) and an EMASE (.h5) output raise NotImplementedError, before any file
    is opened, as do no files or a number of names that differs from the number of files (ValueError)."""
    start_time = time.time()
    bam_files = list(bam_files)
    if not bam_files:
        raise ValueError("convert_samples needs at least one BAM file")
    if sample_names is None:
        sample_names = [os.path.basename(f) for f in bam_files]
    sample_names = list(sample_names)
    if len(sample_names) != len(bam_files):
        raise ValueError("%d sample names for %d BAM files" % (len(sample_names), len(bam_files)))
    if str(ec_filename).lower().endswith(".h5"):
        raise NotImplementedError("convert_samples writes EC files only; an EMASE (.h5) file of several samples is "
                                  "not supported")
    mode = emitter.resolve_mode(False, devices, decode, collate, range_filename is not None)
    if mode.launcher or mode.gpus > 1:
        raise NotImplementedError("convert_samples runs on one GPU (unset ALNTOOLS_GPUS, or run it outside a "
                                  "multi-GPU launcher)")
    budget = emitter.collate_budget() if mode.collate else 0
    limit = emitter.max_read()

    def header(path):
        if mode.python:
            h = bam_io.read_header(path)
            return h.references, h.lengths
        with bamcols.BamColumnReader(path, n_threads=1) as reader:
            return reader.references, reader.lengths

    first = header(bam_files[0])
    for path in bam_files[1:]:
        if header(path) != first:
            raise ValueError("%s does not have the @SQ list (names and lengths) of %s" % (path, bam_files[0]))

    track = range_filename is not None
    references = ranges = None
    valid = 0
    if mode.python:
        tables = TargetTables(first[0], first[1], target_filename)
        section = tables.target_section()
        builder = EcBuilder(tables.num_targets, tables.num_haplotypes, alignments_hint=0, device=device,
                            pageable_results=1, max_read=limit)
    else:
        with bamcols.BamColumnReader(bam_files[0], n_threads=1) as reader:
            tables = reader.build_tables(target_filename)
            section = tables.target_section()
            references = reader.references if track else None
        builder = EcBuilder(tables.num_targets, tables.num_haplotypes, alignments_hint=0, device=device,
                            pageable_results=1, collate_budget=budget, max_read=limit)
    with builder:
        for path in bam_files:
            if mode.python:
                _, records = emitter.read_bam(path)
                cols = emitter.emit_collated(records, tables) if mode.collate else emitter.emit_single(records, tables)
                if cols.valid_alignments:
                    builder.push(cols.read_group, cols.target_idx, cols.hap_idx, order_base=0)
                n, lo_hi = cols.valid_alignments, None
            else:
                n, lo_hi = _stream_sample(path, builder, tables, mode, track)
            builder.close_sample()                         # later pushes count their order keys from 0 again
            valid += n
            if lo_hi is not None:
                ranges = lo_hi if ranges is None else (np.minimum(ranges[0], lo_hi[0]), np.maximum(ranges[1], lo_hi[1]))
        if valid == 0:
            raise RuntimeError("The shape must be a tuple of three positive integers.")   # as convert()
        res = builder.finalize_samples(copy=False)
        LOG.info("# Samples: {:,}".format(len(bam_files)))
        LOG.info("# Valid Alignments: {:,}".format(valid))
        LOG.info("# Equivalence Classes: {:,}".format(res["n_ec"]))
        LOG.info("# Unique Reads: {:,}".format(res["n_reads"]))
        bin_utils.save_outputs(tables, section, sample_names, (res["a_indptr"], res["a_indices"], res["a_data"]),
                               (res["n_indptr"], res["n_indices"], res["n_data"]), False, ec_filename, None,
                               range_filename, references, ranges)
    LOG.info("{} created, total time: {}".format(ec_filename, utils.format_time(start_time, time.time())))
    return {k: v for k, v in res.items() if not hasattr(v, "shape")}


def _stream_sample(path, builder, tables, mode, track_ranges):
    """One file of convert_samples through the feed convert() uses for `mode`, with order keys from 0.
    -> (valid alignments, (range_min, range_max) or None)."""
    import torch
    pinned = torch.cuda.is_available()
    with bamcols.BamColumnReader(path, n_threads=0) as reader:
        reader.set_tables(tables)
        if track_ranges and mode.decode == "host":
            reader.track_ranges(True)
        chunk_rows = int(min(1 << 21, max(1 << 16, os.path.getsize(path) // 2)))
        if mode.decode == "device":
            valid, _, ranges, _ = emitter.stream_single_device(path, reader, builder, tables, track_ranges)
            return valid, ranges
        if mode.collate:
            valid, _, _ = emitter.stream_collated(reader, builder, chunk_rows=chunk_rows, pinned=pinned)
        else:
            valid = emitter.stream_single(reader, builder, chunk_rows=chunk_rows, pinned=pinned)
        return valid, reader.ranges() if track_ranges else None
