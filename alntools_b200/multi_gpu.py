"""Multi-GPU EC build: one process per GPU, shards of contiguous reads, one exchange step.

The reference's only parallelism is a process pool over contiguous BAM chunks whose results are
merged in chunk order (alntools/bam_utils.py:647-724).  Here every rank builds a local EC table from
its shard (order_base = global offset of the shard) and the merge becomes:

  dispatch 1   local ECs {key, first, count} stored straight into the arena of their OWNER rank
               (hash of the key) over peer memory by one kernel                          [NVLink]
  owner merge  equal keys: counts summed, smallest first-occurrence kept                [kernel]
  dispatch 2   every merged EC {key, position, count} to the rank whose SHARD holds its first
               occurrence; there a bitmap over the rank's own positions orders them (ids are ranks of
               first occurrences and the shards partition the positions) and the rows come from the
               rank's LOCAL context - it has met the EC in its own reads.  Rows never travel; every
               rank ends up with one contiguous id range of the final matrices          [NVLink]
  The barriers between these steps are tiny collectives on the stream the kernels run on: nothing in
  between waits for the host.

The per-cell path (distributed_finalize_cells) runs the same two dispatches with (EC, cell) pairs beside the ECs,
after every rank has taken the same cell decision from the all-gathered cell summaries; see the per-cell section
of include/ecb200.h.

torch.distributed is the plumbing (process group, collectives on device tensors); every compute
step is a libecb200 kernel behind the C ABI.
"""
import contextlib
import os
import time

import numpy as np
import torch
import torch.distributed as dist

from . import bin_utils, utils

_TIMING = bool(os.environ.get("ECB_MGPU_TIMING"))
LAST_PHASES = {}   # with ECB_MGPU_TIMING: the (phase, ms) rows of the last call of each exchange, for tools


class _Phases(object):
    """Per-phase wall clock of an exchange (ECB_MGPU_TIMING=1; synchronises after every phase).  rows keeps
    (phase, ms) for callers that report them themselves."""

    def __init__(self, device, name="distributed_finalize"):
        self.device, self.name, self.t, self.rows = device, name, time.perf_counter(), []

    def mark(self, name):
        if _TIMING:
            torch.cuda.synchronize(self.device)
            now = time.perf_counter()
            self.rows.append((name, 1e3 * (now - self.t)))
            self.t = now

    def report(self):
        if _TIMING:
            LAST_PHASES[self.name] = list(self.rows)
        if _TIMING and dist.get_rank() == 0:
            print(self.name + ": " + ", ".join("%s %.2f ms" % r for r in self.rows), flush=True)


_BARRIER_WORD = {}


def _stream_barrier(device, group):
    """A barrier among the ranks that lives on the CUDA stream: a one-word all-reduce.  Work a rank put on the
    stream before it is complete (and its peer-memory stores visible) before any rank's work behind it starts;
    the host does not wait."""
    key = (device, id(group))
    if key not in _BARRIER_WORD:
        _BARRIER_WORD[key] = torch.zeros(1, dtype=torch.int32, device=device)
    dist.all_reduce(_BARRIER_WORD[key], group=group)


class _Failure(object):
    """A rank that fails inside the exchange must not leave its peers waiting in a collective: it carries on with
    what it has, the failure travels with the final all-gather (_gather_rows) and every rank raises."""

    def __init__(self):
        self.exc = None

    def attempt(self, fn):
        try:
            return fn()
        except Exception as exc:     # noqa: BLE001 - re-raised on every rank by _gather_rows
            self.exc = self.exc or exc
            return None


def _gather_rows(values, failure, device, group):
    """All-gather one int64 row per rank (`values` plus this rank's failure flag) and raise on every rank when any
    rank failed.  -> [world] lists of the values."""
    world = dist.get_world_size(group)
    row = torch.cat([torch.as_tensor(values, dtype=torch.int64).to(device).reshape(-1),
                     torch.tensor([1 if failure.exc else 0], dtype=torch.int64, device=device)])
    out = torch.empty(world * row.numel(), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(out, row, group=group)
    rows = out.view(world, -1).tolist()
    if failure.exc is not None:
        raise failure.exc
    if any(r[-1] for r in rows):
        raise RuntimeError("the multi-GPU exchange failed on rank(s) %s" % [r for r in range(world) if rows[r][-1]])
    return [r[:-1] for r in rows]


def _open_arenas(owner, handle, base, device, group):
    """Every rank's arena base as seen from this process: the IPC handles are all-gathered and the peers' mapped."""
    world, me = dist.get_world_size(group), dist.get_rank(group)
    hs = [torch.empty(64, dtype=torch.uint8, device=device) for _ in range(world)]
    dist.all_gather(hs, torch.frombuffer(bytearray(handle), dtype=torch.uint8).to(device), group=group)
    return [base if r == me else owner.arena_open_peer(bytes(hs[r].cpu().tolist())) for r in range(world)]


def distributed_finalize(local, make_owner, device, group=None, result_on="slices"):
    """local: builder holding this rank's shard; make_owner(): builder for the owner role (the same one on every
    step of a job keeps its arena).  The final matrices stay partitioned by EC-id range: rank j holds ids
    [id_base, id_base + n_ec_local).  Returns dict(a_indptr, a_indices, a_data, n_data) of int32 tensors on
    `device` for that slice, with a_indptr local to it, and n_ec (all ranks), id_base, n_ec_local, nnz_local;
    nnz_a is None.  Nothing is padded to the global size on any rank.  result_on="slices" is the only layout."""
    if result_on != "slices":
        raise ValueError('result_on must be "slices", got %r' % (result_on,))
    if device.type != "cuda":
        raise ValueError("device must be a CUDA device (the exchange maps the ranks' GPU memory), got %s" % device)
    world = dist.get_world_size(group)
    # library kernels and torch's collectives must be ordered against each other: both builders work
    # on torch's current stream from here on (NCCL orders itself against that stream)
    cur = torch.cuda.current_stream(device).cuda_stream
    local.set_stream(cur)
    ph = _Phases(device)
    me = dist.get_rank(group)
    # ---- fused partition + dispatch: every local EC is stored straight into its owner's arena
    # over NVLink by ONE kernel (peer memory mapped through CUDA IPC); no staging
    owner = make_owner()
    owner.set_stream(cur)
    arena = getattr(owner, "_exchange_arena", None)
    if arena is not None:
        # the arenas exist (a later step of the same job): clear the header and put ONE small collective on
        # the stream as the barrier between "every arena is clear" and "peers store" - no host round trip;
        # whether everything fits is decided by the overflow flag in the arena header
        owner.arena_reset()
        _stream_barrier(device, group)
    else:
        # first call of a job: size the arenas (an owner receives about one rank's worth of ECs; twice the
        # largest local table leaves room for a skewed partition), create them, map the peers'
        info = torch.tensor([local.stats()["table_used"]], dtype=torch.int64, device=device)
        gathered = [torch.empty_like(info) for _ in range(world)]
        dist.all_gather(gathered, info, group=group)
        need_ec = 2 * max(int(t.item()) for t in gathered) + 1024
        handle, base = owner.arena_create(need_ec)
        bases = _open_arenas(owner, handle, base, device, group)
        arena = {"bases": bases, "cap_ec": need_ec}
        owner._exchange_arena = arena
        dist.barrier(group=group)                     # every arena exists and is zeroed
    ph.mark("setup")
    min_base, max_end = local.export_to_arenas(arena["bases"], arena["cap_ec"])
    ph.mark("dispatch 1")
    # every rank's shard of the read order; the all-gather is the barrier between "store" and "merge"
    mine = torch.tensor([min_base, max_end], dtype=torch.int64, device=device)
    spans = torch.empty(2 * world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(spans, mine, group=group)
    # a rank that fails from here on (an arena that turned out too small) carries on; see _Failure
    failure = _Failure()
    failure.attempt(owner.import_arena)
    owner.arena_reset()              # reused by the second dispatch ...
    _stream_barrier(device, group)   # ... once every rank has merged what it received
    ph.mark("merge")
    spans = spans.tolist()
    lo, hi = spans[0::2], spans[1::2]
    if not any(h > l for l, h in zip(lo, hi)):
        raise RuntimeError("The shape must be a tuple of three positive integers.")  # zero ECs everywhere
    owner.order_dispatch(arena["bases"], arena["cap_ec"], lo, hi)
    _stream_barrier(device, group)   # every rank's ECs have landed
    ph.mark("dispatch 2")
    sl = failure.attempt(lambda: owner.order_build(local, lo[me], hi[me]))
    ph.mark("order build")
    # the id range of a rank starts behind the ECs of the shards in front of it
    sizes = [r[0] for r in _gather_rows([sl["n_ec"] if sl else 0], failure, device, group)]
    id_base = sum(n for r, n in enumerate(sizes) if _in_front(lo, hi, r, me))
    ph.report()
    return {"a_indptr": sl["a_indptr"], "a_indices": sl["a_indices"], "a_data": sl["a_data"],
            "n_data": sl["n_data"], "n_ec": sum(sizes), "id_base": id_base, "n_ec_local": sl["n_ec"],
            "nnz_local": sl["nnz"], "nnz_a": None}


def _in_front(lo, hi, r, me):
    """Whether rank r's slice precedes rank me's in EC-id order: ids are ranks of first occurrences, so slices
    follow the order of the ranks' shards of the read order (ranks without alignments hold nothing)."""
    return hi[r] > lo[r] and (lo[r], r) < (lo[me], me)


def _cells_arena(owner, counts, device, group):
    """The per-cell arenas for the next dispatch, sized from its exact per-destination record counts (all-reduced:
    every rank takes the same decision).  Arenas that are large enough are cleared behind a stream barrier;
    otherwise every rank re-creates its own and the new IPC handles are exchanged before anyone stores."""
    world = dist.get_world_size(group)
    c = counts.tolist()
    need_ec, need_pairs = max(c[:world]), max(c[world:])
    arena = getattr(owner, "_cells_arena", None)
    if arena is not None and need_ec <= arena["cap_ec"] and need_pairs <= arena["cap_pairs"]:
        owner.arena_reset()
        _stream_barrier(device, group)
        return arena
    # a little headroom, so that the steps of a job with similar inputs keep their arenas
    cap_ec = max(need_ec + need_ec // 8, 1024, arena["cap_ec"] if arena else 0)
    cap_pairs = max(need_pairs + need_pairs // 8, 1024, arena["cap_pairs"] if arena else 0)
    dist.barrier(group=group)          # no rank still works on the arenas about to be replaced
    handle, base = owner.cells_arena_create(cap_ec, cap_pairs)
    arena = {"bases": _open_arenas(owner, handle, base, device, group), "cap_ec": cap_ec, "cap_pairs": cap_pairs,
             "created": (arena or {}).get("created", 0) + 1}
    owner._cells_arena = arena
    dist.barrier(group=group)          # every arena exists and its headers are zeroed
    return arena


def distributed_finalize_cells(local, make_owner, device, min_count, cell_map, n_cells, group=None):
    """The per-cell (multisample) exchange.  local: builder (with cells) holding this rank's files, pushed at
    rank-major order keys (order_base = rank * 2^40 + alignments of this rank's earlier files; see the per-cell
    section of include/ecb200.h); make_owner(): builder for the owner role, kept from step to step of a job with
    its arena.  cell_map: int32 device tensor, this rank's cell ids -> global ids (first appearance over the
    ranks' name lists in rank order), or None for identity; n_cells: number of global cell ids.

    The final matrices stay partitioned by EC-id range, as with distributed_finalize.  Returns, for this rank,
    int32 device tensors a_indptr (local to the slice), a_indices, a_data, the N pieces n_col_counts [S] (entries
    of every column held here), n_indices (EC ids local to the slice, ascending inside a column), n_data, and
    n_col_offset [S] (entries of each column held by the slices in front), n_indptr [S + 1] (global), cell_order
    [S] (global cell id of every column); scalars n_ec (all ranks), id_base, n_ec_local, nnz_local, nnz_a, nnz_n,
    n_samples.  Every rank gets the same cell_order, n_indptr and sizes."""
    if device.type != "cuda":
        raise ValueError("device must be a CUDA device (the exchange maps the ranks' GPU memory), got %s" % device)
    world, me = dist.get_world_size(group), dist.get_rank(group)
    cur = torch.cuda.current_stream(device).cuda_stream
    local.set_stream(cur)
    owner = make_owner()
    owner.set_stream(cur)
    ph = _Phases(device, "distributed_finalize_cells")
    # a rank that fails carries on with empty results (see _Failure): a failure before dispatch 1 travels with the
    # all-reduce of its counts and every rank raises there; one after it travels with the final all-gather
    failure = _Failure()
    # ---- cell summary by global id; keys all-gathered, totals summed
    summary = failure.attempt(lambda: local.cells_summary(cell_map, n_cells))
    if summary is None:
        summary = (torch.full((int(n_cells),), -1, dtype=torch.int64, device=device),
                   torch.zeros(int(n_cells), dtype=torch.int64, device=device))
    keys, totals = summary
    keys_all = torch.empty(world * int(n_cells), dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(keys_all, keys, group=group)
    dist.all_reduce(totals, group=group)
    ph.mark("cell summary")
    # ---- the same cell decision on every rank (no kept cell: every rank raises the same ECB_ERR_EMPTY)
    decided = None if failure.exc else failure.attempt(lambda: local.cells_order(keys_all, totals, min_count, cell_map, world))
    ph.mark("cell order")
    # ---- dispatch 1: ECs and kept pairs to the owner of the EC's key; the last word counts failed ranks
    counts = None if failure.exc else failure.attempt(lambda: local.cells_dispatch_counts(world))
    if counts is None:
        counts = torch.zeros(2 * world, dtype=torch.int64, device=device)
    counts = torch.cat([counts, torch.tensor([1 if failure.exc else 0], dtype=torch.int64, device=device)])
    dist.all_reduce(counts, group=group)
    if int(counts[-1]):
        _gather_rows([0], failure, device, group)   # raises on every rank
    n_samples, cell_order = decided
    arena = _cells_arena(owner, counts[:-1], device, group)
    ph.mark("setup 1")
    span = failure.attempt(lambda: local.cells_export_to_arenas(arena["bases"], arena["cap_ec"], arena["cap_pairs"]))
    min_base, max_end = span if span is not None else (0, 0)
    spans = torch.empty(2 * world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(spans, torch.tensor([min_base, max_end], dtype=torch.int64, device=device), group=group)
    ph.mark("dispatch 1")
    spans = spans.tolist()
    lo, hi = spans[0::2], spans[1::2]
    failure.attempt(owner.cells_import_arena)
    ph.mark("merge")
    # ---- dispatch 2: merged ECs with kept reads, and merged pairs, to the rank that holds the first occurrence
    counts = failure.attempt(lambda: owner.cells_dispatch_counts(world, lo, hi))
    if counts is None:
        counts = torch.zeros(2 * world, dtype=torch.int64, device=device)
    dist.all_reduce(counts, group=group)
    arena = _cells_arena(owner, counts, device, group)
    ph.mark("setup 2")
    failure.attempt(lambda: owner.cells_order_dispatch(arena["bases"], arena["cap_ec"], arena["cap_pairs"], lo, hi))
    _stream_barrier(device, group)   # every rank's records have landed
    ph.mark("dispatch 2")
    sl = failure.attempt(lambda: owner.cells_order_build(local, lo[me], hi[me], n_samples))
    ph.mark("order build")
    col = sl["n_col_counts"].to(torch.int64) if sl else torch.zeros(n_samples, dtype=torch.int64, device=device)
    rows = _gather_rows(torch.cat([torch.tensor([sl["n_ec"] if sl else 0, sl["nnz"] if sl else 0], dtype=torch.int64,
                                                device=device), col]), failure, device, group)
    front = [r for r in range(world) if _in_front(lo, hi, r, me)]
    col_all = torch.tensor([r[2:] for r in rows], dtype=torch.int64)
    n_indptr = torch.zeros(n_samples + 1, dtype=torch.int64)
    torch.cumsum(col_all.sum(0), 0, out=n_indptr[1:])
    if int(n_indptr[-1]) > 0x7FFFFFFF:
        raise RuntimeError("the N matrix has more than 2^31-1 entries")
    col_offset = col_all[front].sum(0) if front else torch.zeros(n_samples, dtype=torch.int64)
    ph.report()
    return {"a_indptr": sl["a_indptr"], "a_indices": sl["a_indices"], "a_data": sl["a_data"],
            "n_col_counts": sl["n_col_counts"], "n_indices": sl["n_indices"], "n_data": sl["n_data"],
            "n_col_offset": col_offset.to(torch.int32).to(device), "n_indptr": n_indptr.to(torch.int32).to(device),
            "cell_order": cell_order, "n_ec": sum(r[0] for r in rows), "id_base": sum(rows[r][0] for r in front),
            "n_ec_local": sl["n_ec"], "nnz_local": sl["nnz"], "nnz_a": sum(r[1] for r in rows),
            "nnz_n": int(n_indptr[-1]), "n_samples": n_samples}


@contextlib.contextmanager
def rank_process():
    """This process as one rank of a one-process-per-GPU job (RANK / WORLD_SIZE / LOCAL_RANK / MASTER_* in the
    environment, as torchrun sets them): bound to the CPUs next to its GPU, so that the host buffers it pins land in
    that GPU's NUMA node, with that GPU current, and in a NCCL process group, which is created here unless one
    exists and then destroyed on the way out.  Yields (rank, world size, device)."""
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    utils.bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    own_group = not dist.is_initialized()
    if own_group:
        dist.init_process_group("nccl", device_id=device)
    try:
        yield rank, world, device
    finally:
        if own_group and dist.is_initialized():
            dist.destroy_process_group()


def save_rank_outputs(out, tables, section, sample_names, ec_filename, emase_filename, range_filename=None,
                      references=None, ranges=None):
    """Write the outputs of a multi-GPU convert; every rank calls it with its slice `out` of the final matrices, as
    distributed_finalize or, for the per-cell converter, distributed_finalize_cells returned it.  First, on every
    rank and before any file is touched, the global sizes are checked against the EC file's int32 fields.  The ranks
    write their byte ranges of the EC file once rank 0 has laid it out; rank 0 assembles the EMASE file from every
    rank's slice, and writes the range file from the ranges (range_min, range_max) of every rank's input (None for a
    rank without input) over the header's reference names `references`.  section, sample_names: as
    bin_utils.save_outputs.  -> non-zeros of A over all ranks."""
    rank, world = dist.get_rank(), dist.get_world_size()
    device = out["a_indptr"].device
    cells = "n_indptr" in out                             # distributed_finalize_cells' result
    n_ec, id_base, n_local, nnz_local = (int(out[k]) for k in ("n_ec", "id_base", "n_ec_local", "nnz_local"))
    rows = torch.empty(3 * world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(rows, torch.tensor([id_base, n_local, nnz_local], dtype=torch.int64, device=device))
    rows = rows.view(world, 3).tolist()
    nnz_a = sum(r[2] for r in rows)
    nnz_base = sum(r[2] for r in rows if r[1] and r[0] < id_base)   # the slices in front of this one in id order
    nnz_n = int(out["nnz_n"]) if cells else n_ec
    if n_ec + 1 > 0x7FFFFFFF or nnz_a > 0x7FFFFFFF or nnz_n > 0x7FFFFFFF:
        raise RuntimeError("the EC file's int32 fields cannot hold %d ECs, %d A and %d N non-zeros" % (n_ec, nnz_a, nnz_n))
    host = lambda t: t.cpu().numpy()
    a = (host(out["a_indptr"][:n_local + 1]), host(out["a_indices"][:nnz_local]), host(out["a_data"][:nnz_local]))
    if cells:
        n = tuple(host(out[k]) for k in ("n_indptr", "n_col_counts", "n_col_offset", "n_indices", "n_data"))
    else:
        n = (host(out["n_data"][:n_local]),)
    if ec_filename:
        header = bin_utils.ec_header_bytes(tables.haplotypes, list(tables.main_targets.keys()) if section is None else None,
                                           tables.lengths, sample_names, target_section=section,
                                           n_targets=tables.num_targets)
        write = bin_utils.ecsave2_cells_slice if cells else bin_utils.ecsave2_slice
        args = (ec_filename, header, n_ec, nnz_a, id_base, nnz_base) + a + n
        if rank == 0:
            utils.delete_file(ec_filename)
            write(*args, create=True)
        dist.barrier()                                    # the file is laid out
        if rank != 0:
            write(*args, create=False)
        dist.barrier()
    a_csr = n_csc = None
    if emase_filename:                                    # one writer: the slices travel to rank 0
        parts = [None] * world
        dist.all_gather_object(parts, (id_base, a, n))
        if rank == 0:
            a_csr, n_csc = _assemble(parts, n_ec, cells)
    if range_filename is not None:                        # over every rank's input
        if ranges is None:                                # neutral elements
            ranges = (np.full(len(references), np.iinfo(np.int64).max), np.full(len(references), np.iinfo(np.int64).min))
        lo, hi = (torch.from_numpy(np.asarray(x, dtype=np.int64)).to(device) for x in ranges)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        ranges = (lo.cpu().numpy(), hi.cpu().numpy())
    if rank == 0:
        bin_utils.save_outputs(tables, section, sample_names, a_csr, n_csc, cells, emase_filename=emase_filename,
                               range_filename=range_filename, references=references, ranges=ranges)
    return nnz_a


def _assemble(parts, n_ec, cells):
    """The whole matrices from every rank's (id_base, A pieces, N pieces), in id order (for the EMASE file)."""
    parts = sorted((p for p in parts if len(p[1][0]) > 1), key=lambda p: p[0])
    indptr, at = [np.zeros(1, dtype=np.int64)], 0
    for _, (ip, ix, _d), _n in parts:
        indptr.append(ip[1:].astype(np.int64) + at)
        at += len(ix)
    a_csr = (np.concatenate(indptr).astype(np.int32), np.concatenate([p[1][1] for p in parts]).astype(np.int32),
             np.concatenate([p[1][2] for p in parts]).astype(np.int32))
    if not cells:                                         # one sample: N holds every EC's count
        return a_csr, (np.array([0, n_ec], dtype=np.int32), np.arange(n_ec, dtype=np.int32),
                       np.concatenate([p[2][0] for p in parts]))
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


def shard_bounds(read_group, world):
    """Split an alignment stream into `world` contiguous, read-aligned shards (the reference's
    utils.partition gives each worker a contiguous run of chunks; chunk starts are moved to the next
    read boundary, bam_utils.py:1236-1247).  Returns world+1 offsets."""
    n = len(read_group)
    cuts = [0]
    for k in range(1, world):
        c = max(cuts[-1], n * k // world)
        while 0 < c < n and read_group[c] == read_group[c - 1]:
            c += 1
        cuts.append(c)
    cuts.append(n)
    return cuts
