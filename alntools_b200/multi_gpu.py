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

torch.distributed is the plumbing (process group, collectives on device tensors); every compute
step is a libecb200 kernel behind the C ABI.
"""
import os
import time

import torch
import torch.distributed as dist

_TIMING = bool(os.environ.get("ECB_MGPU_TIMING"))


class _Phases(object):
    """Per-phase wall clock of distributed_finalize (ECB_MGPU_TIMING=1; synchronises after every phase)."""

    def __init__(self, device):
        self.device, self.t, self.rows = device, time.perf_counter(), []

    def mark(self, name):
        if _TIMING:
            torch.cuda.synchronize(self.device)
            now = time.perf_counter()
            self.rows.append((name, 1e3 * (now - self.t)))
            self.t = now

    def report(self):
        if _TIMING and dist.get_rank() == 0:
            print("distributed_finalize: " + ", ".join("%s %.2f ms" % r for r in self.rows), flush=True)


_BARRIER_WORD = {}


def _stream_barrier(device, group):
    """A barrier among the ranks that lives on the CUDA stream: a one-word all-reduce.  Work a rank put on the
    stream before it is complete (and its peer-memory stores visible) before any rank's work behind it starts;
    the host does not wait."""
    key = (device, id(group))
    if key not in _BARRIER_WORD:
        _BARRIER_WORD[key] = torch.zeros(1, dtype=torch.int32, device=device)
    dist.all_reduce(_BARRIER_WORD[key], group=group)


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
        hs = [torch.empty(64, dtype=torch.uint8, device=device) for _ in range(world)]
        dist.all_gather(hs, torch.frombuffer(bytearray(handle), dtype=torch.uint8).to(device), group=group)
        bases = [base if r == me else owner.arena_open_peer(bytes(hs[r].cpu().tolist())) for r in range(world)]
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
    # a rank that fails from here on (an arena that turned out too small) must not leave its peers waiting in
    # a collective: it carries on with what it has, the failure travels with the all-gather of the slice
    # sizes below, and every rank raises
    failure = None
    try:
        owner.import_arena()
    except Exception as exc:         # noqa: BLE001 - re-raised on every rank below
        failure = exc
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
    sl = None
    try:
        sl = owner.order_build(local, lo[me], hi[me])
    except Exception as exc:         # noqa: BLE001
        failure = failure or exc
    ph.mark("order build")
    # the id range of a rank starts behind the ECs of the shards in front of it
    sizes = torch.empty(2 * world, dtype=torch.int64, device=device)
    dist.all_gather_into_tensor(sizes, torch.tensor([sl["n_ec"] if sl else 0, 1 if failure else 0],
                                                    dtype=torch.int64, device=device), group=group)
    sizes = sizes.tolist()
    if failure is not None:
        raise failure
    if any(sizes[1::2]):
        raise RuntimeError("the multi-GPU exchange failed on rank(s) %s" % [r for r in range(world) if sizes[2 * r + 1]])
    sizes = sizes[0::2]
    id_base = sum(n for r, n in enumerate(sizes) if hi[r] > lo[r] and (lo[r], r) < (lo[me], me))
    ph.report()
    return {"a_indptr": sl["a_indptr"], "a_indices": sl["a_indices"], "a_data": sl["a_data"],
            "n_data": sl["n_data"], "n_ec": sum(sizes), "id_base": id_base, "n_ec_local": sl["n_ec"],
            "nnz_local": sl["nnz"], "nnz_a": None}


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
