// ecb_collate.cuh — collation of alignments by read name (ecb_collate_* in include/ecb200.h).
//
// The reference forms reads from runs of equal trimmed names (alntools/bam_utils.py:301-306), so it needs a
// file grouped by name.  Collation forms them over the whole file instead: a read is every valid alignment with
// one name, and reads are ordered by their first alignment.  Positions are file-order indices of the valid
// alignments.  The kernels, in launch order:
//   insert   every alignment finds or claims its name key's slot of an open-addressing table (EcbEntry: first =
//            smallest position, countm1 = alignments - 1) and stores the slot; equal keys of one warp are merged
//            first (match_any), so a grouped file costs one table operation per read and warp
//   mark     one bit per read at its first position, in a bitmap over [0, n)
//   ids      (after the word-rank scan of the bitmap, as ecb_fin_mark/rank do for EC ids) read id = rank of the
//            first position, kept in the slot's aux; alignments per read into a column in read-id order
//   scatter  (after an exclusive scan of that column: read offsets) every alignment goes to offset + a per-read
//            cursor; the cursors end at the read ends
//   cuts     one thread cuts the regrouped columns into pushes of at most `piece` alignments at read ends (a read
//            longer than a piece is a piece of its own)
#pragma once
#include "ecb_common.cuh"

struct CollateParams {
  const u64* key_lo;
  const u64* key_hi;
  u64 n;
  EcbEntry* table;
  u32 mask;
  u32* slot_of;       // [n]
  EcbCounters* ctr;   // scratch[0]: reads claimed, scratch[1]: alignments that found no slot
};

__global__ void __launch_bounds__(256) ecb_collate_insert_kernel(const CollateParams P) {
  const int lane = threadIdx.x & 31;
  const u64 n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 w0 = (((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5) << 5; w0 < P.n; w0 += n_warps << 5) {
    const u64 i = w0 + (u64)lane;
    if (i >= P.n) continue;
    const u32 act = __activemask();
    const Key128 key{P.key_lo[i], P.key_hi[i]};
    const u32 same = __match_any_sync(act, key.lo) & __match_any_sync(act, key.hi);
    const int leader = __ffs(same) - 1;   // the lowest lane holds the smallest position of the key in this warp
    u32 slot = 0;
    if (lane == leader) {
      bool claimed;
      u64 first_seen;
      slot = table_find_or_claim<false>(P.table, P.mask, key, claimed, first_seen);
      if (slot != ECB_NONE) {
        EcbEntry* e = P.table + slot;
        atomicAdd(&e->countm1, (u32)__popc(same));
        if (i < first_seen) atomicMin(&e->first, (unsigned long long)i);
        if (claimed) atomicAdd(&P.ctr->scratch[0], 1u);
      } else {
        atomicAdd(&P.ctr->scratch[1], (u32)__popc(same));
      }
    }
    slot = __shfl_sync(act, slot, leader);
    P.slot_of[i] = slot;
  }
}

__global__ void __launch_bounds__(256) ecb_collate_mark_kernel(const EcbEntry* __restrict__ table, u32 slots,
                                                               u32* __restrict__ bitmap) {
  for (u32 s = blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += gridDim.x * blockDim.x) {
    const u64 first = table[s].first;
    if (first != ~0ull) atomicOr(&bitmap[first >> 5], 1u << (first & 31));
  }
}

__global__ void __launch_bounds__(256) ecb_collate_ids_kernel(EcbEntry* __restrict__ table, u32 slots,
                                                              const u32* __restrict__ bitmap,
                                                              const u32* __restrict__ word_rank, u32* __restrict__ count) {
  for (u32 s = blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += gridDim.x * blockDim.x) {
    EcbEntry* e = table + s;
    const u64 first = e->first;
    if (first == ~0ull) continue;
    const u32 w = (u32)(first >> 5), b = (u32)(first & 31);
    const u32 id = word_rank[w] + (u32)__popc(bitmap[w] & ((1u << b) - 1u));
    e->aux = id;
    count[id] = e->countm1 + 1u;
  }
}

// cursor[id] holds the read's offset on entry and its end on exit.  Alignments of one read inside a warp take
// consecutive places in position order with one atomic.
__global__ void __launch_bounds__(256) ecb_collate_scatter_kernel(const u32* __restrict__ slot_of,
                                                                  const EcbEntry* __restrict__ table,
                                                                  const int32_t* __restrict__ tg_in,
                                                                  const int32_t* __restrict__ hp_in, u64 n,
                                                                  u32* __restrict__ cursor, int32_t* __restrict__ rg,
                                                                  int32_t* __restrict__ tg, int32_t* __restrict__ hp) {
  const int lane = threadIdx.x & 31;
  const u64 n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 w0 = (((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5) << 5; w0 < n; w0 += n_warps << 5) {
    const u64 i = w0 + (u64)lane;
    if (i >= n) continue;
    const u32 act = __activemask();
    const u32 slot = slot_of[i];
    const u32 same = __match_any_sync(act, slot);
    const int leader = __ffs(same) - 1;
    const u32 id = table[slot].aux;
    u32 base = 0;
    if (lane == leader) base = atomicAdd(&cursor[id], (u32)__popc(same));
    base = __shfl_sync(act, base, leader);
    const u32 p = base + (u32)__popc(same & ((1u << lane) - 1u));
    rg[p] = (int32_t)id;   // ecb_push only needs read_group to change between reads
    tg[p] = tg_in[i];
    hp[p] = hp_in[i];
  }
}

// cuts[0] = number of pieces k, cuts[1 .. k+1] = piece boundaries (0, ..., n).  ends[0 .. n_reads) are the read
// ends, ascending.  A piece takes whole reads while they fit in `piece` alignments; one thread, one binary search
// per piece.
__global__ void ecb_collate_cuts_kernel(const u32* __restrict__ ends, u32 n_reads, u64 n, u64 piece, u32* __restrict__ cuts) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  u32 k = 0;
  u64 b = 0;
  cuts[1] = 0;
  while (b < n) {
    u64 cut = n;
    if (b + piece < n) {
      // last read end at or before b + piece
      u32 lo = 0, hi = n_reads;
      while (lo < hi) {
        const u32 mid = lo + (hi - lo) / 2;
        if ((u64)ends[mid] <= b + piece) lo = mid + 1; else hi = mid;
      }
      if (lo > 0 && (u64)ends[lo - 1] > b) {
        cut = ends[lo - 1];
      } else {
        // the read that starts at b is longer than a piece: it is a piece of its own
        lo = 0, hi = n_reads;
        while (lo < hi) {
          const u32 mid = lo + (hi - lo) / 2;
          if ((u64)ends[mid] <= b) lo = mid + 1; else hi = mid;
        }
        cut = ends[lo];
      }
    }
    cuts[2 + k] = (u32)cut;
    ++k;
    b = cut;
  }
  cuts[0] = k;
}
