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
// A collator over its memory budget spills (DESIGN.md section 6.2): the same kernels run per group of name buckets,
// with positions taken from a column, plus the stable partition, the read list, the per-row first position, the
// ids from the read list, the placement of rows in collated order and the scatter of one piece.
#pragma once
#include "ecb_common.cuh"

struct CollateParams {
  const u64* key_lo;
  const u64* key_hi;
  const u32* pos;     // file-order position of every row; NULL: the row index
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
    // the lowest lane holds the smallest position of the key in this warp: rows of one key come in file order
    const int leader = __ffs(same) - 1;
    u32 slot = 0;
    if (lane == leader) {
      bool claimed;
      u64 first_seen;
      const u64 p = P.pos ? (u64)P.pos[i] : i;
      slot = table_find_or_claim<false>(P.table, P.mask, key, claimed, first_seen);
      if (slot != ECB_NONE) {
        EcbEntry* e = P.table + slot;
        atomicAdd(&e->countm1, (u32)__popc(same));
        if (p < first_seen) atomicMin(&e->first, (unsigned long long)p);
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

// ---- spilled collation ------------------------------------------------------------------------------------------
#define COLLATE_TILE 4096         // rows per CTA of the partition
#define COLLATE_BUCKETS 4096      // fine buckets of a spill: the top 12 bits of key_hi
#define COLLATE_MAX_PARTS 4096    // most buckets one partition takes (one shared-memory counter each)

// The rows of one spill: bucket = the top 12 bits of the name key (every read lies in one bucket); a row moves with
// its file-order position pos0 + i.
struct SpillPart {
  const u64 *lo, *hi;
  const int32_t *tg, *hp;
  u64 pos0;
  u64 *olo, *ohi;
  int32_t *otg, *ohp;
  u32* opos;
  __device__ __forceinline__ u32 bucket(u64 i) const { return (u32)(hi[i] >> 52); }
  __device__ __forceinline__ void move(u64 i, u64 p) const {
    olo[p] = lo[i];
    ohi[p] = hi[i];
    otg[p] = tg[i];
    ohp[p] = hp[i];
    opos[p] = (u32)(pos0 + i);
  }
};

// Rows with their places in collated order: bucket = the piece that holds the place (cuts[0 .. k], cuts[0] = 0).
struct PiecePart {
  const u32 *id, *place;
  const int32_t *tg, *hp;
  const u32* cuts;
  u32 k;
  u32 *oid, *oplace;
  int32_t *otg, *ohp;
  __device__ __forceinline__ u32 bucket(u64 i) const {
    const u32 p = place[i];
    u32 lo = 0, hi = k;   // largest j < k with cuts[j] <= p
    while (hi - lo > 1) {
      const u32 mid = (lo + hi) >> 1;
      if (cuts[mid] <= p) lo = mid; else hi = mid;
    }
    return lo;
  }
  __device__ __forceinline__ void move(u64 i, u64 p) const {
    oid[p] = id[i];
    oplace[p] = place[i];
    otg[p] = tg[i];
    ohp[p] = hp[i];
  }
};

// Stable partition of rows [0, m) into nb <= COLLATE_MAX_PARTS buckets, one tile of COLLATE_TILE rows per CTA.
// count: per-CTA shared-memory histogram -> counts[bucket * tiles + tile]; an exclusive scan of counts gives every
// (bucket, tile) its first output row; scatter: the rows of a tile go out in rounds of one row per thread, and the
// warps of a round take their places in warp order (lanes of one bucket inside a warp: one counter update, places in
// lane order), so every bucket keeps the input order.  The scanned counters of tile 0 are the bucket offsets.
template <class Part>
__global__ void __launch_bounds__(256) ecb_part_count_kernel(const Part P, u64 m, u32 nb, u32 tiles, u32* __restrict__ counts) {
  __shared__ u32 h[COLLATE_MAX_PARTS];
  for (u32 b = threadIdx.x; b < nb; b += blockDim.x) h[b] = 0;
  __syncthreads();
  const u64 a = (u64)blockIdx.x * COLLATE_TILE, e = min(m, a + COLLATE_TILE);
  for (u64 i = a + threadIdx.x; i < e; i += blockDim.x) atomicAdd(&h[P.bucket(i)], 1u);
  __syncthreads();
  for (u32 b = threadIdx.x; b < nb; b += blockDim.x) counts[(u64)b * tiles + blockIdx.x] = h[b];
}

template <class Part>
__global__ void __launch_bounds__(256) ecb_part_scatter_kernel(const Part P, u64 m, u32 nb, u32 tiles,
                                                               const u32* __restrict__ base) {
  __shared__ u32 cur[COLLATE_MAX_PARTS];
  for (u32 b = threadIdx.x; b < nb; b += blockDim.x) cur[b] = base[(u64)b * tiles + blockIdx.x];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  const u64 a = (u64)blockIdx.x * COLLATE_TILE, e = min(m, a + COLLATE_TILE);
  for (u64 r = a; r < e; r += blockDim.x) {
    const u64 i = r + threadIdx.x;
    const bool valid = i < e;
    const u32 b = valid ? P.bucket(i) : ECB_NONE;
    const u32 same = __match_any_sync(ECB_FULL, b);
    const int leader = __ffs(same) - 1;
    const u32 below = (u32)__popc(same & ((1u << lane) - 1u));
    for (int w = 0; w < n_warps; ++w) {
      if (warp == w) {
        u32 start = 0;
        if (valid && lane == leader) {
          start = cur[b];
          cur[b] = start + (u32)__popc(same);
        }
        start = __shfl_sync(ECB_FULL, start, leader);
        if (valid) P.move(i, (u64)start + below);
      }
      __syncthreads();
    }
  }
}

// A group's reads as (first position, alignments), one per occupied slot of its table, at list[atomic cursor].
__global__ void __launch_bounds__(256) ecb_collate_list_kernel(const EcbEntry* __restrict__ table, u32 slots,
                                                               uint2* __restrict__ list, u32* __restrict__ n_list) {
  for (u32 s = blockIdx.x * blockDim.x + threadIdx.x; s < slots; s += gridDim.x * blockDim.x) {
    const u64 first = table[s].first;
    if (first == ~0ull) continue;
    list[atomicAdd(n_list, 1u)] = make_uint2((u32)first, table[s].countm1 + 1u);
  }
}

// Every row's read's first position.
__global__ void __launch_bounds__(256) ecb_collate_first_kernel(const u32* __restrict__ slot_of,
                                                                const EcbEntry* __restrict__ table, u64 n,
                                                                u32* __restrict__ first) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    first[i] = (u32)table[slot_of[i]].first;
}

__device__ __forceinline__ u32 collate_rank(const u32* __restrict__ bitmap, const u32* __restrict__ word_rank, u32 first) {
  const u32 w = first >> 5, b = first & 31;
  return word_rank[w] + (u32)__popc(bitmap[w] & ((1u << b) - 1u));
}

// ecb_collate_ids_kernel fed from a read list: alignments of the read whose first position ranks id -> count[id].
__global__ void __launch_bounds__(256) ecb_collate_list_ids_kernel(const uint2* __restrict__ list, u64 n,
                                                                   const u32* __restrict__ bitmap,
                                                                   const u32* __restrict__ word_rank, u32* __restrict__ count) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const uint2 r = list[i];
    count[collate_rank(bitmap, word_rank, r.x)] = r.y;
  }
}

// Every row takes its read id and its place in collated order: the read's offset + a per-read cursor (cursor[id]
// holds the offset on entry; lanes of one read inside a warp take one atomic).  first[] is overwritten by the place.
__global__ void __launch_bounds__(256) ecb_collate_place_kernel(u32* __restrict__ first, u64 n, const u32* __restrict__ bitmap,
                                                                const u32* __restrict__ word_rank, u32* __restrict__ cursor,
                                                                u32* __restrict__ id_out) {
  const int lane = threadIdx.x & 31;
  const u64 n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 w0 = (((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5) << 5; w0 < n; w0 += n_warps << 5) {
    const u64 i = w0 + (u64)lane;
    if (i >= n) continue;
    const u32 act = __activemask();
    const u32 f = first[i];
    const u32 same = __match_any_sync(act, f);
    const int leader = __ffs(same) - 1;
    const u32 id = collate_rank(bitmap, word_rank, f);
    u32 base = 0;
    if (lane == leader) base = atomicAdd(&cursor[id], (u32)__popc(same));
    base = __shfl_sync(act, base, leader);
    id_out[i] = id;
    first[i] = base + (u32)__popc(same & ((1u << lane) - 1u));
  }
}

// One piece [a, a + len) of the collated columns: every row lands at place - a.
__global__ void __launch_bounds__(256) ecb_collate_piece_kernel(const u32* __restrict__ id, const int32_t* __restrict__ tg_in,
                                                                const int32_t* __restrict__ hp_in,
                                                                const u32* __restrict__ place, u64 n, u32 a,
                                                                int32_t* __restrict__ rg, int32_t* __restrict__ tg,
                                                                int32_t* __restrict__ hp) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const u32 p = place[i] - a;
    rg[p] = (int32_t)id[i];
    tg[p] = tg_in[i];
    hp[p] = hp_in[i];
  }
}
