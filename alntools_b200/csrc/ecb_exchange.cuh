// ecb_exchange.cuh — kernels of the multi-GPU exchange (SURVEY 8e).
//
// Reads shard across GPUs by contiguous chunk (the reference's utils.partition + ordered imap,
// alntools/bam_utils.py:647-680); every GPU builds a local EC table.  Global dedup = the chunk merge
// of alntools/bam_utils.py:680-698 (sum the counts of equal keys, EC id = rank of the GLOBAL first
// occurrence).  It runs over peer memory: two dispatches of fixed-size records through IPC-mapped arenas,
// rows never travel, nothing global is built - see "the exchange over peer memory" below.
#pragma once
#include "ecb_common.cuh"
#include "ecb_group.cuh"

#define ECB_MAX_WORLD 64

__device__ __forceinline__ u32 ecb_owner_of(const Key128& k, u32 world) {
  return fmix32((u32)(k.hi >> 32) ^ 0x5bd1e995u) % world;
}

// ---- the exchange over peer memory: two dispatches of fixed-size records, no rows ----------------------
// Every rank owns an ARENA (plain cudaMalloc, mapped into its peers through CUDA IPC): a small header
// {records, unused, overflow} followed by a record area.
//
// Dispatch 1 - by key: every local EC goes as {key_lo, key_hi, first, count} to its OWNER rank (hash of the
// key), which merges equal keys (counts summed, smallest first-occurrence kept).
// Dispatch 2 - by first occurrence: every merged EC goes as {key_lo, key_hi, position inside the shard |
// count << 32} to the rank whose SHARD of the read order holds its first occurrence.  EC ids are ranks of
// first-occurrence positions and the shards partition the positions, so a rank receives one contiguous id
// range and orders it with a bitmap over its OWN positions.
// ROWS NEVER TRAVEL: the rank that holds an EC's first occurrence has met that EC in its own reads, so its
// local context already holds the row; the receiver finds it by key in its local table.  (Round 1 and the
// first form of round 2 sent every row twice - 100 bytes per EC on cfg2, kilobytes on heavily multimapping
// input - and copied it into the owner's arena in between.)
// Space in a remote arena is reserved with ONE remote atomicAdd per CTA tile and destination; the tile's
// records are laid out in shared memory grouped by destination and go out with coalesced 8-byte stores -
// NVLink wants long contiguous writes.
#define ECB_ARENA_HEADER_BYTES 256
#define ECB_KEYREC_WORDS 4    // dispatch 1
#define ECB_ORDREC_WORDS 3    // dispatch 2

struct ArenaTargets {
  unsigned long long* hdr[ECB_MAX_WORLD];   // [0] records, [2] overflow flag
  unsigned long long* rec[ECB_MAX_WORLD];
  unsigned long long cap_words;             // 8-byte words of the record area
};

struct KeyDispatchParams {
  const EcbEntry* table;
  const u32* ec_slot;
  u32 n_ec;
  u32 world;
  const u32* count_of;   // dispatch 1: the count sent for provisional id e (NULL: the EC's own count)
  // dispatch 2 only: shards with alignments, ascending by first position, and the rank that holds each
  u64 lo[ECB_MAX_WORLD];
  u32 dest[ECB_MAX_WORLD];
  u32 n_shards;
};

// ORDER = false: dispatch 1 (destination = owner of the key); true: dispatch 2 (destination = rank of the shard
// that holds the first occurrence).  KEPT_ONLY (dispatch 2 of the per-cell exchange): ECs whose merged count is 0
// - no read in a kept cell on any rank - stay behind.
template <bool ORDER, bool KEPT_ONLY = false>
__global__ void __launch_bounds__(256) ecb_key_dispatch_kernel(const KeyDispatchParams P, const ArenaTargets A) {
  constexpr u32 WORDS = ORDER ? ECB_ORDREC_WORDS : ECB_KEYREC_WORDS;
  __shared__ u32 s_cnt[ECB_MAX_WORLD];                  // per tile: records per destination
  __shared__ u32 s_off[ECB_MAX_WORLD];                  // ... their exclusive prefix over the destinations
  __shared__ unsigned long long s_base[ECB_MAX_WORLD];  // where the tile's share starts in the destination's arena
  __shared__ u32 s_drop[ECB_MAX_WORLD];
  __shared__ __align__(16) unsigned long long s_rec[256 * WORDS];
  const u32 W = P.world;
  const u32 tiles = (P.n_ec + blockDim.x - 1) / blockDim.x;
  for (u32 tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    for (u32 i = threadIdx.x; i < W; i += blockDim.x) s_cnt[i] = 0u;
    __syncthreads();
    const u32 e = tile * blockDim.x + threadIdx.x;
    bool live = e < P.n_ec;
    EcbEntry en{};
    u32 dest = 0, idx = 0;
    u64 rel = 0;
    if (live) en = P.table[P.ec_slot[e]];
    if (KEPT_ONLY && en.countm1 == 0xFFFFFFFFu) live = false;
    if (live) {
      if (ORDER) {
        u32 k = 0;   // the last shard that starts at or before the position
        while (k + 1 < P.n_shards && P.lo[k + 1] <= en.first) ++k;
        dest = P.dest[k];
        rel = en.first - P.lo[k];
      } else {
        dest = ecb_owner_of(Key128{en.key_lo, en.key_hi}, W);
      }
      idx = atomicAdd(&s_cnt[dest], 1u);
    }
    __syncthreads();
    if (threadIdx.x < W) {   // reserve space in the destinations' arenas: one remote atomic each
      const u32 o = threadIdx.x;
      const u32 ce = s_cnt[o];
      s_drop[o] = 0u;
      if (ce) {
        const unsigned long long be = atomicAdd(A.hdr[o] + 0, (unsigned long long)ce);
        s_base[o] = be;
        if ((be + ce) * WORDS > A.cap_words) {
          atomicExch(A.hdr[o] + 2, 1ull);
          s_drop[o] = 1u;
        }
      }
    }
    if (threadIdx.x == 32) {   // meanwhile: tile-local offsets of the destinations' segments
      u32 ae = 0;
      for (u32 o = 0; o < W; ++o) {
        s_off[o] = ae;
        ae += s_cnt[o];
      }
    }
    __syncthreads();
    if (live && !s_drop[dest]) {
      unsigned long long* r = s_rec + (size_t)(s_off[dest] + idx) * WORDS;
      r[0] = en.key_lo;
      r[1] = en.key_hi;
      if (ORDER) {
        r[2] = (rel > 0xFFFFFFFEull ? 0xFFFFFFFFull : rel) | ((unsigned long long)(en.countm1 + 1u) << 32);
      } else {
        r[2] = en.first;
        r[3] = (unsigned long long)(P.count_of ? P.count_of[e] : en.countm1 + 1u);
      }
    }
    __syncthreads();
    for (u32 o = 0; o < W; ++o) {
      if (s_cnt[o] == 0u || s_drop[o]) continue;
      const u32 n_words = s_cnt[o] * WORDS;
      const unsigned long long* src = s_rec + (size_t)s_off[o] * WORDS;
      unsigned long long* dst = A.rec[o] + s_base[o] * WORDS;
      for (u32 w = threadIdx.x; w < n_words; w += blockDim.x) dst[w] = src[w];
    }
    __syncthreads();
  }
}

// Owner merge of dispatch 1 (bam_utils.py:693-698: equal keys - counts summed, smallest first occurrence kept).
// Provisional ids of the new keys are reserved once per CTA tile.
struct KeyImportParams {
  const unsigned long long* rec;
  u32 n_rec;
  EcbEntry* table;
  u32 mask;
  u32* ec_slot;
  EcbCounters* ctr;
};

__global__ void __launch_bounds__(256) ecb_import_keys_kernel(const KeyImportParams P) {
  __shared__ u32 s_scan[10];
  const u32 tiles = (P.n_rec + blockDim.x - 1) / blockDim.x;
  for (u32 tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const u32 i = tile * blockDim.x + threadIdx.x;
    bool claimed = false;
    u32 slot = ECB_NONE;
    if (i < P.n_rec) {
      const unsigned long long* m = P.rec + (size_t)i * ECB_KEYREC_WORDS;
      const Key128 key{m[0], m[1]};
      const u64 first = m[2];
      u64 seen;
      slot = table_find_or_claim<true>(P.table, P.mask, key, claimed, seen);
      if (slot == ECB_NONE) {
        atomicOr(&P.ctr->error, ECB_DEVERR_EC_CAPACITY);
        claimed = false;
      } else {
        EcbEntry* e = P.table + slot;
        atomicAdd(&e->countm1, (u32)m[3]);
        if (first < seen) atomicMin(&e->first, first);
      }
    }
    u32 n_new;
    const u32 id_excl = block_excl_scan_u32(claimed ? 1u : 0u, s_scan, n_new);
    if (threadIdx.x == 0) s_scan[9] = n_new ? atomicAdd(&P.ctr->n_ec, n_new) : 0u;
    __syncthreads();
    const u32 id = s_scan[9] + id_excl;
    __syncthreads();
    if (claimed) {
      P.table[slot].aux = id;
      P.ec_slot[id] = slot;
    }
  }
}

// Lookup in an EC table (slot hash of the EC keys); ECB_NONE if absent.
__device__ __forceinline__ u32 ec_table_find(const EcbEntry* table, u32 mask, const Key128& key) {
  u32 slot = ec_slot_hash(key) & mask;
  for (u32 p = 0; p <= mask; ++p) {
    Key128 k;
    u64 first;
    u32 cm1, aux;
    load_entry_cg(table + slot, k, first, cm1, aux);
    if (key_eq(k, key)) return slot;
    if (key_empty(k)) return ECB_NONE;
    slot = (slot + 1) & mask;
  }
  return ECB_NONE;
}

// Slice assembly at the receiver of dispatch 2, pass 0: one bit per arrived EC at its position inside the shard,
// and the EC's id in the LOCAL context (found by key: this rank has met the EC in its own reads).
__global__ void __launch_bounds__(256) ecb_order_mark_kernel(const unsigned long long* __restrict__ rec, u32 n_rec, u32 span,
                                                            const EcbEntry* __restrict__ local_table, u32 local_mask,
                                                            u32* bitmap, u32* local_id, u32* bad) {
  for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += gridDim.x * blockDim.x) {
    const unsigned long long* m = rec + (size_t)r * ECB_ORDREC_WORDS;
    const u32 rel = (u32)(m[2] & 0xFFFFFFFFull);
    const u32 slot = ec_table_find(local_table, local_mask, Key128{m[0], m[1]});
    local_id[r] = slot == ECB_NONE ? ECB_NONE : local_table[slot].aux;
    if (rel >= span || slot == ECB_NONE) {
      atomicOr(bad, slot == ECB_NONE ? 4u : 1u);
      continue;
    }
    const u32 bit = 1u << (rel & 31);
    if (atomicOr(&bitmap[rel >> 5], bit) & bit) atomicOr(bad, 2u);   // two ECs cannot start with the same read
  }
}

// ... pass 1: the rank of its bit is an EC's id inside the slice; row length (of the LOCAL row), merged count and
// local id go there.
__global__ void __launch_bounds__(256) ecb_order_lens_kernel(const unsigned long long* __restrict__ rec, u32 n_rec, u32 span,
                                                            const u32* __restrict__ bitmap, const u32* __restrict__ word_rank,
                                                            const u32* __restrict__ local_id, const u32* __restrict__ local_row_len,
                                                            int32_t* lens, int32_t* counts, u32* id_of) {
  for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < n_rec; r += gridDim.x * blockDim.x) {
    const unsigned long long w2 = rec[(size_t)r * ECB_ORDREC_WORDS + 2];
    const u32 rel = (u32)(w2 & 0xFFFFFFFFull);
    const u32 lid = local_id[r];
    if (rel >= span || lid == ECB_NONE) continue;
    const u32 w = rel >> 5, b = rel & 31;
    const u32 i = word_rank[w] + (u32)__popc(bitmap[w] & ((1u << b) - 1u));
    if (i >= n_rec) continue;   // (only after a duplicate position, which pass 0 has reported)
    lens[i] = (int32_t)local_row_len[lid];
    counts[i] = (int32_t)(w2 >> 32);
    id_of[i] = lid;
  }
}

// ... pass 2: rows from the local arena to their CSR position (thread per id).
__global__ void __launch_bounds__(256) ecb_order_rows_kernel(const u32* __restrict__ id_of, const u32* __restrict__ local_row_len,
                                                            const u32* __restrict__ local_row_off, const uint2* __restrict__ local_arena,
                                                            const int32_t* __restrict__ indptr, u32 slice_n,
                                                            int32_t* indices, int32_t* data) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < slice_n; i += gridDim.x * blockDim.x) {
    const u32 lid = id_of[i];
    const uint2* src = local_arena + local_row_off[lid];
    const u32 len = local_row_len[lid];
    const size_t dst = (size_t)indptr[i];
    for (u32 j = 0; j < len; ++j) {
      indices[dst + j] = (int32_t)src[j].x;
      data[dst + j] = (int32_t)src[j].y;
    }
  }
}

// Shift the first-occurrence key of every EC of a context by `delta` (ecb_rebase): a rank that decodes one
// shard of a file learns the global position of its shard only when all ranks have counted theirs.
__global__ void __launch_bounds__(256) ecb_rebase_kernel(EcbEntry* table, const u32* __restrict__ ec_slot, u32 n_ec,
                                                         u64 delta) {
  for (u32 e = blockIdx.x * blockDim.x + threadIdx.x; e < n_ec; e += gridDim.x * blockDim.x)
    table[ec_slot[e]].first += delta;
}
