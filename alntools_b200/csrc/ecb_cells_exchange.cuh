// ecb_cells_exchange.cuh — kernels of the per-cell (multisample) multi-GPU exchange.
//
// The EC half reuses the single-sample exchange (ecb_exchange.cuh): ECs go to their owner by key, are merged
// there, go on to the rank whose positions hold their first occurrence, and rows never travel.  What is new
// concerns cells:
//   * every rank summarises its cells by GLOBAL cell id (the ranks agree on ids through their name lists):
//     local sort key and local total; the ranks all-gather the keys and all-reduce the totals;
//   * every rank takes the same cell decision: a cell's global key is (first rank that holds it, that rank's
//     key).  Order keys are rank-major (order_base = rank * 2^40 + ...), so every position of a rank lies
//     behind those of all ranks in front of it and the comparison is exact;
//   * (EC, cell) pairs with a kept column travel with the ECs: to the owner of the EC's key (counts summed),
//     then to the rank that holds the EC's first occurrence, where they take the EC's slice-local id.
//
// One IPC allocation carries both record kinds: [header | EC area | header | pair area].  Each header is the
// {records, unused, overflow} triple of ecb_exchange.cuh.
#pragma once
#include "ecb_common.cuh"
#include "ecb_group.cuh"
#include "ecb_exchange.cuh"

#define ECB_CPAIR1_WORDS 3   // dispatch 1: {key_lo, key_hi, column | count << 32}
#define ECB_CPAIR2_WORDS 2   // dispatch 2: {position inside the shard | column << 32, count}

// Local cell key / total (indexed by local cell id) -> the same indexed by global cell id (map NULL: identity).
__global__ void __launch_bounds__(256) cells_summary_kernel(const u64* __restrict__ key_local, const u64* __restrict__ total_local,
                                                            u32 n_local, const int32_t* __restrict__ map, u32 n_cells,
                                                            u64* __restrict__ key_out, u64* __restrict__ total_out, u32* bad) {
  for (u32 l = blockIdx.x * blockDim.x + threadIdx.x; l < n_local; l += gridDim.x * blockDim.x) {
    const u32 g = map ? (u32)map[l] : l;
    if (g >= n_cells) {
      if (total_local[l]) atomicOr(bad, 1u);   // a cell with reads has no place in the global id space
      continue;
    }
    key_out[g] = key_local[l];
    total_out[g] = total_local[l];
  }
}

// Sort input of the cell decision, pass 1: every cell's key on the first rank that holds it (~0: absent).
__global__ void __launch_bounds__(256) cells_first_key_kernel(const u64* __restrict__ keys_all, u32 world, u32 n_cells,
                                                              u64* __restrict__ sort_k, u32* __restrict__ sort_v) {
  for (u32 c = blockIdx.x * blockDim.x + threadIdx.x; c < n_cells; c += gridDim.x * blockDim.x) {
    u64 k = ~0ull;
    for (u32 r = 0; r < world && k == ~0ull; ++r) k = keys_all[(size_t)r * n_cells + c];
    sort_k[c] = k;
    sort_v[c] = c;
  }
}

// ... pass 2 (a stable sort on the rank follows the sort on the key): the first rank that holds the cell, ~0 when
// none does.  k_out / v_out may alias v_in's buffers.
__global__ void __launch_bounds__(256) cells_first_rank_kernel(const u64* __restrict__ keys_all, u32 world, u32 n_cells,
                                                               const u32* v_in, u64* k_out, u32* v_out) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_cells; i += gridDim.x * blockDim.x) {
    const u32 c = v_in[i];
    u64 rk = ~0ull;
    for (u32 r = 0; r < world; ++r)
      if (keys_all[(size_t)r * n_cells + c] != ~0ull) {
        rk = r;
        break;
      }
    k_out[i] = rk;
    v_out[i] = c;
  }
}

// Output column of every LOCAL cell id.
__global__ void __launch_bounds__(256) cells_local_columns_kernel(const int32_t* __restrict__ map, u32 n_local,
                                                                  const int32_t* __restrict__ column_of_cell, u32 n_cells,
                                                                  int32_t* __restrict__ cell_new) {
  for (u32 l = blockIdx.x * blockDim.x + threadIdx.x; l < n_local; l += gridDim.x * blockDim.x) {
    const u32 g = map ? (u32)map[l] : l;
    cell_new[l] = g < n_cells ? column_of_cell[g] : -1;
  }
}

// Reads of every local EC that fall in kept cells (by provisional id).
__global__ void __launch_bounds__(256) cells_kept_reads_kernel(const EcbEntry* __restrict__ pair_table, u32 pair_mask,
                                                               const EcbEntry* __restrict__ ec_table,
                                                               const int32_t* __restrict__ cell_new, u32* kept) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i <= pair_mask; i += gridDim.x * blockDim.x) {
    const EcbEntry e = pair_table[i];
    if (key_empty(Key128{e.key_lo, e.key_hi})) continue;
    if (cell_new[(u32)(e.key_lo & 0xFFFFFFFFull)] >= 0) atomicAdd(&kept[ec_table[(u32)(e.key_lo >> 32)].aux], e.countm1 + 1u);
  }
}

// Where a record goes and what it says.  ORDER = false (dispatch 1, on a LOCAL context): the pairs of the local
// pair table (key_lo = EC slot << 32 | local cell) with a kept column, to the owner of the EC's key.  ORDER = true
// (dispatch 2, on an OWNER context): the merged pairs (key_lo = owner EC id << 32 | column), to the rank whose
// shard holds the EC's first occurrence.
struct CellPairDispatchParams {
  const EcbEntry* pair_table;
  u32 pair_slots;                // 0: no pairs
  const EcbEntry* ec_table;
  const u32* ec_slot;            // ORDER: owner EC id -> slot
  const int32_t* cell_new;       // !ORDER: local cell -> column
  u32 world;
  u64 lo[ECB_MAX_WORLD];         // ORDER: as KeyDispatchParams
  u32 dest[ECB_MAX_WORLD];
  u32 n_shards;
};

template <bool ORDER>
__device__ __forceinline__ bool cells_pair_route(const CellPairDispatchParams& P, u32 i, u32& dest, unsigned long long* r) {
  const EcbEntry e = P.pair_table[i];
  if (key_empty(Key128{e.key_lo, e.key_hi})) return false;
  const u32 count = e.countm1 + 1u;
  if (ORDER) {
    const u32 column = (u32)(e.key_lo & 0xFFFFFFFFull);
    const u64 first = P.ec_table[P.ec_slot[(u32)(e.key_lo >> 32)]].first;
    u32 k = 0;
    while (k + 1 < P.n_shards && P.lo[k + 1] <= first) ++k;
    dest = P.dest[k];
    const u64 rel = first - P.lo[k];
    r[0] = (rel > 0xFFFFFFFEull ? 0xFFFFFFFFull : rel) | ((unsigned long long)column << 32);
    r[1] = count;
  } else {
    const int32_t column = P.cell_new[(u32)(e.key_lo & 0xFFFFFFFFull)];
    if (column < 0) return false;
    const EcbEntry& en = P.ec_table[(u32)(e.key_lo >> 32)];
    dest = ecb_owner_of(Key128{en.key_lo, en.key_hi}, P.world);
    r[0] = en.key_lo;
    r[1] = en.key_hi;
    r[2] = (u32)column | ((unsigned long long)count << 32);
  }
  return true;
}

// Exact records per destination of both record kinds: counts[dest] (ECs), counts[world + dest] (pairs).  The EC
// half follows ecb_key_dispatch_kernel's routing (dispatch 2: merged ECs with kept reads only).
template <bool ORDER>
__global__ void __launch_bounds__(256) cells_dispatch_count_kernel(const KeyDispatchParams K, const CellPairDispatchParams P,
                                                                   unsigned long long* counts) {
  __shared__ u32 s_cnt[2 * ECB_MAX_WORLD];
  for (u32 i = threadIdx.x; i < 2 * P.world; i += blockDim.x) s_cnt[i] = 0u;
  __syncthreads();
  const u32 stride = gridDim.x * blockDim.x;
  for (u32 e = blockIdx.x * blockDim.x + threadIdx.x; e < K.n_ec; e += stride) {
    const EcbEntry en = K.table[K.ec_slot[e]];
    u32 dest;
    if (ORDER) {
      if (en.countm1 == 0xFFFFFFFFu) continue;   // no kept read anywhere
      u32 k = 0;
      while (k + 1 < K.n_shards && K.lo[k + 1] <= en.first) ++k;
      dest = K.dest[k];
    } else {
      dest = ecb_owner_of(Key128{en.key_lo, en.key_hi}, K.world);
    }
    atomicAdd(&s_cnt[dest], 1u);
  }
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < P.pair_slots; i += stride) {
    u32 dest;
    unsigned long long r[3];
    if (cells_pair_route<ORDER>(P, i, dest, r)) atomicAdd(&s_cnt[P.world + dest], 1u);
  }
  __syncthreads();
  for (u32 i = threadIdx.x; i < 2 * P.world; i += blockDim.x)
    if (s_cnt[i]) atomicAdd(counts + i, (unsigned long long)s_cnt[i]);
}

// The pairs into their destinations' pair areas: the tile scheme of ecb_key_dispatch_kernel (one remote atomic per
// tile and destination, records staged in shared memory by destination, coalesced stores).
template <bool ORDER>
__global__ void __launch_bounds__(256) cells_pair_dispatch_kernel(const CellPairDispatchParams P, const ArenaTargets A) {
  constexpr u32 WORDS = ORDER ? ECB_CPAIR2_WORDS : ECB_CPAIR1_WORDS;
  __shared__ u32 s_cnt[ECB_MAX_WORLD];
  __shared__ u32 s_off[ECB_MAX_WORLD];
  __shared__ unsigned long long s_base[ECB_MAX_WORLD];
  __shared__ u32 s_drop[ECB_MAX_WORLD];
  __shared__ __align__(16) unsigned long long s_rec[256 * WORDS];
  const u32 W = P.world;
  const u32 n = P.pair_slots;
  const u32 tiles = (n + blockDim.x - 1) / blockDim.x;
  for (u32 tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    for (u32 i = threadIdx.x; i < W; i += blockDim.x) s_cnt[i] = 0u;
    __syncthreads();
    const u32 i = tile * blockDim.x + threadIdx.x;
    unsigned long long r[3];
    u32 dest = 0, idx = 0;
    const bool live = i < n && cells_pair_route<ORDER>(P, i, dest, r);
    if (live) idx = atomicAdd(&s_cnt[dest], 1u);
    __syncthreads();
    if (threadIdx.x < W) {
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
    if (threadIdx.x == 32) {
      u32 ae = 0;
      for (u32 o = 0; o < W; ++o) {
        s_off[o] = ae;
        ae += s_cnt[o];
      }
    }
    __syncthreads();
    if (live && !s_drop[dest]) {
      unsigned long long* d = s_rec + (size_t)(s_off[dest] + idx) * WORDS;
      for (u32 w = 0; w < WORDS; ++w) d[w] = r[w];
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

// Owner merge of the pairs of dispatch 1 (after ecb_import_keys_kernel has merged the ECs): key (owner EC id << 32 |
// column), counts summed.
__global__ void __launch_bounds__(256) cells_pair_import_kernel(const unsigned long long* __restrict__ rec, u32 n_rec,
                                                                const EcbEntry* ec_table, u32 ec_mask, EcbEntry* pair_table,
                                                                u32 pair_mask, EcbCounters* ctr) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += gridDim.x * blockDim.x) {
    const unsigned long long* m = rec + (size_t)i * ECB_CPAIR1_WORDS;
    const u32 slot = ec_table_find(ec_table, ec_mask, Key128{m[0], m[1]});
    if (slot == ECB_NONE) {   // every pair's EC travelled in the same dispatch
      atomicOr(&ctr->error, ECB_DEVERR_EC_CAPACITY);
      continue;
    }
    const u32 id = ec_table[slot].aux;
    bool claimed;
    u64 seen;
    const u32 ps = table_find_or_claim(pair_table, pair_mask, Key128{((u64)id << 32) | (m[2] & 0xFFFFFFFFull), 0ull},
                                       claimed, seen);
    if (ps == ECB_NONE) {
      atomicOr(&ctr->error, ECB_DEVERR_EC_CAPACITY);
      continue;
    }
    atomicAdd(&pair_table[ps].countm1, (u32)(m[2] >> 32));
  }
}

// Slice build of the pairs of dispatch 2: the slice-local id of the pair's EC is the rank of its bit in the
// bitmap of ecb_order_mark_kernel.  Sort input: column << 32 | id -> count.  bad: 8 = no EC at the position,
// 16 = column out of range.
__global__ void __launch_bounds__(256) cells_pair_slice_kernel(const unsigned long long* __restrict__ rec, u32 n_rec, u32 span,
                                                               u32 n_samples, const u32* __restrict__ bitmap,
                                                               const u32* __restrict__ word_rank, u64* __restrict__ keys,
                                                               u32* __restrict__ vals, u32* bad) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_rec; i += gridDim.x * blockDim.x) {
    const unsigned long long w0 = rec[(size_t)i * ECB_CPAIR2_WORDS];
    const u32 rel = (u32)(w0 & 0xFFFFFFFFull), column = (u32)(w0 >> 32);
    u32 id = 0;
    if (column >= n_samples) atomicOr(bad, 16u);
    if (rel >= span || !((bitmap[rel >> 5] >> (rel & 31)) & 1u)) atomicOr(bad, 8u);
    else id = word_rank[rel >> 5] + (u32)__popc(bitmap[rel >> 5] & ((1u << (rel & 31)) - 1u));
    keys[i] = ((u64)column << 32) | id;
    vals[i] = (u32)rec[(size_t)i * ECB_CPAIR2_WORDS + 1];
  }
}

// Sorted (column, id) pairs -> per-column entry counts (col_counts zeroed: a column's run [s, e) adds e at its
// last entry and subtracts s at its first - two updates per column, none per entry), indices, data.
__global__ void __launch_bounds__(256) cells_slice_csc_kernel(const u64* __restrict__ keys, const u32* __restrict__ vals, u32 nnz,
                                                              int32_t* col_counts, int32_t* __restrict__ indices,
                                                              int32_t* __restrict__ data) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += gridDim.x * blockDim.x) {
    const u32 col = (u32)(keys[i] >> 32);
    if (i == 0 || (u32)(keys[i - 1] >> 32) != col) atomicSub(&col_counts[col], (int32_t)i);
    if (i + 1 == nnz || (u32)(keys[i + 1] >> 32) != col) atomicAdd(&col_counts[col], (int32_t)(i + 1));
    indices[i] = (int32_t)(keys[i] & 0xFFFFFFFFull);
    data[i] = (int32_t)vals[i];
  }
}
