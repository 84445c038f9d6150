// ecb_finalize.cuh — EC id assignment and CSR/CSC emission.
//
// Replaces the id half of alntools/bam_utils.py:693-698 (ec_idx[k] = len(ec_idx): EC id = rank of the
// key's first occurrence) without a sort: every kept EC sets the bit of its first-occurrence position
// in a bitmap over the pushed alignment range, a device-wide scan of the word popcounts ranks the
// bits, and the rank IS the EC id.  Then alntools/bam_utils.py:827-847 + bin_utils.py:208-232 in one
// pass in EC-id order (ecb_fin_emit_kernel): row lengths -> exclusive scan -> a_indptr, rows copied from
// the arena, counts.
//   mark   provisional order: first position and count out of the table, the bitmap bit
//   rank   provisional order: id = bitmap rank; ecid_of[e] = id and the one scatter prov_of[id] = e
//   emit   id order, in tiles of FIN_EMIT_TILE ids: the row lengths scanned with the look-back of
//          ecb_scan.cuh, a_indptr / N written coalesced, the tile's rows copied to their contiguous
//          output range with coalesced stores
#pragma once
#include "ecb_common.cuh"
#include "ecb_scan.cuh"

struct FinalizeParams {
  const EcbEntry* table;
  const u32* ec_slot;
  const u32* row_len;
  const u32* row_off;   // absolute arena offsets
  const uint2* arena;
  const u32* ec_keep;   // NULL = keep every EC (single-sample)
  u32 n_ec;             // provisional ids
  u64 min_base;
  u32* bitmap;
  const u32* word_rank;
  u64* first_rel;       // [n_ec]
  u32* ecid_of;         // [n_ec] final id or ECB_NONE
  u32* prov_of;         // [E] provisional id of every final id
  u32 n_final;          // E
  int32_t* a_indptr;    // [E+1]
  int32_t* a_indices;
  int32_t* a_data;
  int32_t* n_indices;   // single-sample N matrix
  int32_t* n_data;
  int32_t* n_indptr;    // single-sample N matrix: the pair (0, E)
  u32* count_of;        // [n_ec] reads per EC (copied out of the table by the mark kernel)
  u64* scan_state;      // look-back state of the emit pass (ecb_scan.cuh); the total of the row lengths lands
                        // after the status words
  u32 n_tiles;          // emit tiles
  u64 z_cap;            // room in a_indices / a_data
};

__global__ void __launch_bounds__(256) ecb_fin_mark_kernel(const FinalizeParams P) {
  for (u32 e = blockIdx.x * blockDim.x + threadIdx.x; e < P.n_ec; e += gridDim.x * blockDim.x) {
    const EcbEntry* en = P.table + P.ec_slot[e];
    const u64 rel = en->first - P.min_base;
    P.first_rel[e] = rel;
    if (P.count_of) P.count_of[e] = en->countm1 + 1u;
    if (P.ec_keep == nullptr || P.ec_keep[e]) atomicOr(&P.bitmap[rel >> 5], 1u << (rel & 31));
  }
}

__global__ void __launch_bounds__(256) ecb_fin_rank_kernel(const FinalizeParams P) {
  for (u32 e = blockIdx.x * blockDim.x + threadIdx.x; e < P.n_ec; e += gridDim.x * blockDim.x) {
    const bool kept = P.ec_keep == nullptr || P.ec_keep[e];
    if (!kept) {
      P.ecid_of[e] = ECB_NONE;
      continue;
    }
    const u64 rel = P.first_rel[e];
    const u32 w = (u32)(rel >> 5), b = (u32)(rel & 31);
    const u32 id = P.word_rank[w] + __popc(P.bitmap[w] & ((1u << b) - 1u));
    P.ecid_of[e] = id;
    P.prov_of[id] = e;
  }
}

#define FIN_EMIT_THREADS 256
#define FIN_EMIT_ITEMS 4                                        // consecutive ids per thread
#define FIN_EMIT_TILE (FIN_EMIT_THREADS * FIN_EMIT_ITEMS)
#define FIN_EMIT_WARP_ROWS (32 * FIN_EMIT_ITEMS)

// One tile of FIN_EMIT_TILE final ids per CTA (tiles drawn from the ticket of the look-back state).  Thread t
// owns ids 4t..4t+3 of the tile, so warp w owns the rows of 128 consecutive ids, which fill one contiguous
// range of the output.  The warp walks that range 32 entries at a time: entry j belongs to the first row whose
// end (tile-relative, in shared memory) is beyond j - a search over the warp's 128 row ends - so reads of the
// arena are one row segment per lane group and the stores are coalesced, for rows of any length.
template <bool SINGLE_SAMPLE>
__global__ void __launch_bounds__(FIN_EMIT_THREADS) ecb_fin_emit_kernel(const FinalizeParams P) {
  __shared__ u32 s_end[FIN_EMIT_TILE];   // tile-relative end of every row
  __shared__ u32 s_src[FIN_EMIT_TILE];   // its arena offset
  __shared__ u32 s_scan[9];
  __shared__ u32 s_tile;
  __shared__ u64 s_prefix;
  const u32 tile = scan_take_tile(P.scan_state, &s_tile);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const u32 E = P.n_final;
  const u32 id0 = tile * FIN_EMIT_TILE + threadIdx.x * FIN_EMIT_ITEMS;
  const bool full = id0 + FIN_EMIT_ITEMS <= E;
  u32 e[FIN_EMIT_ITEMS], len[FIN_EMIT_ITEMS], off[FIN_EMIT_ITEMS];
  if (full) {
    const uint4 q = *(const uint4*)(P.prov_of + id0);
    e[0] = q.x; e[1] = q.y; e[2] = q.z; e[3] = q.w;
  } else {
#pragma unroll
    for (int i = 0; i < FIN_EMIT_ITEMS; ++i) e[i] = id0 + i < E ? P.prov_of[id0 + i] : ECB_NONE;
  }
  u32 sum = 0;
#pragma unroll
  for (int i = 0; i < FIN_EMIT_ITEMS; ++i) {
    len[i] = 0;
    off[i] = 0;
    if (e[i] < P.n_ec) {   // (an id no EC took - only when order_base ranges overlapped, which the host then
                           // reports - may hold a stale entry: bounded here, and the stores below by z_cap)
      len[i] = P.row_len[e[i]];
      off[i] = P.row_off[e[i]];
    }
    sum += len[i];
  }
  if (SINGLE_SAMPLE) {
    u32 cnt[FIN_EMIT_ITEMS];
#pragma unroll
    for (int i = 0; i < FIN_EMIT_ITEMS; ++i) cnt[i] = e[i] < P.n_ec ? P.count_of[e[i]] : 0u;
    if (full) {
      *(int4*)(P.n_indices + id0) = make_int4((int)id0, (int)id0 + 1, (int)id0 + 2, (int)id0 + 3);
      *(int4*)(P.n_data + id0) = make_int4((int)cnt[0], (int)cnt[1], (int)cnt[2], (int)cnt[3]);
    } else {
#pragma unroll
      for (int i = 0; i < FIN_EMIT_ITEMS; ++i)
        if (id0 + i < E) {
          P.n_indices[id0 + i] = (int32_t)(id0 + i);
          P.n_data[id0 + i] = (int32_t)cnt[i];
        }
    }
  }
  u32 tile_total;
  const u32 excl = block_excl_scan_u32(sum, s_scan, tile_total);
  if (warp == 0) {
    const u64 p = scan_lookback(P.scan_state, tile, tile_total);
    if (lane == 0) {
      s_prefix = p;
      if (tile == P.n_tiles - 1) {
        const u64 z = p + tile_total;
        P.scan_state[P.n_tiles + 1] = z;
        P.a_indptr[E] = (int32_t)(u32)z;
        if (SINGLE_SAMPLE) {
          P.n_indptr[0] = 0;
          P.n_indptr[1] = (int32_t)E;
        }
      }
    }
  }
  __syncthreads();
  const u64 prefix = s_prefix;
  u32 run = excl, ptr[FIN_EMIT_ITEMS];
#pragma unroll
  for (int i = 0; i < FIN_EMIT_ITEMS; ++i) {
    ptr[i] = (u32)prefix + run;
    run += len[i];
    s_end[threadIdx.x * FIN_EMIT_ITEMS + i] = run;
    s_src[threadIdx.x * FIN_EMIT_ITEMS + i] = off[i];
  }
  if (full) {
    *(int4*)(P.a_indptr + id0) = make_int4((int)ptr[0], (int)ptr[1], (int)ptr[2], (int)ptr[3]);
  } else {
#pragma unroll
    for (int i = 0; i < FIN_EMIT_ITEMS; ++i)
      if (id0 + i < E) P.a_indptr[id0 + i] = (int32_t)ptr[i];
  }
  __syncwarp();   // the warp reads only the row ends its own lanes wrote
  const u32 r0 = warp * FIN_EMIT_WARP_ROWS;
  const u32 w_beg = __shfl_sync(ECB_FULL, excl, 0), w_end = __shfl_sync(ECB_FULL, run, 31);
  for (u32 j = w_beg + lane; j < w_end; j += 32) {
    u32 lo = r0, hi = r0 + FIN_EMIT_WARP_ROWS - 1;   // first row whose end is beyond j (one exists: w_end > j)
    while (lo < hi) {
      const u32 mid = (lo + hi) >> 1;
      if (s_end[mid] > j) hi = mid; else lo = mid + 1;
    }
    const u32 start = lo == r0 ? w_beg : s_end[lo - 1];
    const uint2 v = P.arena[(size_t)s_src[lo] + (j - start)];
    const size_t dst = prefix + j;
    if (dst >= P.z_cap) break;
    P.a_indices[dst] = (int32_t)v.x;
    P.a_data[dst] = (int32_t)v.y;
  }
}
