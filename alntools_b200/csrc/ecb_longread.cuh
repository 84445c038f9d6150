// ecb_longread.cuh — the sort-based pass for reads longer than ECB_MAX_READ_ALIGNMENTS (ECB_OPT_MAX_READ).
//
// The grouping kernel dedups a read inside its warp; past ECB_MAX_READ_ALIGNMENTS that costs O(k^2 / 32)
// shuffles, and the harvest sorts a row in one CTA's shared memory.  So such a read only has its end found
// there and is appended, as (offset, length), to the push's deferred list.  When that list is not empty the
// push runs this pass over the deferred reads' alignments:
//   gather   (read index << 31 | ecb_code(t, h)) for every alignment of every deferred read;
//   sort     the existing LSD radix sort (ecb_sort.cuh) on the bits those keys use: every read's codes come out
//            contiguous and ascending, equal codes next to each other;
//   sums     per read, the sum of ecb_mix over its DISTINCT codes and their number, and a flag at the first code
//            of every (read, target) run, which a device scan turns into row ranks.  ecb_mix summed over the
//            distinct elements is the key the grouping kernel gives the same set (the sum is commutative), so a
//            long read and a short read with one set of (target, haplotype) pairs are one EC;
//   insert   one thread per read into the EC table (count 1, first = rep = the read's offset, len = its length);
//            a read that finds the table too full is inserted again after the push has grown it;
//   rows     for the ECs a deferred read claimed, the row from the sorted codes: distinct targets ascending, the
//            OR of 1 << hap per target, reserved on the arena cursor (at most one entry per alignment);
//   verify   (ECB_OPT_VERIFY_KEYS) every deferred read's distinct set against its EC's row.
// Device memory: 24 bytes per deferred alignment for the sort, 4 for the ranks, 32 per deferred read.
#pragma once
#include "ecb_common.cuh"
#include "ecb_group.cuh"

#define ECB_LONG_THREADS 256

// Per deferred read.  a..d: sum of ecb_mix over its distinct codes; ec: provisional id of the EC it claimed
// (ECB_NONE: the EC was there already); pending: not yet in the table; row_off: its row's place in the arena.
struct LongAcc {
  u32 a, b, c, d;
  u32 distinct;
  u32 ec;
  u32 pending;
  u32 row_off;
};

struct LongParams {
  const int32_t* tg;
  const int32_t* hp;
  const uint2* reads;   // [n_reads] (offset in the push, length), ascending offsets
  const u32* start;     // [n_reads + 1] first place of each read in the gathered array
  u32 n_reads;
  u32 total;            // gathered alignments = start[n_reads]
  int n_targets, n_haps;
  u64* keys;            // [total] gather output = sort input
  u32* vals;
  const u64* sorted;    // [total] sort output
  u32* rank;            // [total + 1] target-run flags, scanned in place into exclusive ranks
  LongAcc* acc;         // [n_reads]
  EcbCounters* ctr;
};

__device__ __forceinline__ u32 long_read_of(const u32* start, u32 n_reads, u32 i) {
  u32 lo = 0, hi = n_reads;   // the last r with start[r] <= i
  while (hi - lo > 1) {
    const u32 mid = (lo + hi) >> 1;
    if (start[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(ECB_LONG_THREADS) ecb_long_gather_kernel(const LongParams L) {
  const u32 stride = gridDim.x * blockDim.x;
  const u32 tid = blockIdx.x * blockDim.x + threadIdx.x;
  for (u32 r = tid; r < L.n_reads; r += stride) L.acc[r] = LongAcc{0u, 0u, 0u, 0u, 0u, ECB_NONE, 1u, 0u};
  bool bad = false;
  for (u32 i = tid; i < L.total; i += stride) {
    const u32 r = long_read_of(L.start, L.n_reads, i);
    const u32 pos = L.reads[r].x + (i - L.start[r]);
    const int t = L.tg[pos], h = L.hp[pos];
    bad |= (u32)t >= (u32)L.n_targets || (u32)h >= (u32)L.n_haps;
    L.keys[i] = ((u64)r << 31) | ecb_code(t, h);
    L.vals[i] = i;
  }
  if (bad) atomicOr(&L.ctr->error, ECB_DEVERR_VALUE_RANGE);
}

// Block-wide sum of five counters into acc[r] (r block-uniform; ECB_NONE: nothing to add).  Ends with the
// accumulators cleared.
__device__ __forceinline__ void long_flush(LongAcc* acc, u32 r, u32 (&v)[5], u32 (*sm)[5]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < 5; ++j) {
    const u32 s = __reduce_add_sync(ECB_FULL, v[j]);
    if (lane == 0) sm[warp][j] = s;
    v[j] = 0u;
  }
  __syncthreads();
  if (threadIdx.x < 5 && r != ECB_NONE) {
    u32 s = 0;
    for (int w = 0; w < ECB_LONG_THREADS / 32; ++w) s += sm[w][threadIdx.x];
    if (s) atomicAdd(&acc[r].a + threadIdx.x, s);   // a, b, c, d, distinct are consecutive
  }
  __syncthreads();
}

// Sums of the sorted codes.  The array is cut into tiles of one block; a tile that holds one read (the usual
// case: a read has more than 16384 codes) adds into the block's registers, which go to acc[] when the read
// changes, with one atomic per counter and block; a tile across a read boundary adds code by code.
__global__ void __launch_bounds__(ECB_LONG_THREADS) ecb_long_sums_kernel(const LongParams L) {
  __shared__ u32 sm[ECB_LONG_THREADS / 32][5];
  u32 v[5] = {0u, 0u, 0u, 0u, 0u};
  u32 cur = ECB_NONE;
  for (u32 t0 = blockIdx.x * ECB_LONG_THREADS; t0 < L.total; t0 += gridDim.x * ECB_LONG_THREADS) {
    const u32 i = t0 + threadIdx.x;
    const bool in = i < L.total;
    u64 k = 0, prev = ~0ull;
    if (in) {
      k = L.sorted[i];
      if (i > 0) prev = L.sorted[i - 1];
    }
    const bool distinct = in && k != prev;
    if (in) L.rank[i] = (i == 0 || (k >> 5) != (prev >> 5)) ? 1u : 0u;   // first code of a (read, target) run
    if (i == L.total) L.rank[i] = 0u;
    const u32 r = (u32)(k >> 31);
    const u32 rf = (u32)(L.sorted[t0] >> 31);
    const u32 rl = (u32)(L.sorted[min(t0 + ECB_LONG_THREADS, L.total) - 1] >> 31);
    Mix4 m = distinct ? ecb_mix((u32)k & 0x7FFFFFFFu) : mix_zero();
    if (rf == rl) {   // block-uniform
      if (rf != cur) {
        long_flush(L.acc, cur, v, sm);
        cur = rf;
      }
      v[0] += m.a; v[1] += m.b; v[2] += m.c; v[3] += m.d; v[4] += distinct ? 1u : 0u;
    } else if (distinct) {
      LongAcc* A = L.acc + r;
      atomicAdd(&A->a, m.a);
      atomicAdd(&A->b, m.b);
      atomicAdd(&A->c, m.c);
      atomicAdd(&A->d, m.d);
      atomicAdd(&A->distinct, 1u);
    }
  }
  if (L.total % ECB_LONG_THREADS == 0 && blockIdx.x == 0 && threadIdx.x == 0) L.rank[L.total] = 0u;
  long_flush(L.acc, cur, v, sm);
}

// One thread per pending deferred read: into the EC table as ecb_replay_kernel does, knowing whether it claimed.
__global__ void __launch_bounds__(ECB_LONG_THREADS) ecb_long_insert_kernel(const GroupParams P, const LongParams L) {
  for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < L.n_reads; r += gridDim.x * blockDim.x) {
    LongAcc* A = L.acc + r;
    if (!A->pending) continue;
    const uint2 rd = L.reads[r];
    const Key128 key = key_of(key_words(Mix4{A->a, A->b, A->c, A->d}));
    bool claimed;
    u64 first_seen;
    const u32 slot = table_find_or_claim<true>(P.table, P.mask, key, claimed, first_seen);
    if (slot != ECB_NONE) {
      EcbEntry* e = P.table + slot;
      atomicAdd(&e->countm1, 1u);
      const u64 pos = P.order_base + rd.x;
      if (pos < first_seen) atomicMin(&e->first, pos);
    }
    const u32 ecl = alloc_ec_ids(P.ctr, claimed);
    if (claimed) {
      P.table[slot].aux = ecl;
      P.ec_slot[ecl] = slot;
      P.ec_rep[ecl] = rd.x;
      P.ec_len[ecl] = rd.y;
    }
    if (slot == ECB_NONE) {   // table too full: the host grows it and calls this kernel again
      atomicAdd(&P.ctr->n_deferred_fail, 1u);
      continue;
    }
    A->ec = claimed ? ecl : ECB_NONE;
    A->pending = 0u;
    if (P.cell) triple_upsert(P, slot, (u32)P.cell[rd.x], P.order_base + rd.x);
    atomicAdd(&P.ctr->n_reads, 1ull);
  }
}

// Row place of every EC a deferred read claimed: its length is the read's number of (read, target) runs.
__global__ void __launch_bounds__(ECB_LONG_THREADS) ecb_long_rows_reserve_kernel(const LongParams L, u32* row_len,
                                                                                 u32* row_off) {
  for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < L.n_reads; r += gridDim.x * blockDim.x) {
    LongAcc* A = L.acc + r;
    if (A->ec == ECB_NONE) continue;
    const u32 len = L.rank[L.start[r + 1]] - L.rank[L.start[r]];
    const u32 off = (u32)atomicAdd((unsigned long long*)&L.ctr->arena_used, (unsigned long long)len);
    A->row_off = off;
    row_off[A->ec] = off;
    row_len[A->ec] = len;
  }
}

// Place of sorted code i in its read's row (its target's rank inside the read); ECB_NONE when its read claimed no EC.
__device__ __forceinline__ u32 long_row_slot(const LongParams& L, u32 i, u64 k, u64 prev, u32& r) {
  r = (u32)(k >> 31);
  const bool head = i == 0 || (k >> 5) != (prev >> 5);
  return L.rank[i] + (head ? 0u : ~0u) - L.rank[L.start[r]];   // rank[i] counts the runs before i
}

// Rows, in two passes: the first code of every target writes (target, 0), then every distinct code ORs its bit.
template <bool OR_PASS>
__global__ void __launch_bounds__(ECB_LONG_THREADS) ecb_long_rows_kernel(const LongParams L, uint2* arena) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < L.total; i += gridDim.x * blockDim.x) {
    const u64 k = L.sorted[i];
    const u64 prev = i > 0 ? L.sorted[i - 1] : ~0ull;
    u32 r;
    const u32 j = long_row_slot(L, i, k, prev, r);
    const LongAcc& A = L.acc[r];
    if (A.ec == ECB_NONE) continue;
    if (!OR_PASS) {
      if (i == 0 || (k >> 5) != (prev >> 5)) arena[(size_t)A.row_off + j] = make_uint2((u32)(k >> 5) & 0x3FFFFFFu, 0u);
    } else if (k != prev) {
      atomicOr(&arena[(size_t)A.row_off + j].y, 1u << ((u32)k & 31u));
    }
  }
}

// ECB_OPT_VERIFY_KEYS: one CTA per deferred read.  Its key is looked up, and its distinct set compared with the
// row of the EC it was counted in: the row has as many targets as the read, every distinct code of the read is in
// the entry of its target's rank, and the row holds no more haplotype bits than the read has distinct codes.
__global__ void __launch_bounds__(ECB_LONG_THREADS) ecb_long_verify_kernel(const LongParams L, const EcbEntry* table,
                                                                           u32 mask, const u32* row_len,
                                                                           const u32* row_off, const uint2* arena) {
  __shared__ u32 s_id, s_bad, s_bits;
  for (u32 r = blockIdx.x; r < L.n_reads; r += gridDim.x) {
    const LongAcc A = L.acc[r];
    if (threadIdx.x == 0) {
      const Key128 key = key_of(key_words(Mix4{A.a, A.b, A.c, A.d}));
      u32 slot = ec_slot_hash(key) & mask, id = ECB_NONE;
      for (u32 p = 0; p <= mask; ++p) {
        Key128 k;
        u64 first;
        u32 cm1, aux;
        load_entry_cg(table + slot, k, first, cm1, aux);
        if (key_eq(k, key)) {
          id = aux;
          break;
        }
        if (key_empty(k)) break;
        slot = (slot + 1) & mask;
      }
      s_id = id;
      s_bad = id == ECB_NONE ||
              row_len[id] != L.rank[L.start[r + 1]] - L.rank[L.start[r]];
      s_bits = 0;
    }
    __syncthreads();
    const u32 id = s_id;
    const bool found = !s_bad;
    __syncthreads();   // every thread has read s_bad before any sets it below
    if (found) {
      const uint2* row = arena + row_off[id];
      const u32 rl = row_len[id];
      u32 bits = 0;
      for (u32 j = threadIdx.x; j < rl; j += blockDim.x) bits += __popc(row[j].y);
      bits = __reduce_add_sync(ECB_FULL, bits);
      if ((threadIdx.x & 31) == 0 && bits) atomicAdd(&s_bits, bits);
      bool bad = false;
      for (u32 i = L.start[r] + threadIdx.x; i < L.start[r + 1]; i += blockDim.x) {
        const u64 k = L.sorted[i];
        const u64 prev = i > 0 ? L.sorted[i - 1] : ~0ull;
        if (k == prev) continue;
        u32 rr;
        const u32 j = long_row_slot(L, i, k, prev, rr);
        if (j >= rl) {
          bad = true;
          continue;
        }
        const uint2 e = row[j];
        bad |= e.x != ((u32)(k >> 5) & 0x3FFFFFFu) || !((e.y >> ((u32)k & 31u)) & 1u);
      }
      if (bad) s_bad = 1u;
    }
    __syncthreads();
    if (threadIdx.x == 0 && (s_bad || s_bits != A.distinct)) atomicOr(&L.ctr->error, ECB_DEVERR_VERIFY);
    __syncthreads();
  }
}
