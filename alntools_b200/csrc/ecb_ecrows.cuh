// ecb_ecrows.cuh — ECs given as the A rows of an EC file (ecb_push_ecs) and count columns over those rows
// (ecb_sample_append): what a merge of EC files feeds into a single-sample context instead of reads.
//
// A row of an EC file is a set of (target, haplotype) elements, stored as ascending targets with a haplotype mask.
// Its key is the sum of ecb_mix over the elements, the key ecb_push gives a read with that set, so an EC-file row
// and a read with one set are one EC.  One push of n rows:
//   keys     one thread per A entry: the value checks, and the entry's ecb_mix sum over its mask bits, reduced per
//            row with a segmented warp scan (a row held by one warp is stored, a row across warps is added with
//            one atomic per warp and word), so that a long row costs per entry what a short one does;
//   insert   one thread per row: find or claim its key, atomicMin of the first occurrence (order key of row r is
//            base + r), provisional ids with one atomic per warp;
//   reserve  one thread per row: the provisional id of every row, and the arena place of the claimed rows with
//            one atomic per CTA.  Every row stamps its EC with the push's tag; a row that finds the tag there already
//            shares its EC with another row of the push: the file is malformed;
//   copy     one thread per A entry of a claimed row: the (target, mask) pairs as they are (rows are canonical);
//   check    one thread per A entry of a row that found an EC: equal length and equal pairs with the row that EC
//            holds.  A difference means two sets share a 128-bit key.  Always on.
// The append maps every N entry (row, count) to (provisional id, count): a flag pass with the value checks, the
// device scan of the flags, and a pass that writes the pairs in input order and every column's count.
#pragma once
#include "ecb_common.cuh"
#include "ecb_group.cuh"
#include "ecb_harvest.cuh"

#define ECR_THREADS 256

// What EcbCounters::ecr_bad[kind] holds: the first bad A entry, row or N entry of that kind (ECB_NONE: none).
enum {
  ECR_BAD_TARGET = 0,   // entry: target outside [0, n_targets)
  ECR_BAD_ORDER,        // entry: target not above the previous one of its row
  ECR_BAD_MASK,         // entry: mask 0, or a bit at or above n_haps
  ECR_BAD_DUPLICATE,    // row: holds the set of another row of the same push
  ECR_BAD_COLLISION,    // row: shares its 128-bit key with an EC whose row differs
  ECR_BAD_PROBE,        // row: the EC table ran out of probes
  ECR_BAD_N_INDEX,      // N entry: row index outside [0, rows of the last push)
  ECR_BAD_N_COUNT,      // N entry: negative count
  ECR_KINDS
};

struct EcrParams {
  const int32_t* indptr;   // [n_rows + 1], strictly ascending (checked by the host)
  const int32_t* indices;  // [nnz] targets
  const int32_t* data;     // [nnz] haplotype masks
  u32 n_rows, nnz;
  int n_targets, n_haps;
  u64 base;                // order key of row 0
  Mix4* acc;               // [n_rows] key sums
  u32* row_slot;           // [n_rows] table slot | 1 << 31 when the row claimed it
  u32* row_ec;             // [n_rows] provisional EC id
  u32* row_dst;            // [n_rows] arena place of a claimed row; ECB_NONE for a row that found its EC
  u32* seen;               // [provisional ids] tag of the last push that had a row on the EC
  u32 tag;                 // this push's tag (never 0, rises with every push)
  EcbCounters* ctr;
};

__device__ __forceinline__ u32 ecr_row_of(const int32_t* indptr, u32 n_rows, u32 i) {
  u32 lo = 0, hi = n_rows;   // the last r with indptr[r] <= i
  while (hi - lo > 1) {
    const u32 mid = (lo + hi) >> 1;
    if ((u32)indptr[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}

__device__ __forceinline__ void ecr_flag(EcbCounters* ctr, int kind, u32 at) { atomicMin(&ctr->ecr_bad[kind], at); }

__global__ void __launch_bounds__(ECR_THREADS) ecb_ecr_keys_kernel(const EcrParams R) {
  const int lane = threadIdx.x & 31;
  // whole warps walk the entries together: the scan below needs every lane
  for (u32 w0 = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); w0 < R.nnz; w0 += gridDim.x * blockDim.x) {
    const u32 i = w0 + lane;
    u32 r = ECB_NONE;
    Mix4 m = mix_zero();
    if (i < R.nnz) {
      r = ecr_row_of(R.indptr, R.n_rows, i);
      const int t = R.indices[i];
      const u32 mask = (u32)R.data[i];
      if ((u32)t >= (u32)R.n_targets) ecr_flag(R.ctr, ECR_BAD_TARGET, i);
      if (i > (u32)R.indptr[r] && R.indices[i - 1] >= t) ecr_flag(R.ctr, ECR_BAD_ORDER, i);
      if (mask == 0u || (mask >> R.n_haps) != 0u) ecr_flag(R.ctr, ECR_BAD_MASK, i);
      for (u32 b = mask; b; b &= b - 1u) mix_add(m, ecb_mix(ecb_code(t, __ffs(b) - 1)));
    }
    // segmented inclusive scan: a row's entries are consecutive, so equal rows at lane and lane - d mean every
    // lane between holds that row too
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const u32 ru = __shfl_up_sync(ECB_FULL, r, d);
      const u32 a = __shfl_up_sync(ECB_FULL, m.a, d), b = __shfl_up_sync(ECB_FULL, m.b, d);
      const u32 c = __shfl_up_sync(ECB_FULL, m.c, d), e = __shfl_up_sync(ECB_FULL, m.d, d);
      if (lane >= d && ru == r) mix_add(m, Mix4{a, b, c, e});
    }
    const u32 rn = __shfl_down_sync(ECB_FULL, r, 1);
    if (r == ECB_NONE || (lane < 31 && rn == r)) continue;   // not the last entry of its row inside this warp
    if ((u32)R.indptr[r] >= w0 && (u32)R.indptr[r + 1] <= w0 + 32u) {
      R.acc[r] = m;   // the whole row lies in this warp
    } else {
      Mix4* A = R.acc + r;
      atomicAdd(&A->a, m.a);
      atomicAdd(&A->b, m.b);
      atomicAdd(&A->c, m.c);
      atomicAdd(&A->d, m.d);
    }
  }
}

// One thread per row.  The host has grown the table so that it stays at most half full after this push.
__global__ void __launch_bounds__(ECR_THREADS) ecb_ecr_insert_kernel(const GroupParams P, const EcrParams R) {
  for (u32 r = blockIdx.x * blockDim.x + threadIdx.x; r < R.n_rows; r += gridDim.x * blockDim.x) {
    const Key128 key = key_of(key_words(R.acc[r]));
    bool claimed;
    u64 first_seen;
    const u32 slot = table_find_or_claim<true>(P.table, P.mask, key, claimed, first_seen);
    const u64 pos = R.base + r;
    if (slot != ECB_NONE && pos < first_seen) atomicMin(&P.table[slot].first, pos);
    const u32 ecl = alloc_ec_ids(P.ctr, claimed);
    if (claimed) {
      P.table[slot].aux = ecl;
      P.ec_slot[ecl] = slot;
      P.ec_rep[ecl] = r;
      P.ec_len[ecl] = (u32)(R.indptr[r + 1] - R.indptr[r]);
    }
    if (slot == ECB_NONE) ecr_flag(R.ctr, ECR_BAD_PROBE, r);
    R.row_slot[r] = slot == ECB_NONE ? ECB_NONE : slot | (claimed ? 0x80000000u : 0u);
  }
}

__global__ void __launch_bounds__(ECR_THREADS) ecb_ecr_reserve_kernel(const EcrParams R, const EcbEntry* table,
                                                                      u32* row_len, u32* row_off) {
  // whole CTAs walk the rows together (the reservation is a CTA-wide step)
  __shared__ u32 s_scan[10];
  for (u32 r0 = blockIdx.x * blockDim.x; r0 < R.n_rows; r0 += gridDim.x * blockDim.x) {
    const u32 r = r0 + threadIdx.x;
    u32 len = 0, id = ECB_NONE;
    bool claimed = false;
    if (r < R.n_rows) {
      const u32 s = R.row_slot[r];
      if (s != ECB_NONE) {
        id = table[s & 0x7FFFFFFFu].aux;
        claimed = (s >> 31) != 0u;
      }
      R.row_ec[r] = id;
      if (id != ECB_NONE && atomicExch(&R.seen[id], R.tag) == R.tag) ecr_flag(R.ctr, ECR_BAD_DUPLICATE, r);
      if (claimed) len = (u32)(R.indptr[r + 1] - R.indptr[r]);
    }
    const u32 off = harvest_block_reserve(R.ctr, len, s_scan);
    if (r < R.n_rows) R.row_dst[r] = claimed ? off : ECB_NONE;
    if (claimed) {
      row_off[id] = off;
      row_len[id] = len;
    }
  }
}

__global__ void __launch_bounds__(ECR_THREADS) ecb_ecr_copy_kernel(const EcrParams R, uint2* arena) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < R.nnz; i += gridDim.x * blockDim.x) {
    const u32 r = ecr_row_of(R.indptr, R.n_rows, i);
    const u32 dst = R.row_dst[r];
    if (dst != ECB_NONE) arena[(size_t)dst + (i - (u32)R.indptr[r])] = make_uint2((u32)R.indices[i], (u32)R.data[i]);
  }
}

__global__ void __launch_bounds__(ECR_THREADS) ecb_ecr_check_kernel(const EcrParams R, const u32* row_len,
                                                                    const u32* row_off, const uint2* arena) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < R.nnz; i += gridDim.x * blockDim.x) {
    const u32 r = ecr_row_of(R.indptr, R.n_rows, i);
    const u32 id = R.row_ec[r];
    if (R.row_dst[r] != ECB_NONE || id == ECB_NONE) continue;   // claimed here, or not in the table
    const u32 j = i - (u32)R.indptr[r];
    const u32 len = (u32)(R.indptr[r + 1] - R.indptr[r]);
    bool bad = row_len[id] != len;
    if (!bad) {
      const uint2 e = arena[(size_t)row_off[id] + j];
      bad = e.x != (u32)R.indices[i] || e.y != (u32)R.data[i];
    }
    if (bad) ecr_flag(R.ctr, ECR_BAD_COLLISION, r);
  }
}

// N entries of the append: flag[i] = 1 for a count > 0; the value checks.
__global__ void __launch_bounds__(ECR_THREADS) ecb_ecr_append_flags_kernel(const int32_t* n_indices, const int32_t* n_data,
                                                                           u32 nnz, u32 n_rows, u32* flag,
                                                                           EcbCounters* ctr) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += gridDim.x * blockDim.x) {
    const bool row_ok = (u32)n_indices[i] < n_rows;
    const int v = n_data[i];
    if (!row_ok) ecr_flag(ctr, ECR_BAD_N_INDEX, i);
    if (v < 0) ecr_flag(ctr, ECR_BAD_N_COUNT, i);
    flag[i] = row_ok && v > 0 ? 1u : 0u;
  }
}

// pos: the exclusive scan of the flags over nnz + 1 items.  Pairs in input order, and every column's count.
__global__ void __launch_bounds__(ECR_THREADS) ecb_ecr_append_pairs_kernel(const int32_t* n_indptr, u32 n_cols,
                                                                           const int32_t* n_indices,
                                                                           const int32_t* n_data, u32 nnz, u32 n_rows,
                                                                           const u32* pos, const u32* row_ec,
                                                                           uint2* pairs, u32* col_count) {
  const u32 stride = gridDim.x * blockDim.x;
  const u32 tid = blockIdx.x * blockDim.x + threadIdx.x;
  for (u32 i = tid; i < nnz; i += stride) {
    const int v = n_data[i];
    if ((u32)n_indices[i] < n_rows && v > 0) pairs[pos[i]] = make_uint2(row_ec[n_indices[i]], (u32)v);
  }
  for (u32 s = tid; s < n_cols; s += stride) col_count[s] = pos[n_indptr[s + 1]] - pos[n_indptr[s]];
}
