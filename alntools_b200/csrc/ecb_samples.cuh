// ecb_samples.cuh — per-sample counts of a single-sample context (ecb_sample_close / ecb_finalize_samples).
//
// Several files pushed one after the other into ONE single-sample context share its EC table, so EC identity, ids
// and the A matrix are those of the concatenated columns.  A file's reads per EC are the growth of the table's
// counts while the file was pushed: ecb_sample_close takes the difference of every EC's count against the count at
// the previous close and records the non-zero ones as (provisional id, delta) pairs.  The finalize maps the
// provisional ids to EC ids, sorts the pairs by (sample, EC id) and writes them as the columns of N (CSC).
#pragma once
#include "ecb_common.cuh"

// One thread per provisional id below n_ec.  Counts are read through ec_slot, which every rehash keeps current,
// after the pushes have completed (stream order), so growth and replay inside a sample need nothing here.  Ids at
// or above n_prev were claimed after the previous close: their count then was 0 and last_count holds nothing for
// them yet.  Pairs are appended with one
// atomic per warp; their order inside a sample does not matter (the finalize sorts them).
__global__ void __launch_bounds__(256) ecb_sample_close_kernel(const EcbEntry* __restrict__ table,
                                                               const u32* __restrict__ ec_slot, u32 n_ec, u32 n_prev,
                                                               u32* __restrict__ last_count, uint2* __restrict__ pairs,
                                                               u32* __restrict__ n_pairs) {
  const int lane = threadIdx.x & 31;
  const u32 stride = gridDim.x * blockDim.x;
  // every lane of a warp runs the same number of iterations, so the ballot below always sees the whole warp
  for (u32 base = blockIdx.x * blockDim.x; base < n_ec; base += stride) {
    const u32 e = base + threadIdx.x;
    u32 delta = 0;
    if (e < n_ec) {
      const u32 count = table[ec_slot[e]].countm1 + 1u;
      delta = count - (e < n_prev ? last_count[e] : 0u);
      last_count[e] = count;
    }
    const u32 m = __ballot_sync(ECB_FULL, delta != 0);
    if (!m) continue;
    u32 at = 0;
    if (lane == __ffs(m) - 1) at = atomicAdd(n_pairs, (u32)__popc(m));
    at = __shfl_sync(ECB_FULL, at, __ffs(m) - 1);
    if (delta) pairs[at + __popc(m & ((1u << lane) - 1u))] = make_uint2(e, delta);
  }
}

// Sort input: key = sample << ec_bits | EC id, value = reads.  A pair's sample is found in the column offsets
// (indptr[s] <= i < indptr[s + 1]; empty samples have equal offsets and are skipped by the search).
__global__ void __launch_bounds__(256) ecb_sample_keys_kernel(const uint2* __restrict__ pairs, u32 n,
                                                              const int32_t* __restrict__ indptr, u32 n_samples,
                                                              const u32* __restrict__ ecid_of, int ec_bits,
                                                              u64* __restrict__ keys, u32* __restrict__ vals) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    u32 lo = 0, hi = n_samples;   // largest s with indptr[s] <= i
    while (hi - lo > 1) {
      const u32 mid = (lo + hi) >> 1;
      if ((u32)indptr[mid] <= i) lo = mid; else hi = mid;
    }
    const uint2 p = pairs[i];
    keys[i] = ((u64)lo << ec_bits) | ecid_of[p.x];
    vals[i] = p.y;
  }
}

// Sorted pairs -> n_indices (EC ids, ascending inside a column) and n_data.
__global__ void __launch_bounds__(256) ecb_sample_csc_kernel(const u64* __restrict__ keys, const u32* __restrict__ vals,
                                                             u32 n, u64 ec_mask, int32_t* __restrict__ indices,
                                                             int32_t* __restrict__ data) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    indices[i] = (int32_t)(keys[i] & ec_mask);
    data[i] = (int32_t)vals[i];
  }
}
