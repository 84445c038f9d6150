// ecb_harvest.cuh — turn one read of every NEW equivalence class into its canonical row: distinct main
// targets ascending, data = OR of (1 << haplotype).
//
// Replaces alntools/bam_utils.py:788-825 (EC key -> per-haplotype (ec, target) COO lists) and the
// canonicalisation scipy performs in alntools/bin_utils.py:208-211 (sum of 2^h * data[h], tocsr()
// with sorted column indices).  Runs right after the grouping kernel of every push (and once more after a
// replay, over the ECs the replay claimed), while the caller's columns are still valid, over the ECs claimed
// in that push only (E rows, not R reads).  The grouping kernel recorded
// for every new EC the offset and the length of one read with that key.  A row's place in the arena is
// reserved when its length is known, with one atomic per warp (short reads) or per row (the rare long
// ones) on the arena cursor: no scan, no host round trip; the host only provides room for one row entry
// per alignment of the push, which is an upper bound.
//   k <= 8        one thread per EC: 8-element sorting network in registers
//   8 < k <= 32   one warp per EC: __match_any_sync / __reduce_or_sync, rank by counting
//   32 < k <= 1024  one warp per EC: warp-synchronous bitonic sort in shared memory (no CTA barrier)
//   k > 1024      one CTA per EC: bitonic sort in shared memory (up to ECB_MAX_READ_ALIGNMENTS)
#pragma once
#include "ecb_common.cuh"
#include "ecb_scan.cuh"

struct HarvestParams {
  const int32_t* rg;
  const int32_t* tg;
  const int32_t* hp;
  int n;
  const u32* ec_rep;
  const u32* ec_len;
  u32 e0;            // first provisional id to harvest; the range ends at ctr->n_ec, read on the device, so
                     // the harvest is launched right after the grouping kernel without a host round trip
  u32* row_len;      // [capacity] out: row length
  u32* row_off;      // [capacity] out: absolute offset inside the arena (reserved here)
  uint2* arena;      // (target, mask) pairs
  int n_targets, n_haps;  // bounds of the column values (checked here, off the streaming path)
  u32* long_list;    // provisional ids whose read has more than 32 alignments
  u32* mid_list;     // provisional ids whose read has 9..32 alignments
  u32* big_list;     // provisional ids whose read has 33..HARVEST_WSORT_MAX alignments
  EcbCounters* ctr;  // scratch[1] = #ECs with 8 < k <= 32, scratch[3] = #ECs with 32 < k <= HARVEST_WSORT_MAX,
                     // n_long = #ECs with more; arena_used = the arena cursor
};

// Reserve `cnt` arena entries for every thread of the (fully converged) 256-thread CTA: ONE atomic per CTA
// (all reservations hit the same cursor; one per warp - 127 k for 4 M ECs - serialise at the L2 and were
// measured to cost more than the scan they replaced).  `smem` needs 10 u32.
__device__ __forceinline__ u32 harvest_block_reserve(EcbCounters* ctr, u32 cnt, u32* smem) {
  u32 total;
  const u32 excl = block_excl_scan_u32(cnt, smem, total);
  if (threadIdx.x == 0) smem[9] = total ? (u32)atomicAdd((unsigned long long*)&ctr->arena_used, (unsigned long long)total) : 0u;
  __syncthreads();
  const u32 base = smem[9];
  __syncthreads();
  return base + excl;
}
#define HARVEST_LONG_MAX 16384
#define HARVEST_WSORT_MAX 1024   // longest read whose row one warp sorts on its own

#define ECB_CSWAP(a, b)            \
  {                                \
    const u32 lo_ = min(a, b);     \
    const u32 hi_ = max(a, b);     \
    a = lo_;                       \
    b = hi_;                       \
  }

// Append `item` to list[] for the lanes where `take` holds: one atomic per warp.
__device__ __forceinline__ void warp_append(u32* list, u32* counter, bool take, u32 item) {
  const u32 act = __activemask();
  const u32 m = __ballot_sync(act, take);
  if (!m) return;
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(m) - 1;
  u32 base = 0;
  if (lane == leader) base = atomicAdd(counter, (u32)__popc(m));
  base = __shfl_sync(act, base, leader);
  if (take) list[base + (u32)__popc(m & ((1u << lane) - 1u))] = item;
}

__global__ void __launch_bounds__(256) ecb_harvest_short_kernel(const HarvestParams P) {
  // whole CTAs walk the id range together (the reservation below is a CTA-wide step)
  __shared__ u32 s_scan[10];
  const u32 n_new = P.ctr->n_ec - P.e0;   // (the ECs before e0 are never handed out again)
  const u32 stride = gridDim.x * blockDim.x;
  for (u32 i0 = blockIdx.x * blockDim.x; i0 < n_new; i0 += stride) {
    const u32 i = i0 + threadIdx.x;
    const bool in = i < n_new;
    const u32 e = P.e0 + (in ? i : 0u);
    const u32 k = in ? P.ec_len[e] : 0u;
    warp_append(P.mid_list, &P.ctr->scratch[1], in && k > 8 && k <= 32, e);
    warp_append(P.big_list, &P.ctr->scratch[3], in && k > 32 && k <= HARVEST_WSORT_MAX, e);
    // ECs first met in a read longer than HARVEST_LONG_MAX get their rows from the long-read pass
    // (ecb_longread.cuh); the grouping kernel has checked every read against the limit
    const bool deferred = in && k > HARVEST_LONG_MAX;
    if (in && k > HARVEST_WSORT_MAX && !deferred) P.long_list[atomicAdd(&P.ctr->n_long, 1u)] = e;
    const bool mine = in && k <= 8;
    const int s = (int)(mine ? P.ec_rep[e] : 0u);
    u32 c[8];
    bool bad = false;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      c[j] = 0xFFFFFFFFu;
      if (mine && (u32)j < k) {
        const int t = P.tg[s + j], h = P.hp[s + j];
        bad |= (u32)t >= (u32)P.n_targets || (u32)h >= (u32)P.n_haps;
        c[j] = ecb_code(t, h);
      }
    }
    if (bad) atomicOr(&P.ctr->error, ECB_DEVERR_VALUE_RANGE);
    // Batcher odd-even merge sort network for 8 keys (19 comparators)
    ECB_CSWAP(c[0], c[1]) ECB_CSWAP(c[2], c[3]) ECB_CSWAP(c[4], c[5]) ECB_CSWAP(c[6], c[7])
    ECB_CSWAP(c[0], c[2]) ECB_CSWAP(c[1], c[3]) ECB_CSWAP(c[4], c[6]) ECB_CSWAP(c[5], c[7])
    ECB_CSWAP(c[1], c[2]) ECB_CSWAP(c[5], c[6])
    ECB_CSWAP(c[0], c[4]) ECB_CSWAP(c[1], c[5]) ECB_CSWAP(c[2], c[6]) ECB_CSWAP(c[3], c[7])
    ECB_CSWAP(c[2], c[4]) ECB_CSWAP(c[3], c[5])
    ECB_CSWAP(c[1], c[2]) ECB_CSWAP(c[3], c[4]) ECB_CSWAP(c[5], c[6])
    // row length = distinct targets; then the row goes to the place reserved for it
    u32 cnt = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (c[j] != 0xFFFFFFFFu && (j == 0 || (c[j] >> 5) != (c[j - 1] >> 5))) ++cnt;
    // the rows of longer reads are built by the kernels below; their place is reserved HERE, with the read
    // length as the upper bound of the row length (rows need not be packed: row_off / row_len index them),
    // so those kernels need no reservation of their own - one atomic per EC on the arena cursor was most of
    // their time on heavily multimapping input
    const u32 want = mine ? cnt : (in && !deferred ? k : 0u);
    const u32 off = harvest_block_reserve(P.ctr, want, s_scan);
    if (in && !mine && !deferred) P.row_off[e] = off;
    if (!mine) continue;
    uint2* out = P.arena + off;
    u32 w = 0, prev_t = 0xFFFFFFFFu, mask = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (c[j] != 0xFFFFFFFFu) {
        const u32 t = c[j] >> 5;
        if (t != prev_t) {
          if (w) out[w - 1] = make_uint2(prev_t, mask);
          ++w;
          prev_t = t;
          mask = 0;
        }
        mask |= 1u << (c[j] & 31u);
      }
    }
    if (w) out[w - 1] = make_uint2(prev_t, mask);
    P.row_len[e] = cnt;
    P.row_off[e] = off;
  }
}

// Rows of reads with 9..32 alignments (listed by the short kernel): one warp per EC, one alignment per lane.
// The 32 element codes are sorted in registers (bitonic network over shuffles, 15 compare-exchange steps), the
// haplotype bits of equal targets are OR-ed with a segmented suffix scan, and the first lane of every run
// writes its (target, mask) at the run's rank.  (A first version grouped the lanes with match_any and reduced
// every group with its own mask: both serialise over the distinct values - 3.4 ms for 4 M such reads.)
__global__ void __launch_bounds__(256) ecb_harvest_warp_kernel(const HarvestParams P) {
  const u32 n_mid = P.ctr->scratch[1];   // listed by the short kernel (same stream, earlier launch)
  const int lane = threadIdx.x & 31;
  const u32 lt = (1u << lane) - 1u;
  const u32 warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const u32 n_warps = (gridDim.x * blockDim.x) >> 5;
  // Every EC costs a chain of dependent loads (list -> start / length / row place -> codes) that is far longer
  // than the sort: the chain of the NEXT two ECs is in flight while the current one is sorted.
  auto load_code = [&](u32 e, int& k_out, u32& off_out) -> u32 {
    const int k = (int)P.ec_len[e];
    const int s = (int)P.ec_rep[e];
    k_out = k;
    off_out = P.row_off[e];   // reserved by the short kernel
    u32 c = 0xFFFFFFFFu;      // lanes beyond the read sort to the end
    if (lane < k) {
      const int t = P.tg[s + lane], h = P.hp[s + lane];
      if ((u32)t >= (u32)P.n_targets || (u32)h >= (u32)P.n_haps) atomicOr(&P.ctr->error, ECB_DEVERR_VALUE_RANGE);
      c = ecb_code(t, h);
    }
    return c;
  };
  u32 e_cur = warp_global < n_mid ? P.mid_list[warp_global] : 0u;
  u32 e_nxt = warp_global + n_warps < n_mid ? P.mid_list[warp_global + n_warps] : 0u;
  int k_cur = 0;
  u32 off_cur = 0;
  u32 c_cur = warp_global < n_mid ? load_code(e_cur, k_cur, off_cur) : 0xFFFFFFFFu;
  for (u32 i = warp_global; i < n_mid; i += n_warps) {
    const u32 e = e_cur, off = off_cur;
    u32 c = c_cur;
    // the next EC's codes and the list entry after it
    const u32 e_nn = i + 2 * n_warps < n_mid ? P.mid_list[i + 2 * n_warps] : 0u;
    if (i + n_warps < n_mid) c_cur = load_code(e_nxt, k_cur, off_cur);
    e_cur = e_nxt;
    e_nxt = e_nn;
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        const u32 o = __shfl_xor_sync(ECB_FULL, c, stride);
        const bool keep_min = ((lane & size) == 0) == ((lane & stride) == 0);
        c = keep_min ? min(c, o) : max(c, o);
      }
    }
    const bool valid = c != 0xFFFFFFFFu;
    const u32 t = c >> 5;
    const u32 prev = __shfl_up_sync(ECB_FULL, c, 1);
    const bool head = lane == 0 || (prev >> 5) != t;            // (the first lane beyond the read is one too)
    const u32 heads = __ballot_sync(ECB_FULL, head);
    u32 m = valid ? (1u << (c & 31u)) : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {                           // OR over the rest of the run
      const u32 o = __shfl_down_sync(ECB_FULL, m, d);
      if (lane + d < 32 && ((heads >> (lane + 1)) & ((1u << d) - 1u)) == 0u) m |= o;
    }
    const u32 vheads = heads & __ballot_sync(ECB_FULL, valid);
    if (head && valid) P.arena[(size_t)off + __popc(vheads & lt)] = make_uint2(t, m);
    if (lane == 0) P.row_len[e] = (u32)__popc(vheads);
  }
}

// Bitonic sort of 32 * R values held R per lane (value i of the sequence = register i / 32 of lane i % 32):
// compare-exchange steps with a stride below 32 are shuffles, the others stay inside the lane.  For 64 and 128
// values this takes about 40 % of the instructions of the shared-memory network below.
template <int R>
__device__ __forceinline__ void harvest_sort_regs(u32 (&v)[R], int lane) {
#pragma unroll
  for (int size = 2; size <= 32 * R; size <<= 1) {
#pragma unroll
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      if (stride >= 32) {
        const int sr = stride >> 5;
#pragma unroll
        for (int r = 0; r < R; ++r) {
          if (r & sr) continue;
          const bool up = ((r << 5) & size) == 0;
          const u32 lo = min(v[r], v[r | sr]), hi = max(v[r], v[r | sr]);
          v[r] = up ? lo : hi;
          v[r | sr] = up ? hi : lo;
        }
      } else {
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const u32 o = __shfl_xor_sync(ECB_FULL, v[r], stride);
          const bool up = (((r << 5) | lane) & size) == 0;
          const bool keep_min = up == ((lane & stride) == 0);
          v[r] = keep_min ? min(v[r], o) : max(v[r], o);
        }
      }
    }
  }
}

// Rows of reads with 33..HARVEST_WSORT_MAX alignments (heavy multimapping): one WARP per EC.  The
// element codes are sorted with a bitonic network in the warp's own slice of shared memory, so the only
// synchronisation is __syncwarp; then one entry per distinct target.
__global__ void __launch_bounds__(256) ecb_harvest_wsort_kernel(const HarvestParams P) {
  const u32 n_big = P.ctr->scratch[3];
  extern __shared__ u32 sm_all[];
  const int lane = threadIdx.x & 31;
  u32* codes = sm_all + (threadIdx.x >> 5) * HARVEST_WSORT_MAX;
  const u32 warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const u32 n_warps = (gridDim.x * blockDim.x) >> 5;
  const u32 lt = (1u << lane) - 1u;
  // the list entry and the start / length / row place of the NEXT ECs are fetched while the current one is sorted
  u32 e_cur = warp_global < n_big ? P.big_list[warp_global] : 0u;
  u32 e_nxt = warp_global + n_warps < n_big ? P.big_list[warp_global + n_warps] : 0u;
  int s_cur = 0;
  u32 k_cur = 0, off_cur = 0;
  if (warp_global < n_big) {
    s_cur = (int)P.ec_rep[e_cur];
    k_cur = P.ec_len[e_cur];
    off_cur = P.row_off[e_cur];
  }
  for (u32 li = warp_global; li < n_big; li += n_warps) {
    const u32 e = e_cur, k = k_cur, off = off_cur;
    const int s = s_cur;
    const u32 e_nn = li + 2 * n_warps < n_big ? P.big_list[li + 2 * n_warps] : 0u;
    if (li + n_warps < n_big) {
      s_cur = (int)P.ec_rep[e_nxt];
      k_cur = P.ec_len[e_nxt];
      off_cur = P.row_off[e_nxt];
    }
    e_cur = e_nxt;
    e_nxt = e_nn;
    u32 np2 = 64;
    while (np2 < k) np2 <<= 1;
    bool bad = false;
    for (u32 i = lane; i < np2; i += 32) {
      u32 code = 0xFFFFFFFFu;
      if (i < k) {
        const int t = P.tg[s + i], h = P.hp[s + i];
        bad |= (u32)t >= (u32)P.n_targets || (u32)h >= (u32)P.n_haps;
        code = ecb_code(t, h);
      }
      codes[i] = code;
    }
    if (bad) atomicOr(&P.ctr->error, ECB_DEVERR_VALUE_RANGE);
    __syncwarp();
    if (np2 == 64u) {          // up to 128 codes are sorted in registers and go back sorted
      u32 v[2] = {codes[lane], codes[32 + lane]};
      harvest_sort_regs<2>(v, lane);
      codes[lane] = v[0];
      codes[32 + lane] = v[1];
      __syncwarp();
    } else if (np2 == 128u) {
      u32 v[4] = {codes[lane], codes[32 + lane], codes[64 + lane], codes[96 + lane]};
      harvest_sort_regs<4>(v, lane);
      codes[lane] = v[0];
      codes[32 + lane] = v[1];
      codes[64 + lane] = v[2];
      codes[96 + lane] = v[3];
      __syncwarp();
    } else
    for (u32 size = 2; size <= np2; size <<= 1) {
      for (u32 stride = size >> 1; stride > 0; stride >>= 1) {
        for (u32 i = lane; i < (np2 >> 1); i += 32) {
          const u32 lo = 2 * i - (i & (stride - 1));
          const u32 hi = lo + stride;
          const bool up = (lo & size) == 0;
          const u32 a = codes[lo], b = codes[hi];
          if ((a > b) == up) {
            codes[lo] = b;
            codes[hi] = a;
          }
        }
        __syncwarp();
      }
    }
    uint2* out = P.arena + (size_t)off;
    u32 run = 0;
    for (u32 base = 0; base < k; base += 32) {
      const u32 i = base + lane;
      u32 code = 0xFFFFFFFFu;
      bool start = false;
      if (i < k) {
        code = codes[i];
        start = (i == 0) || ((codes[i - 1] >> 5) != (code >> 5));
      }
      const u32 m = __ballot_sync(ECB_FULL, start);
      if (start) {
        u32 mask = 0;
        for (u32 j = i; j < k && (codes[j] >> 5) == (code >> 5); ++j) mask |= 1u << (codes[j] & 31u);
        out[run + (u32)__popc(m & lt)] = make_uint2(code >> 5, mask);
      }
      run += (u32)__popc(m);
    }
    if (lane == 0) P.row_len[e] = run;
    __syncwarp();
  }
}

// Rows of long reads (HARVEST_WSORT_MAX+1 .. HARVEST_LONG_MAX alignments): one CTA per EC, bitonic sort of the element
// codes in shared memory, then one entry per distinct target.
__global__ void __launch_bounds__(256) ecb_harvest_long_kernel(const HarvestParams P) {
  const u32 n_long = P.ctr->n_long;
  extern __shared__ u32 sm_codes[];
  __shared__ u32 s_scan[9];
  __shared__ u32 s_run;
  __shared__ u32 s_off;
  for (u32 li = blockIdx.x; li < n_long; li += gridDim.x) {
    const u32 e = P.long_list[li];
    const int s = (int)P.ec_rep[e];
    const u32 k = min(P.ec_len[e], (u32)HARVEST_LONG_MAX);
    u32 np2 = 64;
    while (np2 < k) np2 <<= 1;
    for (u32 i = threadIdx.x; i < np2; i += blockDim.x) {
      u32 code = 0xFFFFFFFFu;
      if (i < k) {
        const int t = P.tg[s + i], h = P.hp[s + i];
        if ((u32)t >= (u32)P.n_targets || (u32)h >= (u32)P.n_haps) atomicOr(&P.ctr->error, ECB_DEVERR_VALUE_RANGE);
        code = ecb_code(t, h);
      }
      sm_codes[i] = code;
    }
    __syncthreads();
    for (u32 size = 2; size <= np2; size <<= 1) {
      for (u32 stride = size >> 1; stride > 0; stride >>= 1) {
        for (u32 i = threadIdx.x; i < (np2 >> 1); i += blockDim.x) {
          const u32 lo = 2 * i - (i & (stride - 1));
          const u32 hi = lo + stride;
          const bool up = (lo & size) == 0;
          const u32 a = sm_codes[lo], b = sm_codes[hi];
          if ((a > b) == up) {
            sm_codes[lo] = b;
            sm_codes[hi] = a;
          }
        }
        __syncthreads();
      }
    }
    if (threadIdx.x == 0) {
      s_run = 0;
      s_off = P.row_off[e];   // reserved by the short kernel
    }
    __syncthreads();
    const size_t out0 = (size_t)s_off;
    for (u32 base = 0; base < k; base += blockDim.x) {
      const u32 i = base + threadIdx.x;
      bool start = false;
      u32 code = 0xFFFFFFFFu;
      if (i < k) {
        code = sm_codes[i];
        start = (i == 0) || ((sm_codes[i - 1] >> 5) != (code >> 5));
      }
      u32 total;
      const u32 excl = block_excl_scan_u32(start ? 1u : 0u, s_scan, total);
      if (start) {
        u32 mask = 0;
        for (u32 j = i; j < k && (sm_codes[j] >> 5) == (code >> 5); ++j) mask |= 1u << (sm_codes[j] & 31u);
        P.arena[out0 + s_run + excl] = make_uint2(code >> 5, mask);
      }
      __syncthreads();
      if (threadIdx.x == 0) s_run += total;
      __syncthreads();
    }
    if (threadIdx.x == 0) P.row_len[e] = s_run;
    __syncthreads();
  }
}
