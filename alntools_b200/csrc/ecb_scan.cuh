// ecb_scan.cuh — device-wide exclusive prefix sum over uint32 in ONE launch (decoupled look-back).  Used
// for EC ranking (popcounts of the first-occurrence bitmap), CSR row offsets and stream compaction.
//
// Every CTA draws its tile from an atomic ticket (not blockIdx), scans the tile, publishes the tile's
// aggregate in a status word, and one warp walks back over the status words of the tiles before it until it
// meets an inclusive prefix.  A tile only ever waits on tiles whose CTAs have already started, so progress
// does not depend on the order in which CTAs are scheduled.  The state (ticket + one status word per tile)
// is cleared by a stream-ordered memset before each launch.  Status word: bits 63..62 the flag (0 not yet
// published, 1 aggregate, 2 inclusive prefix), bits 61..0 the value; a tile's aggregate is the u32 sum of its
// items (as the sums were before), prefixes are u64.
#pragma once
#include "ecb_common.cuh"

#define SCAN_THREADS 256
#define SCAN_ITEMS 16
#define SCAN_BLOCK (SCAN_THREADS * SCAN_ITEMS)

__device__ __forceinline__ u32 warp_incl_scan_u32(u32 v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    u32 o = __shfl_up_sync(ECB_FULL, v, d);
    if (lane >= d) v += o;
  }
  return v;
}

__device__ __forceinline__ u64 warp_incl_scan_u64(u64 v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    u64 o = __shfl_up_sync(ECB_FULL, v, d);
    if (lane >= d) v += o;
  }
  return v;
}

// Exclusive scan of one value per thread across a 256-thread CTA; returns the exclusive prefix and
// the CTA total.  `smem` needs 9 u32.
__device__ __forceinline__ u32 block_excl_scan_u32(u32 v, u32* smem, u32& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  u32 inc = warp_incl_scan_u32(v, lane);
  if (lane == 31) smem[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    u32 w = lane < (SCAN_THREADS / 32) ? smem[lane] : 0u;
    u32 winc = warp_incl_scan_u32(w, lane);
    if (lane < (SCAN_THREADS / 32)) smem[lane] = winc - w;
    if (lane == (SCAN_THREADS / 32) - 1) smem[8] = winc;
  }
  __syncthreads();
  u32 res = smem[warp] + inc - v;
  total = smem[8];
  __syncthreads();
  return res;
}

#define SCAN_FLAG_AGG (1ull << 62)
#define SCAN_FLAG_INC (2ull << 62)
#define SCAN_VALUE_MASK ((1ull << 62) - 1ull)

// Scan state: word 0 the tile ticket, words 1..n_tiles the status words, word n_tiles + 1 the total.
__device__ __forceinline__ u32 scan_take_tile(u64* state, u32* s_tile) {
  if (threadIdx.x == 0) *s_tile = atomicAdd((unsigned int*)state, 1u);
  __syncthreads();
  return *s_tile;
}

// Called by ONE whole warp: publishes the tile's aggregate, looks back for the exclusive prefix of the tile,
// publishes the inclusive prefix and returns the exclusive one (on every lane).
__device__ __forceinline__ u64 scan_lookback(u64* state, u32 tile, u64 aggregate) {
  volatile u64* status = (volatile u64*)(state + 1);
  const int lane = threadIdx.x & 31;
  if (tile == 0) {
    if (lane == 0) status[0] = SCAN_FLAG_INC | aggregate;
    return 0;
  }
  if (lane == 0) status[tile] = SCAN_FLAG_AGG | aggregate;
  u64 excl = 0;
  long long top = (long long)tile - 1;   // the 32 tiles top, top-1, ... are looked at together
  while (true) {
    const long long idx = top - lane;
    u64 s;
    do {
      s = idx >= 0 ? status[idx] : SCAN_FLAG_INC;
    } while (__any_sync(ECB_FULL, (s >> 62) == 0ull));
    const u32 inc = __ballot_sync(ECB_FULL, (s >> 62) == 2ull);
    const int stop = inc ? __ffs(inc) - 1 : 31;   // the nearest tile with an inclusive prefix ends the walk
    u64 v = lane <= stop ? (s & SCAN_VALUE_MASK) : 0ull;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(ECB_FULL, v, d);
    excl += v;
    if (inc) break;
    top -= 32;
  }
  if (lane == 0) status[tile] = SCAN_FLAG_INC | ((excl + aggregate) & SCAN_VALUE_MASK);
  return excl;
}

// in may be a u32 array (POPC=false) or a bitmap whose popcounts are scanned (POPC=true); in may alias out.
// The last tile writes the total to state[n_tiles + 1].
template <bool POPC>
__global__ void __launch_bounds__(SCAN_THREADS) scan_kernel(const u32* in, u64 n, u32* out, u32 base_offset,
                                                            u64* __restrict__ state, u32 n_tiles) {
  __shared__ u32 sm[9];
  __shared__ u32 s_tile;
  __shared__ u64 s_prefix;
  const u32 tile = scan_take_tile(state, &s_tile);
  // blocked arrangement: thread t owns SCAN_ITEMS consecutive elements
  const u64 base = (u64)tile * SCAN_BLOCK + (u64)threadIdx.x * SCAN_ITEMS;
  u32 v[SCAN_ITEMS];
  u32 s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    u64 idx = base + i;
    u32 x = 0;
    if (idx < n) {
      x = in[idx];
      if (POPC) x = (u32)__popc(x);
    }
    v[i] = x;
    s += x;
  }
  u32 total;
  u32 excl = block_excl_scan_u32(s, sm, total);
  if (threadIdx.x < 32) {
    const u64 p = scan_lookback(state, tile, total);
    if (threadIdx.x == 0) {
      s_prefix = p;
      if (tile == n_tiles - 1) state[n_tiles + 1] = p + total;
    }
  }
  __syncthreads();
  u32 run = base_offset + (u32)s_prefix + excl;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    u64 idx = base + i;
    if (idx < n) out[idx] = run;
    run += v[i];
  }
}
