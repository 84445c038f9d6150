// ecb_common.cuh — shared device types and primitives of libecb200 (sm_100a only).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

typedef unsigned int u32;
typedef unsigned long long u64;

#define ECB_FULL 0xFFFFFFFFu
#define ECB_MAX_PROBE 192
#define ECB_NONE 0xFFFFFFFFu

// Device allocation that only ever grows (host-side bookkeeping).
struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

// One slot of an open-addressing table in HBM.  32 bytes = one DRAM/L2 sector, so a probe touches
// exactly one sector.  memset(0xFF) is the empty state: key = all ones, first = +inf,
// countm1 = count - 1 (mod 2^32) = 0xFFFFFFFF <=> count 0, aux = ECB_NONE.
struct __align__(32) EcbEntry {
  u64 key_lo;
  u64 key_hi;
  u64 first;    // smallest global order key (order_base + offset of the read's first alignment)
  u32 countm1;  // number of reads - 1
  u32 aux;      // EC table: provisional (claim-order) EC id
};

struct Key128 {
  u64 lo, hi;
};

__host__ __device__ __forceinline__ bool key_eq(const Key128& a, const Key128& b) {
  return a.lo == b.lo && a.hi == b.hi;
}
__host__ __device__ __forceinline__ bool key_empty(const Key128& a) { return (a.lo & a.hi) == ~0ull; }

// 128-bit compare-and-swap in global memory (ATOMG.E.CAS.128 on sm_100a).
__device__ __forceinline__ Key128 atomic_cas128(void* addr, Key128 cmp, Key128 val) {
  Key128 old;
  asm volatile(
      "{\n\t.reg .b128 c, v, o;\n\t"
      "mov.b128 c, {%2, %3};\n\t"
      "mov.b128 v, {%4, %5};\n\t"
      "atom.global.cas.b128 o, [%6], c, v;\n\t"
      "mov.b128 {%0, %1}, o;\n\t}"
      : "=l"(old.lo), "=l"(old.hi)
      : "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi), "l"(addr)
      : "memory");
  return old;
}

// Whole-sector (256-bit) load of a table slot through L2 only (LDG.E.ENL2.256): slots are written by
// atomics from every SM, so L1 must not serve them.
__device__ __forceinline__ void load_entry_cg(const EcbEntry* e, Key128& key, u64& first, u32& countm1,
                                              u32& aux) {
  u64 w3;
  asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];"
               : "=l"(key.lo), "=l"(key.hi), "=l"(first), "=l"(w3)
               : "l"(e));
  countm1 = (u32)w3;
  aux = (u32)(w3 >> 32);
}

__host__ __device__ __forceinline__ u32 fmix32(u32 h) {
  h ^= h >> 16;
  h *= 0x85ebca6bu;
  h ^= h >> 13;
  h *= 0xc2b2ae35u;
  h ^= h >> 16;
  return h;
}

// Element code of one alignment: (main target, haplotype) packed in 31 bits.
__host__ __device__ __forceinline__ u32 ecb_code(int target, int hap) { return ((u32)target << 5) | (u32)hap; }

// 128-bit contribution of one DISTINCT (target, haplotype) element.  A read's key is the lane-wise
// sum (mod 2^32) of the contributions of its distinct elements: a commutative set hash, so no
// per-read sort is needed on the streaming path.  Word a is a bijective scramble g of the 31-bit code
// (multiply-add / xor-shift / multiply / xor-shift: distinct codes never share it and no code gives 0 - an
// element whose four words are all zero would vanish from every set that holds it); words b, c, d are
// multiply-folds of g by three constants (low ^ high half of the 64-bit product: not linear in g, so equal
// sums of g do not carry over to them).  12 instructions per element.  Measured on all 9.7 M pairs of 4400
// adjacent codes: every word collides as often as a random 32-bit function would (10.8-11.1 k against
// 10.9 k expected) and no two pairs share any 64-bit half.
struct Mix4 {
  u32 a, b, c, d;
};
// multiply-fold: low ^ high half of a 32x32 -> 64 bit product (one IMAD.WIDE + one LOP3)
__host__ __device__ __forceinline__ u32 mum32(u32 x, u32 k) {
  const u64 p = (u64)x * k;
  return (u32)p ^ (u32)(p >> 32);
}
__host__ __device__ __forceinline__ Mix4 ecb_mix(u32 code) {
  u32 g = code * 0x9E3779B1u + 0x80000000u;   // = (code + 2^31) * K: zero only for code 2^31, which no element has
  g ^= g >> 15;
  g *= 0x85EBCA77u;
  g ^= g >> 13;
  Mix4 m;
  m.a = g;
  m.b = mum32(g, 0xC2B2AE3Du);
  m.c = mum32(g, 0x27D4EB2Fu);
  m.d = mum32(g, 0x165667B1u);
  return m;
}
__host__ __device__ __forceinline__ void mix_add(Mix4& x, const Mix4& y) {
  x.a += y.a; x.b += y.b; x.c += y.c; x.d += y.d;
}
__host__ __device__ __forceinline__ Mix4 mix_zero() { return Mix4{0u, 0u, 0u, 0u}; }

__host__ __device__ __forceinline__ Key128 mix_to_key(const Mix4& m) {
  Key128 k;
  k.lo = ((u64)m.b << 32) | m.a;
  k.hi = ((u64)m.d << 32) | m.c;
  if (key_empty(k)) k.lo = 0;  // all-ones is the empty marker
  return k;
}
// Slot hash over all 128 key bits (EC keys are already uniform; (file, EC, cell) keys are not).
__device__ __forceinline__ u32 key_slot_hash(const Key128& k) {
  const u32 h = (u32)k.lo * 0x9e3779b1u ^ (u32)(k.lo >> 32) * 0x85ebca6bu ^ (u32)k.hi * 0xc2b2ae35u ^
                (u32)(k.hi >> 32) * 0x27d4eb2fu;
  return fmix32(h);
}

// Slot hash of the EC table: EC keys are sums of well-mixed words, two of them are enough.
__device__ __forceinline__ u32 ec_slot_hash(const Key128& k) { return (u32)k.lo ^ (u32)(k.hi >> 32); }

// Counters shared between kernels and the host (one small device struct per context).
struct EcbCounters {
  u32 n_ec;           // provisional EC ids handed out so far (== ECs in the table)
  u32 n_overflow;     // reads whose insert ran out of probes in the current push
  u32 n_long;         // new ECs whose representative read is longer than a warp (harvest)
  u32 error;          // sticky device-side error bits
  u64 n_reads;        // reads counted
  u32 n_triples;      // entries in the (file, EC, cell) table
  u32 n_triple_overflow;
  u32 n_spill;        // hot-cache entries parked because the table was too full
  u32 chunk_next;     // next unclaimed chunk of the grouping kernel (reset before every launch)
  u64 arena_used;     // (target, mask) pairs in the row arena
  u32 scratch[8];
  u32 n_deferred;     // reads of the current push longer than ECB_MAX_READ_ALIGNMENTS (ecb_longread.cuh)
  u32 n_deferred_fail;// ... of them that found the table too full (inserted again after a growth)
  u32 ecr_bad[8];     // EC rows: first bad entry / row of each kind (ecb_ecrows.cuh; ECB_NONE = none)
};

#define ECB_DEVERR_EC_CAPACITY 1u   // provisional id space exhausted
#define ECB_DEVERR_READ_TOO_LONG 2u
#define ECB_DEVERR_VALUE_RANGE 4u   // target/hap outside the declared bounds
#define ECB_DEVERR_VERIFY 8u        // key verification found a 128-bit hash collision
