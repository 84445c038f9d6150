// ecb_group.cuh — the grouping + hash-insert kernel (the hot path), the overflow replay kernel and
// the table rehash kernels.
//
// What it replaces: alntools/bam_utils.py:258-344 (per-alignment loop: group consecutive alignments
// by read, collapse duplicate tids, ec[key] += 1) and the ordering half of :680-698 (EC id = rank of
// the key's first occurrence), on int32 columns.
//
// Shape of the kernel (HBM-bound integer work, no tensor cores; after the column stream the binding
// resources are the latency of the random table sectors and the dependent chains inside a window):
//   * one persistent CTA per SM (grid = 148), 32 warps; every WARP walks chunks of the alignment
//     stream on its own — no CTA-wide barrier, no cross-warp carry;
//   * a warp looks at a WINDOW of 32 consecutive alignments (lane = alignment) that always starts at
//     a read start.  One ballot of the read_group changes gives every lane its read start (positions
//     beyond the push hold a sentinel), duplicate (target, haplotype) pairs inside a read are found
//     with shuffled compares (match_any only for windows with reads longer than 8), a segmented
//     shuffle scan with only ceil(log2(longest read in the window)) steps adds the 128-bit element
//     mixes of a read (commutative set hash -> no per-read sort).  The window then advances to its
//     last read start, so no read ever straddles two windows; the columns of the next window are
//     requested before the current one is inserted and the lines further ahead are pulled into L2 by
//     prefetches.  Reads that fill a whole window take a warp-cooperative path;
//   * a read is owned by the chunk it STARTS in (chunks are handed out by a global counter); the
//     owner runs past the chunk end until the read closes;
//   * closed reads first try the per-CTA shared-memory cache of hot ECs (4096 entries, lock-free hit
//     path, keys admitted on their second miss).  Misses are parked in a per-warp shared-memory queue
//     - with an L2 prefetch of their table sector - and inserted into the HBM table 64 at a time, two
//     per lane: one 256-bit sector load per probe, a 128-bit atomicCAS only when the slot looks empty,
//     RED.ADD on the count and atomicMin on the first-occurrence key only when it can lower it.  The
//     first load and the first CAS of both reads of a lane are in flight together: a warp pays for the
//     slowest lane's chain of round trips once per batch.  The cache is flushed when the CTA is done.
#pragma once
#include <cstddef>
#include "ecb_common.cuh"

#define ECB_GWARPS 32                  // warps per CTA of the grouping kernel
#define ECB_GTHREADS (32 * ECB_GWARPS)
#ifndef ECB_SHUFFLE_DEDUP
#define ECB_SHUFFLE_DEDUP 1
#endif
#ifndef ECB_ADMIT_SECOND
#define ECB_ADMIT_SECOND 1             // a key enters the hot-EC cache on its second miss in the CTA
#endif
#define ECB_SEEN_WORDS 2048            // 64 Kbit "missed once already" filter per CTA
#ifndef ECB_CACHE
#define ECB_CACHE 4096                 // per-CTA hot-EC cache entries
#endif
#define ECB_MQ 96                      // per-warp miss queue (entries); 64 are inserted at a time, two per lane
#ifndef ECB_PF_DIST
#define ECB_PF_DIST 256                // L2 prefetch distance of the column stream (alignments)
#endif

// A hot-cache entry that could not be flushed because the table was too full (replayed after growth).
struct EcbSpill {
  u64 lo, hi;
  u32 count, first, rep, len;
};

struct GroupParams {
  const int32_t* rg;
  const int32_t* tg;
  const int32_t* hp;
  const int32_t* cell;
  int n;           // alignments in this push
  int chunk_len;   // alignments per work chunk, multiple of 32
  u64 order_base;
  int drop_last;
  int use_cache;
  int n_targets;
  int n_haps;
  EcbEntry* table;
  u32 mask;
  u32* ec_slot;    // [capacity] provisional id -> table slot
  u32* ec_rep;     // [capacity] provisional id -> offset (in this push) of a read with that key
  u32* ec_len;     // [capacity] provisional id -> number of alignments of that read
  EcbCounters* ctr;
  u32* overflow_bits;  // [ceil(n/32)] reads that must be replayed after a table growth
  EcbSpill* spill;     // [grid * ECB_CACHE] cache entries that must be replayed after a table growth
  EcbEntry* ttable;    // (file, EC slot, cell) table, with cells only
  u32 tmask;
  u32 push_id;
  int max_read;        // longest read accepted (ECB_OPT_MAX_READ)
  uint2* deferred;     // [ctr->n_deferred] (offset, length) of the reads longer than ECB_MAX_READ_ALIGNMENTS
};

// Probe for `key` from `slot` on (linear probing, at most max_probe slots): find it or claim the
// first empty slot.  Returns the slot or ECB_NONE; first_seen = the entry's `first` as loaded (+inf
// when unknown/new).
__device__ __forceinline__ u32 table_probe_from(EcbEntry* table, u32 mask, const Key128& key, u32 slot,
                                                int max_probe, bool& claimed, u64& first_seen) {
  for (int p = 0; p < max_probe; ++p) {
    EcbEntry* e = table + slot;
    Key128 k;
    u64 first;
    u32 cm1, aux;
    load_entry_cg(e, k, first, cm1, aux);
    if (key_eq(k, key)) {
      first_seen = first;
      return slot;
    }
    if (key_empty(k)) {
      Key128 old = atomic_cas128(e, Key128{~0ull, ~0ull}, key);
      if (key_empty(old)) {
        claimed = true;
        return slot;
      }
      if (key_eq(old, key)) return slot;
    }
    slot = (slot + 1) & mask;
  }
  return ECB_NONE;
}


// Find `key` or claim an empty slot for it.  EC selects the EC table's slot hash.
template <bool EC = false>
__device__ __forceinline__ u32 table_find_or_claim(EcbEntry* table, u32 mask, const Key128& key,
                                                   bool& claimed, u64& first_seen) {
  claimed = false;
  first_seen = ~0ull;
  const u32 slot = (EC ? ec_slot_hash(key) : key_slot_hash(key)) & mask;
  return table_probe_from(table, mask, key, slot, ECB_MAX_PROBE, claimed, first_seen);
}

// Lookup only (no claim); ECB_NONE if absent.
__device__ __forceinline__ u32 table_find(const EcbEntry* table, u32 mask, const Key128& key) {
  u32 slot = key_slot_hash(key) & mask;
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

__device__ __forceinline__ Key128 triple_key(u32 slot, u32 cell, u32 push_id) {
  return Key128{((u64)slot << 32) | cell, (u64)push_id};
}

// Insert `count` occurrences of (file, EC, cell).  The triple table is sized by the host so that it
// cannot fill up; running out of probes is reported as a device error.
__device__ __forceinline__ void triple_upsert(const GroupParams& P, u32 slot, u32 cell, u64 pos) {
  bool claimed;
  u64 first_seen;
  if ((int)cell < 0) {
    atomicOr(&P.ctr->error, ECB_DEVERR_VALUE_RANGE);
    return;
  }
  u32 ts = table_find_or_claim(P.ttable, P.tmask, triple_key(slot, cell, P.push_id), claimed, first_seen);
  if (ts == ECB_NONE) {
    atomicAdd(&P.ctr->n_triple_overflow, 1u);
    return;
  }
  EcbEntry* te = P.ttable + ts;
  atomicAdd(&te->countm1, 1u);
  if (pos < first_seen) atomicMin(&te->first, pos);
  if (claimed) atomicAdd(&P.ctr->n_triples, 1u);
}

// Provisional EC id for the lanes that just claimed a slot: one atomic per converged group of lanes.
__device__ __forceinline__ u32 alloc_ec_ids(EcbCounters* ctr, bool claimed) {
  const u32 act = __activemask();
  const u32 cm = __ballot_sync(act, claimed);
  if (!cm) return ECB_NONE;
  const int lane = threadIdx.x & 31;
  const int leader = __ffs(cm) - 1;
  u32 base = 0;
  if (lane == leader) base = atomicAdd(&ctr->n_ec, (u32)__popc(cm));
  base = __shfl_sync(act, base, leader);
  return claimed ? base + (u32)__popc(cm & ((1u << lane) - 1u)) : ECB_NONE;
}

// Add `count` reads with key `key` to the HBM table.  s/len describe one read with that key (used
// when the key is new).  Returns the slot or ECB_NONE when the table is too full (caller records it).
__device__ __forceinline__ u32 global_upsert(const GroupParams& P, const Key128& key, u32 count, u32 first_local,
                                             u32 s, u32 len) {
  bool claimed;
  u64 first_seen;
  const u32 slot = table_find_or_claim<true>(P.table, P.mask, key, claimed, first_seen);
  if (slot != ECB_NONE) {
    EcbEntry* e = P.table + slot;
    atomicAdd(&e->countm1, count);
    const u64 pos = P.order_base + first_local;
    if (pos < first_seen) atomicMin(&e->first, pos);
  }
  const u32 ecl = alloc_ec_ids(P.ctr, claimed);
  if (claimed) {
    P.table[slot].aux = ecl;
    P.ec_slot[ecl] = slot;
    P.ec_rep[ecl] = s;
    P.ec_len[ecl] = len;
  }
  return slot;
}

// Two reads per lane go into the HBM table together.  The probe sequences of a warp's lanes are
// chains of dependent round trips to L2/HBM and every lane waits for the slowest, so the first
// load and the first compare-and-swap of both reads are issued before either result is used: the
// warp pays the chain once for 64 reads.  Returns the slots (ECB_NONE: absent read or table full).
__device__ __forceinline__ void global_upsert2(const GroupParams& P, const Key128& keyA, u32 sA, u32 lenA, bool hasA,
                                               const Key128& keyB, u32 sB, u32 lenB, bool hasB, u32& slotA,
                                               u32& slotB) {
  const Key128 EMPTY{~0ull, ~0ull};
  const u32 hA = ec_slot_hash(keyA) & P.mask, hB = ec_slot_hash(keyB) & P.mask;
  Key128 kA = EMPTY, kB = EMPTY;
  u64 fA = ~0ull, fB = ~0ull;
  u32 cm1, aux;
  if (hasA) load_entry_cg(P.table + hA, kA, fA, cm1, aux);
  if (hasB) load_entry_cg(P.table + hB, kB, fB, cm1, aux);
  const bool eqA = hasA && key_eq(kA, keyA), eqB = hasB && key_eq(kB, keyB);
  const bool casA = hasA && !eqA && key_empty(kA), casB = hasB && !eqB && key_empty(kB);
  if (casA) kA = atomic_cas128(P.table + hA, EMPTY, keyA);
  if (casB) kB = atomic_cas128(P.table + hB, EMPTY, keyB);
  bool clA = casA && key_empty(kA), clB = casB && key_empty(kB);
  if (casA) fA = ~0ull;  // the loaded `first` belongs to the empty state
  if (casB) fB = ~0ull;
  slotA = (eqA || clA || (casA && key_eq(kA, keyA))) ? hA : ECB_NONE;
  slotB = (eqB || clB || (casB && key_eq(kB, keyB))) ? hB : ECB_NONE;
  if (hasA && slotA == ECB_NONE) {  // the home slot holds another key: walk on
    fA = ~0ull;
    slotA = table_probe_from(P.table, P.mask, keyA, (hA + 1) & P.mask, ECB_MAX_PROBE - 1, clA, fA);
  }
  if (hasB && slotB == ECB_NONE) {
    fB = ~0ull;
    slotB = table_probe_from(P.table, P.mask, keyB, (hB + 1) & P.mask, ECB_MAX_PROBE - 1, clB, fB);
  }
  if (slotA != ECB_NONE) {
    EcbEntry* e = P.table + slotA;
    atomicAdd(&e->countm1, 1u);
    const u64 pos = P.order_base + sA;
    if (pos < fA) atomicMin(&e->first, pos);
  }
  if (slotB != ECB_NONE) {
    EcbEntry* e = P.table + slotB;
    atomicAdd(&e->countm1, 1u);
    const u64 pos = P.order_base + sB;
    if (pos < fB) atomicMin(&e->first, pos);
  }
  // provisional ids of the new ECs: one atomic for both halves
  const u32 act = __activemask();
  const u32 mA = __ballot_sync(act, clA), mB = __ballot_sync(act, clB);
  if (mA | mB) {
    const int lane = threadIdx.x & 31;
    const int leader = __ffs(act) - 1;
    u32 base = 0;
    if (lane == leader) base = atomicAdd(&P.ctr->n_ec, (u32)(__popc(mA) + __popc(mB)));
    base = __shfl_sync(act, base, leader);
    const u32 lt = (1u << lane) - 1u;
    if (clA) {
      const u32 id = base + (u32)__popc(mA & lt);
      P.table[slotA].aux = id;
      P.ec_slot[id] = slotA;
      P.ec_rep[id] = sA;
      P.ec_len[id] = lenA;
    }
    if (clB) {
      const u32 id = base + (u32)__popc(mA) + (u32)__popc(mB & lt);
      P.table[slotB].aux = id;
      P.ec_slot[id] = slotB;
      P.ec_rep[id] = sB;
      P.ec_len[id] = lenB;
    }
  }
}

struct GroupSmem {
  // hot-EC cache of this CTA (direct mapped, first come first installed, flushed at the end)
  alignas(16) uint4 c_key[ECB_CACHE];  // all ones = empty; written once, by the lane that holds c_lock
  u32 c_lock[ECB_CACHE];               // 0 = free, 1 = an installer owns the entry
  u32 c_cnt[ECB_CACHE];                // reads counted in this entry
  u32 c_first[ECB_CACHE];              // smallest offset (in this push) of a read with this key
  alignas(8) uint2 c_rep[ECB_CACHE];   // offset and length of one read with this key (the installer's)
  u32 seen[ECB_SEEN_WORDS];            // one bit per key hash: a read with such a key missed before
  // per-warp queues of reads that missed the cache
  alignas(16) uint4 q_key[ECB_GWARPS][ECB_MQ];
  alignas(8) uint2 q_rep[ECB_GWARPS][ECB_MQ];  // offset, length
};

// Shared-memory accesses of the hot loop through 32-bit shared-window addresses (computed once per
// thread): generic pointers cost an address-space conversion per access.
__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint4 lds128(u32 a) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds64(u32 a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ u32 lds32(u32 a) {
  u32 v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts128(u32 a, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts64(u32 a, u32 x, u32 y) {
  asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void reds_add(u32 a, u32 v) { asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void reds_min(u32 a, u32 v) { asm volatile("red.shared.min.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ u32 atoms_or(u32 a, u32 v) {
  u32 old;
  asm volatile("atom.shared.or.b32 %0, [%1], %2;" : "=r"(old) : "r"(a), "r"(v) : "memory");
  return old;
}
__device__ __forceinline__ u32 atoms_cas(u32 a, u32 cmp, u32 v) {
  u32 old;
  asm volatile("atom.shared.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "r"(a), "r"(cmp), "r"(v) : "memory");
  return old;
}

#define ECB_RG_SENTINEL ((int)0x80000000)  // stands for read_group beyond the end of the push

__device__ __forceinline__ Key128 key_of(const uint4& k) {
  return Key128{((u64)k.y << 32) | k.x, ((u64)k.w << 32) | k.z};
}
__host__ __device__ __forceinline__ uint4 key_words(const Mix4& m) {
  uint4 k = make_uint4(m.a, m.b, m.c, m.d);
  if ((k.x & k.y & k.z & k.w) == 0xFFFFFFFFu) k.x = k.y = 0u;  // all-ones is the empty marker (as mix_to_key)
  return k;
}
// Column loads: read once (twice by overlapping windows, which L1 absorbs), so they are marked
// evict-first in L2 and leave the cache to the EC table.
#ifndef ECB_EVICT_FIRST
#define ECB_EVICT_FIRST 1
#endif
__device__ __forceinline__ u64 make_evict_first_policy() {
  u64 pol;
  asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ int ld_col(const int32_t* p, u64 pol) {
#if ECB_EVICT_FIRST
  int v;
  asm volatile("ld.global.nc.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
#else
  return __ldg(p);
#endif
}
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Reads that missed the cache go into the HBM table, two per lane (entries qa and qb of the warp's queue).
template <bool WITH_CELLS>
__device__ __forceinline__ void insert_misses(const GroupParams& P, u32 qk, u32 qr, u32 qa, bool hasA, u32 qb,
                                              bool hasB) {
  uint4 kA = make_uint4(0u, 0u, 0u, 0u), kB = kA;
  uint2 rA = make_uint2(0u, 0u), rB = rA;
  if (hasA) {
    kA = lds128(qk + qa * 16u);
    rA = lds64(qr + qa * 8u);
  }
  if (hasB) {
    kB = lds128(qk + qb * 16u);
    rB = lds64(qr + qb * 8u);
  }
  u32 slotA, slotB;
  global_upsert2(P, key_of(kA), rA.x, rA.y, hasA, key_of(kB), rB.x, rB.y, hasB, slotA, slotB);
  if (hasA) {
    if (slotA == ECB_NONE) {  // table too full: the host grows it and replays the flagged reads
      atomicOr(&P.overflow_bits[rA.x >> 5], 1u << (rA.x & 31));
      atomicAdd(&P.ctr->n_overflow, 1u);
    } else if (WITH_CELLS) {
      triple_upsert(P, slotA, (u32)P.cell[rA.x], P.order_base + rA.x);
    }
  }
  if (hasB) {
    if (slotB == ECB_NONE) {
      atomicOr(&P.overflow_bits[rB.x >> 5], 1u << (rB.x & 31));
      atomicAdd(&P.ctr->n_overflow, 1u);
    } else if (WITH_CELLS) {
      triple_upsert(P, slotB, (u32)P.cell[rB.x], P.order_base + rB.x);
    }
  }
}

struct LongRead {
  uint4 key;
  int len;
};

// Key and length of a read that starts at w and fills a whole window (>= 32 alignments).
// Warp-cooperative: walks the read in blocks of 32; duplicates inside a block come from one
// match, duplicates against the earlier blocks of the read from shuffled compares.  A read longer than
// ECB_MAX_READ_ALIGNMENTS stops the compares once it passes that length (the walk to its end goes on):
// up to max_read it is deferred to the sort-based pass of ecb_longread.cuh (its key here is not used),
// beyond it the push fails.  The read the push drops (its last alignment is drop_pos) is not deferred.
__device__ __noinline__ LongRead ecb_long_read(const int32_t* __restrict__ rg, const int32_t* __restrict__ tg,
                                               const int32_t* __restrict__ hp, int n, int w, int n_targets,
                                               int n_haps, EcbCounters* ctr, int max_read, int drop_pos,
                                               uint2* deferred) {
  const int lane = threadIdx.x & 31;
  const u32 lt_mask = (1u << lane) - 1u;
  const int rg0 = rg[w];
  Mix4 sum = mix_zero();
  int len = 0;
  bool bad = false, too_long = false;
  for (int b = 0;; ++b) {
    const int pos = w + 32 * b + lane;
    bool in = pos < n;
    const int r = in ? rg[pos] : 0;
    const int t = in ? tg[pos] : 0, h = in ? hp[pos] : 0;
    in = in && r == rg0;
    const u32 m = __ballot_sync(ECB_FULL, in);  // the read is contiguous: m is a run of low bits
    const u32 code = in ? ecb_code(t, h) : (0x80000000u | (u32)lane);
    bad |= in && ((u32)t >= (u32)n_targets || (u32)h >= (u32)n_haps);
    bool dup = (__match_any_sync(ECB_FULL, code) & lt_mask) != 0u;
    if (!too_long) {
      for (int e = 0; e < b; ++e) {
        const int pe = w + 32 * e + lane;
        const u32 ce = ecb_code(tg[pe], hp[pe]);
#pragma unroll 8
        for (int j = 0; j < 32; ++j) dup |= __shfl_sync(ECB_FULL, ce, j) == code;
      }
    }
    if (in && !dup) mix_add(sum, ecb_mix(code));
    len += __popc(m);
    if (m != ECB_FULL) break;
    if (len > ECB_MAX_READ_ALIGNMENTS) too_long = true;
  }
  if (bad) atomicOr(&ctr->error, ECB_DEVERR_VALUE_RANGE);
  if (len > ECB_MAX_READ_ALIGNMENTS && lane == 0) {
    if (len > max_read) atomicOr(&ctr->error, ECB_DEVERR_READ_TOO_LONG);
    else if (w + len - 1 != drop_pos) deferred[atomicAdd(&ctr->n_deferred, 1u)] = make_uint2((u32)w, (u32)len);
  }
  sum.a = __reduce_add_sync(ECB_FULL, sum.a);
  sum.b = __reduce_add_sync(ECB_FULL, sum.b);
  sum.c = __reduce_add_sync(ECB_FULL, sum.c);
  sum.d = __reduce_add_sync(ECB_FULL, sum.d);
  LongRead r;
  r.key = key_words(sum);
  r.len = len;
  return r;
}

template <bool WITH_CELLS>
__global__ void __launch_bounds__(ECB_GTHREADS, 1) ecb_group_insert_kernel(const GroupParams P) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  GroupSmem& S = *reinterpret_cast<GroupSmem*>(smem_raw);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const u32 lt_mask = (1u << lane) - 1u;
  const u32 le_mask = (2u << lane) - 1u;
  const int n = P.n;
  const bool use_cache = !WITH_CELLS && P.use_cache;
  const int32_t* __restrict__ const c_rg = P.rg;
  const int32_t* __restrict__ const c_tg = P.tg;
  const int32_t* __restrict__ const c_hp = P.hp;
  // lanes 0..2 pull one column each into L2 ahead of the window
  const int32_t* const pf_col = (lane == 0 ? c_rg : (lane == 1 ? c_tg : c_hp)) + ECB_PF_DIST;
  const int pf_end = lane < 3 ? n - ECB_PF_DIST : 0;
  const int drop_pos = P.drop_last ? n - 1 : -1;  // the read that ends here is not counted
  const u64 col_policy = make_evict_first_policy();

  if (use_cache) {
    for (int i = tid; i < ECB_CACHE; i += ECB_GTHREADS) {
      S.c_key[i] = make_uint4(~0u, ~0u, ~0u, ~0u);
      S.c_lock[i] = 0u;
      S.c_cnt[i] = 0u;
      S.c_first[i] = 0xFFFFFFFFu;
    }
    for (int i = tid; i < ECB_SEEN_WORDS; i += ECB_GTHREADS) S.seen[i] = 0u;
  }
  __syncthreads();

  const u32 qk = smem_u32(S.q_key[warp]);  // this warp's miss queue (shared-window addresses)
  const u32 qr = smem_u32(S.q_rep[warp]);
  const u32 a_key = smem_u32(S.c_key), a_lock = smem_u32(S.c_lock), a_cnt = smem_u32(S.c_cnt);
  const u32 a_first = smem_u32(S.c_first), a_rep = smem_u32(S.c_rep), a_seen = smem_u32(S.seen);
  u32 qn = 0, qh = 0;     // reads parked in this warp's miss queue (a ring of ECB_MQ) and index of the oldest (warp-uniform)
  u32 reads_counted = 0;  // per lane

  for (;;) {
    // ---- next chunk of the stream (dynamic: whichever warp is free takes it) -------------------------
    u32 ci = 0;
    if (lane == 0) ci = atomicAdd(&P.ctr->chunk_next, 1u);
    ci = __shfl_sync(ECB_FULL, ci, 0);
    const long long cb64 = (long long)ci * P.chunk_len;
    if (cb64 >= n) break;
    const int cb = (int)cb64;
    const int ce = (int)min(cb64 + P.chunk_len, (long long)n);

    // first read start inside the chunk (a read belongs to the chunk it starts in)
    int w = cb;
    if (cb > 0) {
      w = -1;
      for (int b = cb; b < ce; b += 32) {
        const int pos = b + lane;
        const bool hd = pos < ce && c_rg[pos] != c_rg[pos - 1];
        const u32 m = __ballot_sync(ECB_FULL, hd);
        if (m) {
          w = b + __ffs(m) - 1;
          break;
        }
      }
      if (w < 0) continue;  // one long read covers the whole chunk
    }

    int rgv = ECB_RG_SENTINEL, tgv = 0, hpv = 0;
    if (w + lane < n) {
      rgv = ld_col(c_rg + w + lane, col_policy);
      tgv = ld_col(c_tg + w + lane, col_policy);
      hpv = ld_col(c_hp + w + lane, col_policy);
    }

    // ---- windows of 32 alignments, each starting at a read start -------------------------------------
    do {
      // read starts: positions beyond the end hold the sentinel, so the first of them closes the last read
      const int prev = __shfl_up_sync(ECB_FULL, rgv, 1);
      const u32 hb = __ballot_sync(ECB_FULL, rgv != prev) | 1u;

      bool ins;    // this lane holds the last alignment of a complete, owned read
      uint4 key;   // ... its key
      u32 s, len;  // ... its first alignment and its number of alignments
      int wnext;
      if (hb == 1u) {
        // one read fills the window
        const LongRead lr = ecb_long_read(c_rg, c_tg, c_hp, n, w, P.n_targets, P.n_haps, P.ctr, P.max_read, drop_pos,
                                          P.deferred);
        key = lr.key;
        s = (u32)w;
        len = (u32)lr.len;
        wnext = w + lr.len;
        ins = lane == 0 && wnext - 1 != drop_pos && lr.len <= ECB_MAX_READ_ALIGNMENTS;
      } else {
        const int last_head = 31 - __clz(hb);          // >= 1; lanes below it form complete reads
        const int st = 31 - __clz(hb & le_mask);       // lane of this alignment's read start
        const bool active = lane < last_head;
        const u32 code = ecb_code(tgv, hpv);
        // (target / haplotype bounds are checked by the harvest kernels: every distinct element of the
        // input is part of the representative read of some new EC)
        // an element counts once per read: drop it if a lower lane of the same read has the same code.
        // Windows whose complete reads have at most 8 alignments (the usual case) compare against the
        // up to 7 lanes below with shuffles; match_any, which walks the distinct values of the warp one
        // by one, is kept for windows with longer reads.
        u32 run = ~hb & ((1u << last_head) - 1u);  // lanes that continue a read
        const u32 run2 = run & (run >> 1), run4 = run2 & (run2 >> 2);
        bool dup = false;
#if ECB_SHUFFLE_DEDUP
        if ((run4 & (run4 >> 4)) == 0u) {
          const int reach = lane - st;  // lanes of the same read below this one
#define ECB_DUP_STEP(D) dup |= (__shfl_up_sync(ECB_FULL, code, D) == code) && reach >= D;
          if (run) {
            ECB_DUP_STEP(1)
            if (run2) {
              ECB_DUP_STEP(2)
              ECB_DUP_STEP(3)
              if (run4) {
                ECB_DUP_STEP(4)
                ECB_DUP_STEP(5)
                ECB_DUP_STEP(6)
                ECB_DUP_STEP(7)
              }
            }
          }
#undef ECB_DUP_STEP
        } else
#endif
        {
          const u32 same = __match_any_sync(ECB_FULL, code);
          dup = ((same & lt_mask) >> st) != 0u;
        }
        const bool contrib = active && !dup;
        Mix4 X = ecb_mix(code);
        if (!contrib) X = mix_zero();
        // segmented inclusive scan over the lanes of each read, with only as many doubling steps as
        // the longest complete read of the window needs (warp-uniform, from the head ballot)
#define ECB_SEG_STEP(D)                                \
  {                                                    \
    const u32 va = __shfl_up_sync(ECB_FULL, X.a, D);   \
    const u32 vb = __shfl_up_sync(ECB_FULL, X.b, D);   \
    const u32 vc = __shfl_up_sync(ECB_FULL, X.c, D);   \
    const u32 vd = __shfl_up_sync(ECB_FULL, X.d, D);   \
    if (lane - D >= st) {                              \
      X.a += va; X.b += vb; X.c += vc; X.d += vd;      \
    }                                                  \
  }
        if (run) {
          ECB_SEG_STEP(1)
          if (run2) {
            ECB_SEG_STEP(2)
            if (run4) {
              ECB_SEG_STEP(4)
              run = run4 & (run4 >> 4);
              if (run) {
                ECB_SEG_STEP(8)
                run &= run >> 8;
                if (run) ECB_SEG_STEP(16)
              }
            }
          }
        }
#undef ECB_SEG_STEP
        wnext = w + last_head;
        s = (u32)(w + st);
        len = (u32)(lane - st + 1);
        // lane + 1 is a head, the read is complete, starts in this chunk and is not the dropped one
        ins = (((hb >> 1) >> lane) & 1u) && active && (int)s < ce && w + lane != drop_pos;
        key = key_words(X);
      }

      // ---- request the next window's columns now; they arrive while this window is inserted ---------
      {
        const int np = wnext + lane;
        rgv = ECB_RG_SENTINEL;
        if (np < n) {
          rgv = ld_col(c_rg + np, col_policy);
          tgv = ld_col(c_tg + np, col_policy);
          hpv = ld_col(c_hp + np, col_policy);
        }
        if (wnext < pf_end) prefetch_l2(pf_col + wnext);
      }
      w = wnext;

      // ---- closed reads: hot-EC cache first --------------------------------------------------------
      bool miss = ins;
      if (ins) ++reads_counted;
      if (use_cache && ins) {
        const u32 cidx = (key.y >> 7) & (ECB_CACHE - 1);
        const uint4 ck = lds128(a_key + cidx * 16u);
        const u32 cf = lds32(a_first + cidx * 4u);
        bool hit = ck.x == key.x && ck.y == key.y && ck.z == key.z && ck.w == key.w;
        if (!hit && (ck.x & ck.y & ck.z & ck.w) == 0xFFFFFFFFu) {
          // empty entry.  Most keys occur once in a CTA's share of the stream and would only use up
          // the cache: a key is admitted when a read with the same hash bits has missed before.
          // Then one lane wins the lock, its read becomes the key's representative, and the single
          // 128-bit store of the key publishes the entry.
#if ECB_ADMIT_SECOND
          const u32 sbit = 1u << (key.z & 31u);
          const bool again = (atoms_or(a_seen + ((key.z >> 5) & (ECB_SEEN_WORDS - 1)) * 4u, sbit) & sbit) != 0u;
#else
          const bool again = true;
#endif
          if (again && atoms_cas(a_lock + cidx * 4u, 0u, 1u) == 0u) {
            sts64(a_rep + cidx * 8u, s, len);
            sts128(a_key + cidx * 16u, key);
            hit = true;
          }
        }
        if (hit) {
          reds_add(a_cnt + cidx * 4u, 1u);
          if (s < cf) reds_min(a_first + cidx * 4u, s);
          miss = false;
        }
      }
      // ---- misses: park in the warp's queue (pulling their home slots into L2), insert 64 at a time --
      const u32 mm = __ballot_sync(ECB_FULL, miss);
      if (mm) {
        if (miss) {
          u32 q = qh + qn + __popc(mm & lt_mask);
          if (q >= ECB_MQ) q -= ECB_MQ;
          sts128(qk + q * 16u, key);
          sts64(qr + q * 8u, s, len);
          prefetch_l2(P.table + (ec_slot_hash(key_of(key)) & P.mask));
        }
        qn += __popc(mm);
        __syncwarp();
        if (qn >= 64u) {
          // the OLDEST 64 go: the home slots of the newest are still on their way into L2
          u32 qa = qh + lane, qb = qh + 32 + lane;
          if (qa >= ECB_MQ) qa -= ECB_MQ;
          if (qb >= ECB_MQ) qb -= ECB_MQ;
          insert_misses<WITH_CELLS>(P, qk, qr, qa, true, qb, true);
          qh += 64u;
          if (qh >= ECB_MQ) qh -= ECB_MQ;
          qn -= 64u;
          __syncwarp();
        }
      }
    } while (w < ce);
  }

  // ---- leftovers of the miss queue, then the cache goes into the HBM table ---------------------------
  if (qn) {
    u32 qa = qh + lane, qb = qh + 32 + lane;
    if (qa >= ECB_MQ) qa -= ECB_MQ;
    if (qb >= ECB_MQ) qb -= ECB_MQ;
    insert_misses<WITH_CELLS>(P, qk, qr, qa, (u32)lane < qn, qb, (u32)lane + 32u < qn);
  }
  reads_counted = __reduce_add_sync(ECB_FULL, reads_counted);
  if (lane == 0 && reads_counted) atomicAdd(&P.ctr->n_reads, (u64)reads_counted);
  __syncthreads();
  if (use_cache) {
    for (int i = tid; i < ECB_CACHE; i += ECB_GTHREADS) {
      const u32 cnt = S.c_cnt[i];
      if (cnt) {
        const Key128 key = key_of(S.c_key[i]);
        const u32 first = S.c_first[i];
        const uint2 rep = S.c_rep[i];
        const u32 slot = global_upsert(P, key, cnt, first, rep.x, rep.y);
        if (slot == ECB_NONE) {  // table too full: park the entry, the host grows the table and replays it
          const u32 si = atomicAdd(&P.ctr->n_spill, 1u);
          P.spill[si] = EcbSpill{key.lo, key.hi, cnt, first, rep.x, rep.y};
        }
      }
    }
  }
}

// Number of reads (runs of equal read_group) in a push.
__global__ void __launch_bounds__(256) ecb_count_reads_kernel(const int32_t* __restrict__ rg, int n, u32* out) {
  u32 cnt = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    cnt += (i == 0 || rg[i] != rg[i - 1]) ? 1u : 0u;
  cnt = __reduce_add_sync(ECB_FULL, cnt);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(out, cnt);
}

// Key of the read that starts at offset s, computed serially (replay / verification path).
__device__ inline Key128 ecb_serial_read_key(const int32_t* rg, const int32_t* tg, const int32_t* hp, int n,
                                             int s, int* len_out) {
  const int my = rg[s];
  Mix4 sum = mix_zero();
  int j = s;
  for (; j < n && rg[j] == my; ++j) {
    const u32 cj = ecb_code(tg[j], hp[j]);
    bool dup = false;
    for (int m = s; m < j; ++m)
      if (ecb_code(tg[m], hp[m]) == cj) {
        dup = true;
        break;
      }
    if (!dup) mix_add(sum, ecb_mix(cj));
  }
  if (len_out) *len_out = j - s;
  return mix_to_key(sum);
}

// ECB_OPT_VERIFY_KEYS: prove that no two different reads of this push were merged by the 128-bit key.
// One thread per read: its key is recomputed serially, its EC looked up, and the read's set of
// (target, haplotype) pairs compared with the EC's row: every pair must be in the row and the number of
// distinct pairs must equal the number of bits set in the row's masks.  O(k * row) per read - a
// debugging aid, not part of the streaming path.
struct VerifyParams {
  const int32_t* rg;
  const int32_t* tg;
  const int32_t* hp;
  int n;
  int drop_last;
  const EcbEntry* table;
  u32 mask;
  const u32* row_len;
  const u32* row_off;
  const uint2* arena;
  EcbCounters* ctr;
};

__global__ void __launch_bounds__(256) ecb_verify_kernel(const VerifyParams P) {
  for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < P.n; s += gridDim.x * blockDim.x) {
    if (s > 0 && P.rg[s] == P.rg[s - 1]) continue;   // not a read start
    int end = s + 1;
    while (end < P.n && P.rg[end] == P.rg[s]) ++end;
    if (end - s > ECB_MAX_READ_ALIGNMENTS) continue;   // deferred: verified by ecb_long_verify_kernel
    int len = 0;
    const Key128 key = ecb_serial_read_key(P.rg, P.tg, P.hp, P.n, s, &len);
    if (P.drop_last && s + len == P.n) continue;
    u32 slot = ec_slot_hash(key) & P.mask;
    bool found = false;
    for (u32 p = 0; p <= P.mask; ++p) {
      Key128 k;
      u64 first;
      u32 cm1, aux;
      load_entry_cg(P.table + slot, k, first, cm1, aux);
      if (key_eq(k, key)) {
        found = true;
        const uint2* row = P.arena + P.row_off[aux];
        const u32 rl = P.row_len[aux];
        u32 bits = 0, distinct = 0;
        for (u32 j = 0; j < rl; ++j) bits += __popc(row[j].y);
        bool ok = true;
        for (int i = s; i < s + len && ok; ++i) {
          const u32 t = (u32)P.tg[i], h = (u32)P.hp[i];
          bool seen_before = false;
          for (int m = s; m < i; ++m) seen_before |= (u32)P.tg[m] == t && (u32)P.hp[m] == h;
          if (seen_before) continue;
          ++distinct;
          bool in_row = false;
          for (u32 j = 0; j < rl; ++j) in_row |= row[j].x == t && ((row[j].y >> h) & 1u);
          ok = in_row;
        }
        if (!ok || distinct != bits) atomicOr(&P.ctr->error, ECB_DEVERR_VERIFY);
        break;
      }
      if (key_empty(k)) break;
      slot = (slot + 1) & P.mask;
    }
    if (!found) atomicOr(&P.ctr->error, ECB_DEVERR_VERIFY);
  }
}

// Replay the reads flagged in overflow_bits after the table has been grown.  One thread per flagged
// read (rare path).  Bits of reads that went in are cleared; n_overflow counts the ones that did not.
template <bool WITH_CELLS>
__global__ void __launch_bounds__(256) ecb_replay_kernel(const GroupParams P) {
  const int n_words = (P.n + 31) >> 5;
  for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += gridDim.x * blockDim.x) {
    u32 bits = P.overflow_bits[w];
    while (bits) {
      const int b = __ffs(bits) - 1;
      bits &= bits - 1;
      const int s = (w << 5) + b;
      int len = 0;
      const Key128 key = ecb_serial_read_key(P.rg, P.tg, P.hp, P.n, s, &len);
      const u32 slot = global_upsert(P, key, 1u, (u32)s, (u32)s, (u32)len);
      if (slot == ECB_NONE) {
        atomicAdd(&P.ctr->n_overflow, 1u);
        continue;
      }
      if (WITH_CELLS) triple_upsert(P, slot, (u32)P.cell[s], P.order_base + (u32)s);
      atomicAnd(&P.overflow_bits[w], ~(1u << b));
    }
  }
}

// Replay parked hot-cache entries after the table has been grown.  Entries that still do not fit are
// compacted to the front of the list (n_spill counts them).
__global__ void __launch_bounds__(256) ecb_spill_replay_kernel(const GroupParams P, const EcbSpill* __restrict__ in,
                                                               u32 n_in) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n_in; i += gridDim.x * blockDim.x) {
    const EcbSpill e = in[i];
    const u32 slot = global_upsert(P, Key128{e.lo, e.hi}, e.count, e.first, e.rep, e.len);
    if (slot == ECB_NONE) {
      const u32 si = atomicAdd(&P.ctr->n_spill, 1u);
      P.spill[si] = e;
    }
  }
}

// Move every entry of `old_table` into `new_table` (capacity change).  remap (optional) records
// old slot -> new slot so that tables keyed by EC slot can be rewritten.
__global__ void __launch_bounds__(256) ecb_rehash_kernel(const EcbEntry* __restrict__ old_table, u32 old_slots,
                                                         EcbEntry* new_table, u32 new_mask, u32* ec_slot,
                                                         u32* remap, EcbCounters* ctr) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < old_slots; i += gridDim.x * blockDim.x) {
    Key128 k;
    u64 first;
    u32 cm1, aux;
    load_entry_cg(old_table + i, k, first, cm1, aux);
    if (remap) remap[i] = ECB_NONE;
    if (key_empty(k)) continue;
    u32 slot = ec_slot_hash(k) & new_mask;
    for (;;) {
      Key128 old = atomic_cas128(new_table + slot, Key128{~0ull, ~0ull}, k);
      if (key_empty(old)) break;
      slot = (slot + 1) & new_mask;
    }
    EcbEntry* e = new_table + slot;
    e->first = first;
    e->countm1 = cm1;
    e->aux = aux;
    if (ec_slot && aux != ECB_NONE) ec_slot[aux] = slot;
    if (remap) remap[i] = slot;
  }
}

// Rewrite the EC-slot half of every triple key after an EC-table rehash and move the entry into a
// fresh triple table.
__global__ void __launch_bounds__(256) ecb_triple_remap_kernel(const EcbEntry* __restrict__ old_table, u32 old_slots,
                                                               EcbEntry* new_table, u32 new_mask,
                                                               const u32* __restrict__ remap) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < old_slots; i += gridDim.x * blockDim.x) {
    Key128 k;
    u64 first;
    u32 cm1, aux;
    load_entry_cg(old_table + i, k, first, cm1, aux);
    if (key_empty(k)) continue;
    if (remap) {
      const u32 old_slot = (u32)(k.lo >> 32);
      k.lo = ((u64)remap[old_slot] << 32) | (k.lo & 0xFFFFFFFFull);
    }
    u32 slot = key_slot_hash(k) & new_mask;
    for (;;) {
      Key128 old = atomic_cas128(new_table + slot, Key128{~0ull, ~0ull}, k);
      if (key_empty(old)) break;
      slot = (slot + 1) & new_mask;
    }
    EcbEntry* e = new_table + slot;
    e->first = first;
    e->countm1 = cm1;
    e->aux = aux;
  }
}
