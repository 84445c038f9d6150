// ecb_bam.cuh — device decode of single-sample BAM windows (ecb_bam_* in include/ecb200.h): BGZF inflate, the
// record hop, and the single-sample rules of libbamcols' process_window (bamcols.cpp), producing the same
// int32 columns bamcols_emit produces.
//
// A window is a run of whole BGZF blocks inflated behind the bytes the previous window left over (the start of a
// record that continues in this window).  Per window:
//   inflate   one thread per block (ecb_inflate.cuh), Huffman tables in shared memory;
//   hop       the window is cut into segments of ECB_BAM_SEG bytes; every segment guesses its first record
//             (two plausible record headers in a row, as bamcols.cpp:plausible_record) and hops by block_size to
//             its end, with bamcols' HOP_END / HOP_BAD rules.  Segment 0 starts at a known record.  A segment
//             whose start is not the landing offset of the segment in front of it is hopped again from that
//             offset, in rounds, until every start equals its predecessor's landing offset: then every chain is
//             the sequential hop by induction from segment 0 (the first segment that disagrees in a round is
//             hopped from a correct offset, so each round fixes at least one segment for good);
//   rules     validity and format checks per record; valid records are compacted in order (an exclusive sum),
//             each compares its trimmed name with the previous valid record's (the record before it in the
//             compacted list, or the name carried from the previous window), and read_group is the number of
//             reads started before the window plus an inclusive sum of the starts.
#pragma once
#include "ecb_common.cuh"
#include "ecb_inflate.cuh"

#define ECB_BAM_SEG 2048u            // bytes per hop segment
#define ECB_BAM_NONE 0xFFFFFFFFu
#define ECB_BAM_INFLATE_THREADS 64   // 64 x 708 bytes of Huffman tables per CTA

#define BAM_HOP_END 1u   // a partial record (or fewer than 4 bytes) at the landing offset
#define BAM_HOP_BAD 2u   // block_size < 32 at the landing offset

#define BAM_ERR_INFLATE 1u
#define BAM_ERR_NAME 2u
#define BAM_ERR_TID 4u

// What the rows of one call hand to the next: the open read and the trimmed name of the last valid record.  Shared
// by the BAM and SAM decoders (ecb_sam.cuh).
struct ReadCarry {
  unsigned long long open_row;       // first row of the read that is still open
  int have_name;              // a valid record has been seen
  u32 name_len;
  char name[256];             // trimmed name of the last valid record
};

// One BGZF block of a call: raw DEFLATE payload in the compressed buffer, inflated bytes in the window buffer.
struct BamBlock {
  u64 src_off;
  u32 src_len;
  u32 isize;
  u64 dst_off;
};

// Device state of one decoder, mirrored to the host after each step that needs it.
struct BamDevState {
  u32 error;                  // BAM_ERR_* bits
  u32 changed;                // segments hopped again in the last round
  long long bad_block;        // first corrupt block (index among the call's blocks)
  int bad_tid;                // a refID outside the header
  u32 hop_state, hop_land, hop_bs;   // end of the window's hop: state, offset, block_size there
  ReadCarry carry;
};

__device__ __forceinline__ u32 bam_le32(const uint8_t* p) {
  return (u32)p[0] | (u32)p[1] << 8 | (u32)p[2] << 16 | (u32)p[3] << 24;
}
__device__ __forceinline__ u32 bam_le16(const uint8_t* p) { return (u32)p[0] | (u32)p[1] << 8; }

__device__ __forceinline__ u32 bam_trimmed_len(const uint8_t* s, u32 n) {
  for (u32 i = 0; i < n; ++i)
    if (s[i] == ' ') return i > 0 ? i : n;
  return n;
}

// The single-sample filter (alntools/bam_utils.py:264-270; bamcols.cpp:record_validity and emitter._valid on the
// host) on one alignment's fields, for both device decoders: ECB_REC_BAD_TID is a valid alignment whose refID lies
// outside [0, n_ref).
enum { ECB_REC_FILTERED = 0, ECB_REC_VALID = 1, ECB_REC_BAD_TID = 2 };
__device__ __forceinline__ int ecb_alignment_rule(u32 flag, int tid, int ntid, int npos, int n_ref) {
  if (flag & 0x4) return ECB_REC_FILTERED;
  if ((flag & 0x1) && ((flag & 0x80) || !(flag & 0x2) || tid != ntid || npos < 0)) return ECB_REC_FILTERED;
  if (tid < 0 || tid >= n_ref) return ECB_REC_BAD_TID;
  return ECB_REC_VALID;
}

__global__ void __launch_bounds__(ECB_BAM_INFLATE_THREADS) ecb_bam_inflate_kernel(const uint8_t* __restrict__ comp,
                                                                                   const BamBlock* __restrict__ blocks,
                                                                                   long long b0, long long b1,
                                                                                   uint8_t* __restrict__ win,
                                                                                   BamDevState* st) {
  __shared__ ecbinf::Tables tabs[ECB_BAM_INFLATE_THREADS];
  const long long i = b0 + (long long)blockIdx.x * ECB_BAM_INFLATE_THREADS + threadIdx.x;
  if (i >= b1) return;
  const BamBlock B = blocks[i];
  if (!ecbinf::inflate_block(comp + B.src_off, B.src_len, win + B.dst_off, B.isize, tabs[threadIdx.x])) {
    atomicOr(&st->error, BAM_ERR_INFLATE);
    atomicMin(&st->bad_block, i);
  }
}

// bamcols.cpp:plausible_record (a heuristic: a wrong answer costs a second hop, never correctness)
__device__ bool bam_plausible(const uint8_t* base, u32 q, u32 wend, int n_ref) {
  if ((u64)q + 36 > wend) return false;
  const u32 bs = bam_le32(base + q);
  if (bs < 34 || bs > (1u << 26)) return false;
  const uint8_t* c = base + q + 4;
  const int tid = (int)bam_le32(c), pos = (int)bam_le32(c + 4), ntid = (int)bam_le32(c + 20);
  const u32 l_name = c[8], n_cigar = bam_le16(c + 12);
  const u32 l_seq = bam_le32(c + 16);
  if (tid < -1 || tid >= n_ref || ntid < -1 || ntid >= n_ref || pos < -1 || l_name == 0) return false;
  if (l_seq > bs || 32ull + l_name + 4ull * n_cigar + ((u64)l_seq + 1) / 2 + l_seq > bs) return false;
  if ((u64)q + 36 + l_name > wend) return true;
  const uint8_t* nm = c + 32;
  if (nm[l_name - 1] != 0) return false;
  for (u32 i = 0; i + 1 < l_name; ++i)
    if (nm[i] < 0x20 || nm[i] > 0x7e) return false;
  return true;
}

struct BamHop {
  const uint8_t* win;
  u32 p0, wend, n_seg;
  int n_ref;
  u32* start;     // [n_seg] first record of the segment (ECB_BAM_NONE: no guess)
  u32* cnt;       // [n_seg] records of the chain
  u32* state;     // [n_seg] HOP_* of the chain
};

__device__ __forceinline__ u32 seg_lo(const BamHop& H, u32 t) { return H.p0 + t * ECB_BAM_SEG; }
__device__ __forceinline__ u32 seg_hi(const BamHop& H, u32 t) {
  return t + 1 == H.n_seg ? H.wend : H.p0 + (t + 1) * ECB_BAM_SEG;
}

// bamcols.cpp:hop_chain for segment t from `from`: the records starting before the segment's end, their offsets
// into `out` (or, without out, their count and the HOP_* state into cnt / state).  Returns the landing offset.
__device__ u32 bam_hop_segment(const BamHop& H, u32 t, u32 from, u32* out) {
  u32 p = from, n = 0, state = 0;
  const u32 limit = seg_hi(H, t);
  if (from == ECB_BAM_NONE) {
    H.cnt[t] = 0;
    H.state[t] = 0;
    return ECB_BAM_NONE;
  }
  while (p < limit) {
    if ((u64)p + 4 > H.wend) { state = BAM_HOP_END; break; }
    const u32 bs = bam_le32(H.win + p);
    if (bs < 32) { state = BAM_HOP_BAD; break; }
    if ((u64)p + 4 + bs > H.wend) { state = BAM_HOP_END; break; }
    if (out) out[n] = p;
    ++n;
    p += 4 + bs;
  }
  if (!out) {
    H.cnt[t] = n;
    H.state[t] = state;
  }
  return p;
}

// Guess every segment's first record and hop it.
__global__ void ecb_bam_guess_kernel(BamHop H, u32* __restrict__ land) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= H.n_seg) return;
  u32 g = ECB_BAM_NONE;
  if (t == 0) {
    g = H.p0;
  } else {
    const u32 hi = seg_hi(H, t);
    for (u32 q = seg_lo(H, t); q < hi; ++q) {
      if (!bam_plausible(H.win, q, H.wend, H.n_ref)) continue;
      const u64 nx = (u64)q + 4 + bam_le32(H.win + q);
      if (nx + 36 <= H.wend && !bam_plausible(H.win, (u32)nx, H.wend, H.n_ref)) continue;
      g = q;
      break;
    }
  }
  H.start[t] = g;
  land[t] = bam_hop_segment(H, t, g, nullptr);
}

// One round of the join: a segment that does not start where the one in front of it lands is hopped again from there.
__global__ void ecb_bam_round_kernel(BamHop H, const u32* __restrict__ land_in, u32* __restrict__ land_out, u32* changed) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= H.n_seg) return;
  if (t == 0 || H.start[t] == land_in[t - 1]) {
    land_out[t] = land_in[t];
    return;
  }
  const u32 from = land_in[t - 1];
  H.start[t] = from;
  land_out[t] = bam_hop_segment(H, t, from, nullptr);
  atomicAdd(changed, 1u);
}

// Offsets of every record, at the chains' places (base = exclusive sum of cnt); the window's landing state.
__global__ void ecb_bam_offsets_kernel(BamHop H, const u32* __restrict__ base, const u32* __restrict__ land,
                                       u32* __restrict__ off, BamDevState* st) {
  const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= H.n_seg) return;
  bam_hop_segment(H, t, H.start[t], off + base[t]);
  if (t + 1 == H.n_seg) {
    const u32 p = land[t];
    st->hop_state = H.state[t];
    st->hop_land = p;
    st->hop_bs = H.state[t] == BAM_HOP_BAD ? bam_le32(H.win + p) : 0u;
  }
}

struct BamRules {
  const uint8_t* win;
  const u32* off;        // [n_rec] record offsets
  u32 n_rec;
  int n_ref;
  const int32_t* tid_target;
  const int32_t* tid_hap;
  int32_t* range_min;    // NULL: ranges not tracked
  int32_t* range_max;
  BamDevState* st;
};

// bamcols.cpp:record_validity per record: valid[i] = 1 for a valid alignment.
__global__ void ecb_bam_validity_kernel(BamRules R, u32* __restrict__ valid) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R.n_rec) return;
  const uint8_t* rec = R.win + R.off[i];
  const u32 bs = bam_le32(rec);
  const uint8_t* q = rec + 4;
  const int tid = (int)bam_le32(q);
  const u32 l_name = q[8];
  const u32 flag = bam_le16(q + 14);
  const int ntid = (int)bam_le32(q + 20), npos = (int)bam_le32(q + 24);
  u32 v = 0;
  if (32 + l_name > bs || l_name == 0) {
    atomicOr(&R.st->error, BAM_ERR_NAME);
  } else {
    const int rule = ecb_alignment_rule(flag, tid, ntid, npos, R.n_ref);
    if (rule == ECB_REC_BAD_TID) {
      atomicOr(&R.st->error, BAM_ERR_TID);
      R.st->bad_tid = tid;
    } else if (rule == ECB_REC_VALID) {
      v = 1;
      if (R.range_min) {
        const int pos = (int)bam_le32(q + 4);
        atomicMin(&R.range_min[tid], pos);
        atomicMax(&R.range_max[tid], pos);
      }
    }
  }
  valid[i] = v;
}

__global__ void ecb_bam_compact_kernel(BamRules R, const u32* __restrict__ valid, const u32* __restrict__ rowpos,
                                       u32* __restrict__ vrec) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= R.n_rec || !valid[i]) return;
  vrec[rowpos[i]] = R.off[i];
}

// The valid records of a call in order, as the shared starts and rows kernels read them: record k's trimmed name and
// refID.  BamRecordAt reads them from the inflated window; SamRecordAt (ecb_sam.cuh) from the parsed lines.
struct BamRecordAt {
  const uint8_t* win;
  const u32* vrec;       // [n_valid] record offsets
  __device__ __forceinline__ const uint8_t* name(u32 k, u32& len) const {
    const uint8_t* q = win + vrec[k] + 4;
    len = bam_trimmed_len(q + 32, (u32)q[8] - 1);
    return q + 32;
  }
  __device__ __forceinline__ int tid(u32 k) const { return (int)bam_le32(win + vrec[k] + 4); }
};

// starts[k] = 1 iff valid record k's trimmed name differs from the previous valid record's (bamcols.cpp:single_starts)
template <class Rec>
__global__ void ecb_read_starts_kernel(Rec A, u32 n_valid, const ReadCarry* carry, u32* __restrict__ starts) {
  const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_valid) return;
  u32 nl, pl;
  const uint8_t* nm = A.name(k, nl);
  const uint8_t* pn;
  if (k > 0) {
    pn = A.name(k - 1, pl);
  } else if (carry->have_name) {
    pn = (const uint8_t*)carry->name;
    pl = carry->name_len;
  } else {
    starts[k] = 1;
    return;
  }
  u32 differ = nl != pl;
  for (u32 j = 0; j < nl && !differ; ++j) differ = nm[j] != pn[j];
  starts[k] = differ;
}

// Rows of the valid records at row0 + k; the open read and the carried name are updated.
template <class Rec>
__global__ void ecb_read_rows_kernel(Rec A, u32 n_valid, const u32* __restrict__ starts, const u32* __restrict__ starts_x,
                                     long long group0, unsigned long long row0, const int32_t* __restrict__ tid_target,
                                     const int32_t* __restrict__ tid_hap, ReadCarry* carry, int32_t* __restrict__ rg,
                                     int32_t* __restrict__ tg, int32_t* __restrict__ hp) {
  const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_valid) return;
  const int tid = A.tid(k);
  const unsigned long long row = row0 + k;
  rg[row] = (int32_t)(group0 + (long long)starts_x[k] + (long long)starts[k]);
  tg[row] = tid_target[tid];
  hp[row] = tid_hap[tid];
  if (starts[k]) atomicMax(&carry->open_row, row);
  if (k + 1 == n_valid) {
    u32 nl;
    const uint8_t* nm = A.name(k, nl);
    for (u32 j = 0; j < nl; ++j) carry->name[j] = (char)nm[j];
    carry->name_len = nl;
    carry->have_name = 1;
  }
}
