// ecb_sam.cuh — device parse of single-sample SAM text (ecb_sam_* in include/ecb200.h): line finding, the first eight
// fields of every alignment line, and the single-sample rules, producing the int32 columns ecb_bam_decode produces for
// the BAM file that holds the same alignments (DESIGN.md section 6.5).
//
// A call is whole lines of text.  Per call:
//   lines   the text is cut into segments of SAM_SEG bytes, one warp per segment, read with 16-byte loads.  A count pass
//           gives every segment's '\n' and '\t' bytes; their exclusive scans (device_scan) give the line and tab
//           prefix at every segment's start, and a write pass stores, per line, the offset of its '\n' and the tab
//           prefix there.  A line's field count is the tab prefix at its end minus the one at its start, plus one;
//   fields  one thread per line parses QNAME, FLAG, RNAME, POS, RNEXT and PNEXT (RNAME and RNEXT through an open
//           addressing table of the @SQ names, confirmed byte for byte), applies the filter (ecb_alignment_rule) and
//           reports the first bad line of the call with one 64-bit atomicMin of (line << 4 | kind);
//   rules   valid lines are compacted in order, and the starts and rows kernels the BAM decoder uses
//           (ecb_read_starts_kernel / ecb_read_rows_kernel with SamRecordAt) give read_group, target_idx and hap_idx.
#pragma once
#include "ecb_bam.cuh"
#include "ecb_scan.cuh"

#define SAM_SEG 4096u                 // bytes per line-finding segment (one warp)
#define SAM_WORDS (SAM_SEG / 16u)     // 16-byte words per segment
#define SAM_MAX_QNAME 254u

// Kinds of a bad line, in the order one line is checked (sam_utils.iter_records checks in the same order).
enum {
  SAM_BAD_HEADER = 1,   // a line starting with '@' after the first alignment line
  SAM_BAD_FIELDS = 2,   // fewer than 11 tab-separated fields
  SAM_BAD_QNAME = 3,
  SAM_BAD_FLAG = 4,
  SAM_BAD_RNAME = 5,
  SAM_BAD_POS = 6,
  SAM_BAD_RNEXT = 7,
  SAM_BAD_PNEXT = 8,
  SAM_BAD_TID = 9,      // a valid alignment whose RNAME is '*'
};
#define SAM_NO_ERROR 0xFFFFFFFFFFFFFFFFull

struct SamDevState {
  unsigned long long bad;     // (line index in the call << 4 | kind) of the first bad line; SAM_NO_ERROR: none
  ReadCarry carry;
};

// One slot of the @SQ name table: the name's 64-bit hash and its tid (-1: empty).
struct SamNameSlot {
  unsigned long long hash;
  int tid;
  int pad;
};

struct SamNames {
  const SamNameSlot* slots;
  u32 mask;                   // slots - 1 (a power of two)
  const char* blob;           // names back to back
  const int64_t* off;         // [n_ref + 1]
};

// FNV-1a, 64 bits; the host builds the table with the same function.
__host__ __device__ __forceinline__ unsigned long long sam_hash(const uint8_t* s, u32 n) {
  unsigned long long h = 1469598103934665603ull;
  for (u32 i = 0; i < n; ++i) h = (h ^ s[i]) * 1099511628211ull;
  return h;
}

// tid of the @SQ name s[0, n), or -2 when there is none
__device__ int sam_lookup(const SamNames& N, const uint8_t* s, u32 n) {
  const unsigned long long h = sam_hash(s, n);
  for (u32 i = (u32)h & N.mask;; i = (i + 1) & N.mask) {
    const SamNameSlot e = N.slots[i];
    if (e.tid < 0) return -2;
    if (e.hash != h) continue;
    const int64_t a = N.off[e.tid];
    if (N.off[e.tid + 1] - a != (int64_t)n) continue;
    u32 j = 0;
    while (j < n && (uint8_t)N.blob[a + j] == s[j]) ++j;
    if (j == n) return e.tid;
  }
}

// bit i set iff byte i of the 16-byte word equals c (c4: c in all four bytes)
__device__ __forceinline__ u32 sam_byte_mask(const uint4 w, u32 c4) {
  const u32 x[4] = {w.x, w.y, w.z, w.w};
  u32 m = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const u32 e = __vcmpeq4(x[i], c4);
    m |= ((e >> 7) & 1u | (e >> 14) & 2u | (e >> 21) & 4u | (e >> 28) & 8u) << (4 * i);
  }
  return m;
}

// '\n' and '\t' bytes of every segment.  The text is padded with zero bytes to a whole segment.
__global__ void __launch_bounds__(256) ecb_sam_count_kernel(const uint4* __restrict__ text, u32 n_seg,
                                                            u32* __restrict__ seg_nl, u32* __restrict__ seg_tab) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= n_seg) return;
  u32 nl = 0, tab = 0;
  const uint4* w = text + (u64)s * SAM_WORDS;
#pragma unroll 4
  for (u32 i = lane; i < SAM_WORDS; i += 32) {
    const uint4 v = w[i];
    nl += __popc(sam_byte_mask(v, 0x0A0A0A0Au));
    tab += __popc(sam_byte_mask(v, 0x09090909u));
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    nl += __shfl_xor_sync(ECB_FULL, nl, d);
    tab += __shfl_xor_sync(ECB_FULL, tab, d);
  }
  if (lane == 0) {
    seg_nl[s] = nl;
    seg_tab[s] = tab;
  }
}

// Per line k: line_end[k] = offset of its '\n', tabs_end[k] = '\t' bytes in the text before it.  nl_x / tab_x: the
// exclusive scans of the count pass.
__global__ void __launch_bounds__(256) ecb_sam_lines_kernel(const uint4* __restrict__ text, u32 n_seg,
                                                            const u32* __restrict__ nl_x, const u32* __restrict__ tab_x,
                                                            u32* __restrict__ line_end, u32* __restrict__ tabs_end) {
  const u32 s = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (s >= n_seg) return;
  u32 nl_base = nl_x[s], tab_base = tab_x[s];
  const uint4* w = text + (u64)s * SAM_WORDS;
  for (u32 i = lane; i < SAM_WORDS; i += 32) {
    const uint4 v = w[i];
    const u32 mnl = sam_byte_mask(v, 0x0A0A0A0Au), mtab = sam_byte_mask(v, 0x09090909u);
    const u32 cnl = __popc(mnl), ctab = __popc(mtab);
    const u32 inl = warp_incl_scan_u32(cnl, lane), itab = warp_incl_scan_u32(ctab, lane);
    u32 k = nl_base + inl - cnl;
    const u32 t0 = tab_base + itab - ctab;
    for (u32 m = mnl; m; m &= m - 1) {
      const int b = __ffs(m) - 1;
      line_end[k] = s * SAM_SEG + i * 16u + (u32)b;
      tabs_end[k] = t0 + __popc(mtab & ((1u << b) - 1u));
      ++k;
    }
    nl_base += __shfl_sync(ECB_FULL, inl, 31);
    tab_base += __shfl_sync(ECB_FULL, itab, 31);
  }
}

// Parsed fields of one line that the rules read.
struct SamLine {
  u32 name_off;   // QNAME's offset in the call's text
  u32 name_len;   // trimmed length
  int tid;
};

struct SamFields {
  const uint8_t* text;
  const u32* line_end;
  const u32* tabs_end;
  u32 n_lines;
  SamNames names;
  int n_ref;
  int32_t* range_min;   // NULL: ranges not tracked
  int32_t* range_max;
  SamDevState* st;
};

// A decimal integer of the bytes [a, b): at least one ASCII digit and nothing else, at most `lim`; -1 otherwise.
__device__ __forceinline__ long long sam_decimal(const uint8_t* t, u32 a, u32 b, long long lim) {
  if (a == b) return -1;
  long long v = 0;
  for (u32 i = a; i < b; ++i) {
    const u32 d = (u32)t[i] - '0';
    if (d > 9) return -1;
    v = v * 10 + d;
    if (v > lim) return -1;
  }
  return v;
}

// RNAME / RNEXT: '*' -> -1, '=' (eq_tid >= -1 allows it) -> eq_tid, an @SQ name -> its tid, otherwise -2
__device__ __forceinline__ int sam_ref(const SamNames& N, const uint8_t* t, u32 a, u32 b, int eq_tid) {
  if (b == a + 1 && t[a] == '*') return -1;
  if (eq_tid >= -1 && b == a + 1 && t[a] == '=') return eq_tid;
  return sam_lookup(N, t + a, b - a);
}

// One thread per line: the fields, the checks in SAM_BAD_* order, the filter and the ranges.  valid[k] = 1 for a valid
// alignment.
__global__ void ecb_sam_fields_kernel(SamFields F, SamLine* __restrict__ out, u32* __restrict__ valid) {
  const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= F.n_lines) return;
  const uint8_t* t = F.text;
  const u32 start = k ? F.line_end[k - 1] + 1 : 0u, end = F.line_end[k];
  const u32 fields = F.tabs_end[k] - (k ? F.tabs_end[k - 1] : 0u) + 1;
  u32 kind = 0, v = 0;
  if (start < end && t[start] == '@') {
    kind = SAM_BAD_HEADER;
  } else if (fields < 11) {
    kind = SAM_BAD_FIELDS;
  } else {
    u32 cut[9];                     // cut[f]: start of field f; cut[f + 1] - 1: its end
    cut[0] = start;
    u32 p = start;
    for (int f = 1; f <= 8; ++f) {
      while (t[p] != '\t') ++p;     // the line holds at least ten tabs
      cut[f] = ++p;
    }
    const u32 qlen = cut[1] - 1 - cut[0];
    const long long flag = sam_decimal(t, cut[1], cut[2] - 1, 65535);
    const int tid = sam_ref(F.names, t, cut[2], cut[3] - 1, -3);
    const long long pos = sam_decimal(t, cut[3], cut[4] - 1, 0x7FFFFFFF);
    const int ntid = tid >= -1 ? sam_ref(F.names, t, cut[6], cut[7] - 1, tid) : -1;
    const long long pnext = sam_decimal(t, cut[7], cut[8] - 1, 0x7FFFFFFF);
    if (qlen == 0 || qlen > SAM_MAX_QNAME) kind = SAM_BAD_QNAME;
    else if (flag < 0) kind = SAM_BAD_FLAG;
    else if (tid < -1) kind = SAM_BAD_RNAME;
    else if (pos < 0) kind = SAM_BAD_POS;
    else if (ntid < -1) kind = SAM_BAD_RNEXT;
    else if (pnext < 0) kind = SAM_BAD_PNEXT;
    else {
      const int rule = ecb_alignment_rule((u32)flag, tid, ntid, (int)(pnext - 1), F.n_ref);
      if (rule == ECB_REC_BAD_TID) {
        kind = SAM_BAD_TID;
      } else if (rule == ECB_REC_VALID) {
        v = 1;
        out[k] = SamLine{start, bam_trimmed_len(t + start, qlen), tid};
        if (F.range_min) {
          atomicMin(&F.range_min[tid], (int)(pos - 1));
          atomicMax(&F.range_max[tid], (int)(pos - 1));
        }
      }
    }
  }
  if (kind) atomicMin(&F.st->bad, ((unsigned long long)k << 4) | kind);
  valid[k] = v;
}

__global__ void ecb_sam_compact_kernel(const u32* __restrict__ valid, const u32* __restrict__ rowpos, u32 n_lines,
                                       u32* __restrict__ vline) {
  const u32 k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_lines || !valid[k]) return;
  vline[rowpos[k]] = k;
}

// The valid lines of a call for ecb_read_starts_kernel / ecb_read_rows_kernel (ecb_bam.cuh).
struct SamRecordAt {
  const uint8_t* text;
  const SamLine* lines;
  const u32* vline;      // [n_valid] line index
  __device__ __forceinline__ const uint8_t* name(u32 k, u32& len) const {
    const SamLine L = lines[vline[k]];
    len = L.name_len;
    return text + L.name_off;
  }
  __device__ __forceinline__ int tid(u32 k) const { return lines[vline[k]].tid; }
};
