// ecb_inflate.cuh — raw DEFLATE (RFC 1951) decoder for one BGZF block, written once for the device and the host.
//
// Under nvcc the functions are __host__ __device__ (the BAM decode kernels of ecb_bam.cuh run them one thread per
// block); plain g++ compiles the same source, which is how tests/test_device_inflate_host.py checks it against
// zlib under AddressSanitizer / UBSan on a machine without a GPU.
//
// Acceptance is zlib's (what libbamcols' Inflater::run decides with inflate(Z_FINISH)): a block is accepted iff
// the stream is well formed up to the end-of-block code of its final block, every bit it uses lies inside the
// input, and it produces exactly dst_len bytes.  Bytes after the final block are ignored, CRC32 is not checked,
// and dst_len == 0 is accepted without looking at the input.  Rejected, as zlib rejects them: block type 3, stored
// LEN != ~NLEN, HLIT > 286 or HDIST > 30, an over-subscribed code, an incomplete code (except a literal/length or
// distance code of one 1-bit code), an incomplete or empty code-length code, a repeat with nothing to repeat or
// beyond HLIT + HDIST, no end-of-block code, literal/length symbols 286/287 and distance symbols 30/31, a
// distance before the first output byte, running out of input, and more or fewer than dst_len output bytes.
//
// Huffman codes are decoded canonically, one code bit at a time against the count of codes of each length (as
// zlib's contrib/puff does): 708 bytes of tables per decoder, small enough for shared memory per thread.  Every
// read of src and write of dst is bounds-checked; nothing outside [src, src + src_len) and [dst, dst + dst_len)
// is touched whatever the input.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define ECB_INF_FN __host__ __device__ __forceinline__
#else
#define ECB_INF_FN static inline
#endif

namespace ecbinf {

template <int N>
struct Huff {
  uint16_t count[16];   // codes of each length (count[0]: symbols without a code)
  uint16_t symbol[N];   // symbols in canonical order
};

struct Tables {
  Huff<288> lit;   // literal/length code; also holds the code-length code while a dynamic header is read
  Huff<32> dist;
  uint16_t pad[2];   // 177 words: consecutive threads' tables start in different shared-memory banks
};

struct Bits {
  const uint8_t* src;
  uint32_t len;     // input bytes
  uint32_t pos;     // next byte to load (may run past len: zeros are loaded there, and overran() notices)
  uint64_t buf;
  int cnt;          // bits in buf
};

ECB_INF_FN void refill(Bits& b) {
  while (b.cnt <= 56) {
    const uint64_t byte = b.pos < b.len ? b.src[b.pos] : 0u;
    b.buf |= byte << b.cnt;
    ++b.pos;
    b.cnt += 8;
  }
}

// more bits were consumed than the input holds
ECB_INF_FN bool overran(const Bits& b) { return (uint64_t)b.pos * 8u - (uint64_t)b.cnt > (uint64_t)b.len * 8u; }

ECB_INF_FN uint32_t take(Bits& b, int n) {
  if (b.cnt < n) refill(b);
  const uint32_t v = (uint32_t)(b.buf & ((1ull << n) - 1));
  b.buf >>= n;
  b.cnt -= n;
  return v;
}

// -1: no symbol has this code
template <int N>
ECB_INF_FN int decode(Bits& b, const Huff<N>& h) {
  if (b.cnt < 15) refill(b);
  int code = 0, first = 0, index = 0;
  for (int len = 1; len <= 15; ++len) {
    code |= (int)(b.buf & 1u);
    b.buf >>= 1;
    b.cnt--;
    const int count = h.count[len];
    if (code - count < first) return h.symbol[index + (code - first)];
    index += count;
    first += count;
    first <<= 1;
    code <<= 1;
  }
  return -1;
}

// Canonical code from code lengths.  Returns 0 complete (or no codes at all), > 0 incomplete, < 0 over-subscribed.
template <int N>
ECB_INF_FN int construct(Huff<N>& h, const uint8_t* length, int n) {
  for (int len = 0; len < 16; ++len) h.count[len] = 0;
  for (int s = 0; s < n; ++s) h.count[length[s]]++;
  if (h.count[0] == n) return 0;
  int left = 1;
  for (int len = 1; len < 16; ++len) {
    left <<= 1;
    left -= h.count[len];
    if (left < 0) return left;
  }
  uint16_t offs[16];
  offs[1] = 0;
  for (int len = 1; len < 15; ++len) offs[len + 1] = (uint16_t)(offs[len] + h.count[len]);
  for (int s = 0; s < n; ++s)
    if (length[s]) h.symbol[offs[length[s]]++] = (uint16_t)s;
  return left;
}

// Literal/length and distance codes of one block body.  false: malformed, out of input or out of output room.
ECB_INF_FN bool codes(Bits& b, const Tables& t, uint8_t* dst, uint32_t dst_len, uint32_t& out) {
  for (;;) {
    int sym = decode(b, t.lit);
    if (sym < 0 || overran(b)) return false;
    if (sym < 256) {
      if (out >= dst_len) return false;
      dst[out++] = (uint8_t)sym;
      continue;
    }
    if (sym == 256) return true;
    sym -= 257;
    if (sym >= 29) return false;   // 286, 287 (fixed code only)
    // RFC 1951 3.2.5 bases and extra bits, computed rather than looked up: no per-thread tables
    uint32_t length;
    if (sym < 8) {
      length = 3u + (uint32_t)sym;
    } else if (sym == 28) {
      length = 258u;
    } else {
      const int extra = (sym - 4) >> 2;
      length = ((4u + (uint32_t)(sym & 3)) << extra) + 3u + take(b, extra);
    }
    const int ds = decode(b, t.dist);
    if (ds < 0 || ds >= 30) return false;
    uint32_t distance;
    if (ds < 4) {
      distance = 1u + (uint32_t)ds;
    } else {
      const int extra = (ds - 2) >> 1;
      distance = ((2u + (uint32_t)(ds & 1)) << extra) + 1u + take(b, extra);
    }
    if (overran(b)) return false;
    if (distance > out || length > dst_len - out) return false;
    for (uint32_t i = 0; i < length; ++i, ++out) dst[out] = dst[out - distance];
  }
}

ECB_INF_FN void fixed_tables(Tables& t) {
  uint8_t lens[288];
  for (int s = 0; s < 144; ++s) lens[s] = 8;
  for (int s = 144; s < 256; ++s) lens[s] = 9;
  for (int s = 256; s < 280; ++s) lens[s] = 7;
  for (int s = 280; s < 288; ++s) lens[s] = 8;
  construct(t.lit, lens, 288);
  for (int s = 0; s < 30; ++s) lens[s] = 5;
  construct(t.dist, lens, 30);   // incomplete on purpose: codes 30 and 31 decode to nothing
}

ECB_INF_FN bool dynamic_tables(Bits& b, Tables& t) {
  const uint8_t ORDER[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
  uint8_t lens[286 + 30];
  const int nlen = (int)take(b, 5) + 257, ndist = (int)take(b, 5) + 1, ncode = (int)take(b, 4) + 4;
  if (nlen > 286 || ndist > 30) return false;
  for (int i = 0; i < 19; ++i) lens[ORDER[i]] = i < ncode ? (uint8_t)take(b, 3) : 0;
  if (overran(b)) return false;
  if (construct(t.lit, lens, 19) != 0) return false;   // the code-length code must be complete
  int index = 0;
  while (index < nlen + ndist) {
    int sym = decode(b, t.lit);
    if (sym < 0) return false;
    if (sym < 16) {
      lens[index++] = (uint8_t)sym;
    } else {
      uint8_t len = 0;
      if (sym == 16) {
        if (index == 0) return false;
        len = lens[index - 1];
        sym = 3 + (int)take(b, 2);
      } else if (sym == 17) {
        sym = 3 + (int)take(b, 3);
      } else {
        sym = 11 + (int)take(b, 7);
      }
      if (index + sym > nlen + ndist) return false;
      while (sym--) lens[index++] = len;
    }
    if (overran(b)) return false;
  }
  if (lens[256] == 0) return false;
  // an incomplete code is accepted only when it is a single 1-bit code
  int err = construct(t.lit, lens, nlen);
  if (err < 0 || (err > 0 && nlen != t.lit.count[0] + t.lit.count[1])) return false;
  err = construct(t.dist, lens + nlen, ndist);
  if (err < 0 || (err > 0 && ndist != t.dist.count[0] + t.dist.count[1])) return false;
  return true;
}

// One raw DEFLATE stream into exactly dst_len bytes.  true = accepted (see the file comment).
ECB_INF_FN bool inflate_block(const uint8_t* src, uint32_t src_len, uint8_t* dst, uint32_t dst_len, Tables& t) {
  if (dst_len == 0) return true;
  Bits b;
  b.src = src;
  b.len = src_len;
  b.pos = 0;
  b.buf = 0;
  b.cnt = 0;
  uint32_t out = 0;
  for (;;) {
    const uint32_t last = take(b, 1), type = take(b, 2);
    if (overran(b)) return false;
    if (type == 0) {
      take(b, b.cnt & 7);   // to the byte boundary
      const uint32_t len = take(b, 16), nlen = take(b, 16);
      if (overran(b) || len != (~nlen & 0xFFFFu)) return false;
      const uint32_t at = b.pos - (uint32_t)(b.cnt >> 3);   // first byte not yet consumed
      if (at > src_len || len > src_len - at || len > dst_len - out) return false;
      for (uint32_t i = 0; i < len; ++i) dst[out++] = src[at + i];
      b.pos = at + len;
      b.buf = 0;
      b.cnt = 0;
    } else if (type == 1) {
      fixed_tables(t);
      if (!codes(b, t, dst, dst_len, out)) return false;
    } else if (type == 2) {
      if (!dynamic_tables(b, t)) return false;
      if (!codes(b, t, dst, dst_len, out)) return false;
    } else {
      return false;
    }
    if (last) break;
  }
  return out == dst_len && !overran(b);
}

}  // namespace ecbinf
