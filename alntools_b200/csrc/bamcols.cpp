// bamcols.cpp — libbamcols.so: BGZF/BAM decode + the reference's per-alignment filters and read-name
// grouping, emitting the int32 columns libecb200 consumes (C ABI in include/bamcols.h).
//
// Replaces the front half of alntools/bam_utils.py:253-306 and bam_utils_multisample.py:209-300, which
// the reference runs one pysam object at a time inside Python.  Here: the file is memory-mapped,
// BGZF blocks are inflated a batch at a time by a pool of worker threads (blocks are independent
// deflate streams, SAM spec 4.1), and one pass over the fixed-offset record fields produces the rows.
#include <zlib.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <algorithm>
#include <atomic>
#include <chrono>
#include <climits>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <string_view>
#include <thread>
#include <unordered_map>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "../../include/bamcols.h"
#include "fast_inflate.h"

namespace {

thread_local std::string g_open_error;

inline uint32_t le32(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
inline uint32_t le16(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }

struct BlockJob {
  const uint8_t* src;
  uint32_t src_len;
  uint32_t isize;
  size_t dst_off;
};

}  // namespace

// Cell dictionary: ids in order of first appearance (bam_utils_multisample.py:270-280).  Open addressing
// over 64-bit name hashes (the hash can be computed by the parallel passes, the sequential part of a
// lookup is one probe and one memcmp).
struct bamcols_cells {
  std::vector<std::string> names;
  std::vector<uint64_t> slot_hash;   // 0 = empty
  std::vector<int32_t> slot_id;
  size_t mask = 0;
  static uint64_t hash_of(const char* s, size_t n) {
    uint64_t h = 0x9E3779B97F4A7C15ull ^ (uint64_t)n;
    size_t i = 0;
    for (; i + 8 <= n; i += 8) {
      uint64_t w;
      memcpy(&w, s + i, 8);
      h = (h ^ w) * 0xFF51AFD7ED558CCDull;
      h ^= h >> 32;
    }
    uint64_t w = 0;
    if (i < n) memcpy(&w, s + i, n - i);
    h = (h ^ w) * 0xC4CEB9FE1A85EC53ull;
    h ^= h >> 29;
    return h ? h : 1;
  }
  void grow() {
    const size_t cap = mask ? (mask + 1) * 2 : 1024;
    std::vector<uint64_t> h(cap, 0);
    std::vector<int32_t> id(cap, 0);
    for (size_t i = 0; i <= mask && mask; ++i)
      if (slot_hash[i]) {
        size_t j = slot_hash[i] & (cap - 1);
        while (h[j]) j = (j + 1) & (cap - 1);
        h[j] = slot_hash[i];
        id[j] = slot_id[i];
      }
    slot_hash.swap(h);
    slot_id.swap(id);
    mask = cap - 1;
  }
  // read-only lookup (safe from several threads while nobody inserts): id, or -1
  int32_t find(const char* s, size_t n, uint64_t h) const {
    if (mask == 0) return -1;
    for (size_t j = h & mask; slot_hash[j]; j = (j + 1) & mask)
      if (slot_hash[j] == h) {
        const std::string& nm = names[(size_t)slot_id[j]];
        if (nm.size() == n && memcmp(nm.data(), s, n) == 0) return slot_id[j];
      }
    return -1;
  }
  int32_t id_of(const char* s, size_t n, uint64_t h) {
    if ((names.size() + 1) * 2 > mask + 1 || mask == 0) grow();
    size_t j = h & mask;
    for (; slot_hash[j]; j = (j + 1) & mask)
      if (slot_hash[j] == h) {
        const std::string& nm = names[(size_t)slot_id[j]];
        if (nm.size() == n && memcmp(nm.data(), s, n) == 0) return slot_id[j];
      }
    const int32_t id = (int32_t)names.size();
    slot_hash[j] = h;
    slot_id[j] = id;
    names.emplace_back(s, n);
    return id;
  }
  int32_t id_of(const char* s, size_t n) { return id_of(s, n, hash_of(s, n)); }
};

// Grow-only buffer without value initialisation (std::vector::resize would write every new element first:
// 128 MiB of window and 100 MiB of staged rows per refill), large ones on transparent huge pages so that the
// first touch by the worker threads takes hundreds of page faults instead of tens of thousands.
template <class T>
struct RawBuf {
  T* p = nullptr;
  size_t n = 0, cap = 0;
  bool mapped = false;
  RawBuf() = default;
  RawBuf(const RawBuf&) = delete;
  RawBuf& operator=(const RawBuf&) = delete;
  ~RawBuf() { release(p, cap, mapped); }
  static void release(T* q, size_t c, bool m) {
    if (!q) return;
    if (m) munmap(q, c * sizeof(T)); else free(q);
  }
  T* data() { return p; }
  const T* data() const { return p; }
  size_t size() const { return n; }
  T& operator[](size_t i) { return p[i]; }
  const T& operator[](size_t i) const { return p[i]; }
  void resize(size_t want) {   // keeps the first min(n, want) elements; new elements are uninitialised
    if (want > cap) {
      size_t c = std::max(want, cap + cap / 2);
      const size_t HUGE = (size_t)2 << 20;
      T* q = nullptr;
      bool m = false;
      if (c * sizeof(T) >= 2 * HUGE) {
        const size_t bytes = (c * sizeof(T) + HUGE - 1) / HUGE * HUGE;
        void* a = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (a != MAP_FAILED) {
#ifdef MADV_HUGEPAGE
          madvise(a, bytes, MADV_HUGEPAGE);
#endif
          q = (T*)a;
          c = bytes / sizeof(T);
          m = true;
        }
      }
      if (!q) q = (T*)malloc(c * sizeof(T));
      if (!q) throw std::bad_alloc();
      if (n) memcpy(q, p, std::min(n, want) * sizeof(T));
      release(p, cap, mapped);
      p = q;
      cap = c;
      mapped = m;
    }
    n = want;
  }
};

struct bamcols {
  int fd = -1;
  const uint8_t* file = nullptr;
  size_t file_size = 0;
  size_t cpos = 0;               // compressed offset of the next BGZF block
  bool file_done = false;        // every block (of the range) has been inflated
  // a reader may be confined to a range of records [begin, end) given as BGZF virtual offsets (compressed
  // offset of a block << 16 | offset inside the inflated block): one shard of a file that several readers
  // share (bamcols_plan_shards / bamcols_set_range)
  size_t end_c = SIZE_MAX;       // compressed offset of the block that holds the end of the range
  uint32_t end_u = 0;            // ... and how many of its inflated bytes belong to the range
  int64_t first_voffset = 0;     // virtual offset of the first record (set by bamcols_open)
  size_t last_batch_c0 = 0, last_batch_keep = 0;   // where the latest refill started: file offset and window offset
  RawBuf<uint8_t> win;           // inflated window
  size_t wpos = 0, wend = 0;     // unread part of the window
  int n_threads = 1;
  size_t batch_blocks = 2048;    // up to 128 MiB inflated per refill
  // header
  std::vector<std::string> ref_names;
  std::vector<int32_t> ref_lengths;
  std::string ref_blob;          // every reference name followed by a NUL, in tid order
  std::vector<int32_t> tid_target, tid_hap;
  // grouping state (persists across emit calls)
  bool started = false;          // a valid alignment has been seen
  std::string current;           // remembered read name
  int64_t group = -1;
  bool pending = false;          // per-cell: the current read's cell is resolved at the next valid alignment
  int32_t cell = 0;
  bool records_done = false;
  int64_t all_alignments = 0;
  // staged rows of the current inflated window, produced by all worker threads
  RawBuf<int32_t> st_rg, st_tg, st_hp, st_cell;
  RawBuf<uint64_t> st_klo, st_khi;   // key mode (bamcols_emit_keys): 128-bit name keys in place of read_group
  size_t pending_row = 0;       // per-cell: stage row whose cell is resolved by the next valid alignment
  // per-cell scratch, kept between windows (fresh allocations of this size are page-faulted in every time)
  std::vector<size_t> sc_openers;
  std::vector<std::vector<size_t>> sc_mine;
  std::vector<const char*> sc_cell_ptr;
  std::vector<size_t> sc_cell_len;
  std::vector<uint64_t> sc_cell_hash;
  std::vector<int32_t> sc_cell_id, sc_group_cell;
  size_t st_pos = 0;             // next row to hand out
  size_t st_whole = 0;           // rows [st_pos, st_whole) are whole reads; [st_whole, size) is the open last read
  std::vector<size_t> rec_off;   // scratch: record offsets of the window
  std::vector<uint8_t> rec_flag; // scratch: per record of the window, see Window::fl
  int mode = 0;                  // 0 undecided, 1 single-sample, 2 per-cell, 3 name keys
  size_t grain = 4096;           // records per worker thread below which no further thread is used
  double phase_s[6] = {0, 0, 0, 0, 0, 0};  // inflate, record hop, validity, read starts, rows, copy-out
  // --rangefile (bam_utils.py:282-286): smallest / largest reference_start of the valid alignments per tid
  // header tables built natively (bamcols_build_tables)
  std::string tb_targets;        // main target names, each followed by a NUL, in main-target order
  std::string tb_haps;           // sorted haplotype names, each followed by a NUL
  std::vector<int32_t> tb_lengths;  // [n_targets x n_haps]
  int32_t tb_n_targets = 0, tb_n_haps = 0;
  std::string tb_section;        // the targets section of the EC file, built on demand
  // the first batch of blocks is inflated in the background while the caller builds its header tables
  std::thread prefetch;
  int prefetch_rc = 0;
  bool track_ranges = false;
  std::vector<int32_t> range_min, range_max;
  std::string err;
};

namespace {

// lap(p) adds the wall time since the previous lap, or since the clock was made, to phase p of bamcols::phase_s.
struct PhaseClock {
  double* phase_s;
  std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
  explicit PhaseClock(double* s) : phase_s(s) {}
  void lap(int phase) {
    const auto now = std::chrono::steady_clock::now();
    phase_s[phase] += std::chrono::duration<double>(now - t0).count();
    t0 = now;
  }
};

int fail(bamcols* r, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (r) r->err = buf; else g_open_error = buf;
  return code;
}

// Locate the next BGZF block at `off`: payload pointer/length and inflated size.  0 = ok, 1 = clean
// end of file, <0 = error.
int parse_block(bamcols* r, size_t off, BlockJob* job, size_t* bsize_out) {
  const size_t n = r->file_size;
  if (off == n) return 1;
  if (off + 18 > n) return fail(r, BAMCOLS_ERR_FORMAT, "truncated BGZF block header at offset %zu", off);
  const uint8_t* p = r->file + off;
  if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4))
    return fail(r, BAMCOLS_ERR_FORMAT, "not a BGZF block at offset %zu", off);
  const size_t xlen = le16(p + 10);
  if (off + 12 + xlen > n) return fail(r, BAMCOLS_ERR_FORMAT, "truncated BGZF extra field at offset %zu", off);
  size_t bsize = 0;
  for (size_t q = 12; q + 4 <= 12 + xlen;) {
    const size_t slen = le16(p + q + 2);
    if (p[q] == 'B' && p[q + 1] == 'C' && slen == 2) bsize = (size_t)le16(p + q + 4) + 1;
    q += 4 + slen;
  }
  if (bsize == 0) return fail(r, BAMCOLS_ERR_FORMAT, "BGZF block without BC field at offset %zu", off);
  if (bsize < 12 + xlen + 8 || off + bsize > n)
    return fail(r, BAMCOLS_ERR_FORMAT, "truncated BGZF block at offset %zu", off);
  job->src = p + 12 + xlen;
  job->src_len = (uint32_t)(bsize - 12 - xlen - 8);
  job->isize = le32(p + bsize - 4);
  // the spec caps ISIZE at 64 KiB, but writers that ignore the cap exist (and inflate does not care)
  if (job->isize > (1u << 30)) return fail(r, BAMCOLS_ERR_FORMAT, "BGZF block at offset %zu claims %u bytes", off, job->isize);
  *bsize_out = bsize;
  return 0;
}

// Per-worker inflate state: the whole-buffer decoder's tables and a zlib stream for the blocks it declines.
struct Inflater {
  z_stream zs;
  bool zs_ready = false;
  fastinflate::Tables scratch, fixed;
  bool fixed_ready = false;
  bool zlib_only = false;   // BAMCOLS_ZLIB_ONLY: timing comparisons and tests
  Inflater() { memset(&zs, 0, sizeof zs); }
  ~Inflater() {
    if (zs_ready) inflateEnd(&zs);
  }
  // raw deflate stream of known inflated size; true iff it decoded cleanly into exactly dst_len bytes
  bool run(const uint8_t* src, size_t src_len, uint8_t* dst, size_t dst_len) {
    if (dst_len == 0) return true;
    if (!zlib_only && fastinflate::fast_inflate(src, src_len, dst, dst_len, scratch, fixed, fixed_ready)) return true;
    // anything the fast decoder does not like is judged by zlib
    if (!zs_ready) {
      if (inflateInit2(&zs, -15) != Z_OK) return false;
      zs_ready = true;
    } else if (inflateReset(&zs) != Z_OK) {
      return false;
    }
    zs.next_in = const_cast<Bytef*>(src);
    zs.avail_in = (uInt)src_len;
    zs.next_out = dst;
    zs.avail_out = (uInt)dst_len;
    const int rc = inflate(&zs, Z_FINISH);
    return rc == Z_STREAM_END && zs.avail_out == 0;
  }
};

// Inflate the next batch of blocks behind the unread part of the window.  Returns 0, or <0 on error;
// sets file_done when the file has no more blocks.
int refill(bamcols* r) {
  if (r->file_done) return 0;
  PhaseClock clock(r->phase_s);
  // keep the unread tail at the front
  const size_t keep = r->wend - r->wpos;
  if (r->wpos > 0 && keep > 0) memmove(r->win.data(), r->win.data() + r->wpos, keep);
  r->wpos = 0;
  r->wend = keep;
  std::vector<BlockJob> jobs;
  jobs.reserve(r->batch_blocks);
  size_t total = 0, spill = 0;   // spill: inflated bytes of the last block that lie beyond the end of the range
  r->last_batch_c0 = r->cpos;
  r->last_batch_keep = keep;
  while (jobs.size() < r->batch_blocks) {
    if (r->cpos > r->end_c || (r->cpos == r->end_c && r->end_u == 0)) {
      r->file_done = true;
      break;
    }
    BlockJob job;
    size_t bsize = 0;
    const int rc = parse_block(r, r->cpos, &job, &bsize);
    if (rc < 0) return rc;
    if (rc == 1) {
      r->file_done = true;
      break;
    }
    job.dst_off = keep + total;
    if (r->cpos == r->end_c) {   // the range ends inside this block (at a record boundary)
      if (r->end_u > job.isize) return fail(r, BAMCOLS_ERR_INVALID, "range end lies beyond its block");
      total += r->end_u;
      spill = job.isize - r->end_u;
      r->cpos += bsize;
      jobs.push_back(job);
      r->file_done = true;
      break;
    }
    total += job.isize;
    r->cpos += bsize;
    jobs.push_back(job);
  }
  if (jobs.empty()) return 0;
  if (r->win.size() < keep + total + spill) r->win.resize(keep + total + spill);
  uint8_t* base = r->win.data();
  const int nt = (int)std::max<size_t>(1, std::min<size_t>((size_t)r->n_threads, (jobs.size() + 15) / 16));
  std::atomic<size_t> next(0);
  std::atomic<int> bad(0);
  const bool zlib_only = getenv("BAMCOLS_ZLIB_ONLY") != nullptr;
  auto work = [&]() {
    std::unique_ptr<Inflater> inf(new Inflater());
    inf->zlib_only = zlib_only;
    for (;;) {
      const size_t i0 = next.fetch_add(8);
      if (i0 >= jobs.size()) break;
      const size_t i1 = std::min(jobs.size(), i0 + 8);
      for (size_t i = i0; i < i1; ++i)
        if (!inf->run(jobs[i].src, jobs[i].src_len, base + jobs[i].dst_off, jobs[i].isize)) bad.store(1);
    }
  };
  if (nt == 1) {
    work();
  } else {
    std::vector<std::thread> pool;
    for (int t = 0; t < nt; ++t) pool.emplace_back(work);
    for (auto& t : pool) t.join();
  }
  if (bad.load()) return fail(r, BAMCOLS_ERR_FORMAT, "corrupt BGZF block (inflate failed) before offset %zu", r->cpos);
  r->wend = keep + total;
  clock.lap(0);
  return 0;
}

// Make at least `need` unread bytes available.  Returns 1 if they are, 0 at a clean end of data
// (fewer than `need` bytes left in the whole file), <0 on error.
int ensure_bytes(bamcols* r, size_t need) {
  while (r->wend - r->wpos < need) {
    if (r->file_done) return 0;
    const int rc = refill(r);
    if (rc < 0) return rc;
  }
  return 1;
}

int read_header(bamcols* r) {
  int rc = ensure_bytes(r, 12);
  if (rc < 0) return rc;
  if (rc == 0 || memcmp(r->win.data() + r->wpos, "BAM\1", 4) != 0) return fail(r, BAMCOLS_ERR_FORMAT, "not a BAM stream");
  const size_t l_text = le32(r->win.data() + r->wpos + 4);
  rc = ensure_bytes(r, 12 + l_text);
  if (rc <= 0) return rc < 0 ? rc : fail(r, BAMCOLS_ERR_FORMAT, "truncated BAM header");
  const size_t n_ref = le32(r->win.data() + r->wpos + 8 + l_text);
  r->wpos += 12 + l_text;
  r->ref_names.reserve(n_ref);
  r->ref_lengths.reserve(n_ref);
  for (size_t i = 0; i < n_ref; ++i) {
    rc = ensure_bytes(r, 4);
    if (rc <= 0) return rc < 0 ? rc : fail(r, BAMCOLS_ERR_FORMAT, "truncated BAM reference list");
    const size_t l_name = le32(r->win.data() + r->wpos);
    rc = ensure_bytes(r, 8 + l_name);
    if (rc <= 0) return rc < 0 ? rc : fail(r, BAMCOLS_ERR_FORMAT, "truncated BAM reference list");
    const uint8_t* p = r->win.data() + r->wpos;
    r->ref_names.emplace_back((const char*)p + 4, l_name ? l_name - 1 : 0);
    r->ref_blob.append(r->ref_names.back());
    r->ref_blob.push_back('\0');
    r->ref_lengths.push_back((int32_t)le32(p + 4 + l_name));
    r->wpos += 8 + l_name;
  }
  return 0;
}

// bam_utils.py:301-304: cut the name at the first blank unless the blank is its first character.
inline size_t trimmed_len(const char* s, size_t n) {
  const void* sp = memchr(s, ' ', n);
  if (!sp) return n;
  const size_t i = (const char*)sp - s;
  return i > 0 ? i : n;
}

// 128-bit key of a trimmed read name (bamcols_emit_keys): two multiply-fold hashes with different seeds and
// constants over the 8-byte words of the name (the last one zero-padded), the length folded into both seeds,
// each finished with the murmur3 64-bit mix.  All ones is the empty slot of the device table: mapped away.
inline uint64_t mum64(uint64_t x, uint64_t k) {
  const unsigned __int128 p = (unsigned __int128)x * k;
  return (uint64_t)p ^ (uint64_t)(p >> 64);
}
inline uint64_t fmix64(uint64_t h) {
  h ^= h >> 33;
  h *= 0xff51afd7ed558ccdull;
  h ^= h >> 33;
  h *= 0xc4ceb9fe1a85ec53ull;
  h ^= h >> 33;
  return h;
}
inline void name_key(const char* s, size_t n, uint64_t* lo, uint64_t* hi) {
  uint64_t a = 0x9E3779B97F4A7C15ull ^ ((uint64_t)n * 0xD6E8FEB86659FD93ull);
  uint64_t b = 0x243F6A8885A308D3ull + ((uint64_t)n * 0xA0761D6478BD642Full);
  size_t i = 0;
  for (; i + 8 <= n; i += 8) {
    uint64_t w;
    memcpy(&w, s + i, 8);
    a = mum64(a ^ w, 0xE7037ED1A0B428DBull);
    b = mum64(b ^ w, 0x8EBC6AF09C88C6E3ull) + w;
  }
  if (i < n) {
    uint64_t w = 0;
    memcpy(&w, s + i, n - i);
    a = mum64(a ^ w, 0xE7037ED1A0B428DBull);
    b = mum64(b ^ w, 0x8EBC6AF09C88C6E3ull) + w;
  }
  a = fmix64(a);
  b = fmix64(b);
  if ((a & b) == ~0ull) a = 0;
  *lo = a;
  *hi = b;
}

// Field 14 of name.split('|||') (bam_utils_multisample.py:273): separators are found left to right and
// do not overlap.  false: fewer than 15 fields.
inline bool cell_field_scalar(const char* s, size_t n, const char** out, size_t* len) {
  size_t start = 0, i = 0;
  int seps = 0;
  while (i + 3 <= n) {
    const void* bar = memchr(s + i, '|', n - 2 - i);
    if (!bar) break;
    i = (size_t)((const char*)bar - s);
    if (s[i + 1] == '|' && s[i + 2] == '|') {
      if (seps == 14) {
        *out = s + start;
        *len = i - start;
        return true;
      }
      ++seps;
      i += 3;
      start = i;
    } else {
      ++i;
    }
  }
  if (seps < 14) return false;
  *out = s + start;
  *len = n - start;
  return true;
}

#if defined(__SSE2__)
// Names of up to 128 bytes (all 10x-style names): one bit per '|' from 16-byte compares, then the starts
// of "|||" as m & m>>1 & m>>2, walked greedily.
inline bool cell_field(const char* s, size_t n, const char** out, size_t* len) {
  if (n > 128) return cell_field_scalar(s, n, out, len);
  unsigned __int128 m = 0;
  const __m128i bar = _mm_set1_epi8('|');
  size_t i = 0;
  for (; i + 16 <= n; i += 16) {
    const __m128i v = _mm_loadu_si128((const __m128i*)(s + i));
    m |= (unsigned __int128)(unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(v, bar)) << i;
  }
  if (i < n) {
    char tail[16] = {0};
    memcpy(tail, s + i, n - i);
    const __m128i v = _mm_loadu_si128((const __m128i*)tail);
    m |= (unsigned __int128)(unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(v, bar)) << i;
  }
  unsigned __int128 m3 = m & (m >> 1) & (m >> 2);   // bit p: s[p..p+2] == "|||"
  size_t start = 0;
  int seps = 0;
  uint64_t part[2] = {(uint64_t)m3, (uint64_t)(m3 >> 64)};
  for (int h = 0; h < 2; ++h) {
    uint64_t w = part[h];
    while (w) {
      const size_t p = (size_t)__builtin_ctzll(w) + 64 * (size_t)h;
      w &= w - 1;
      if (p < start) continue;   // overlaps the separator just taken ("||||")
      if (seps == 14) {
        *out = s + start;
        *len = p - start;
        return true;
      }
      ++seps;
      start = p + 3;
    }
  }
  if (seps < 14) return false;
  *out = s + start;
  *len = n - start;
  return true;
}
#else
inline bool cell_field(const char* s, size_t n, const char** out, size_t* len) { return cell_field_scalar(s, n, out, len); }
#endif
inline bool cell_field(const std::string& name, const char** out, size_t* len) {
  return cell_field(name.data(), name.size(), out, len);
}

// Lock-free min / max on plain int32 slots shared by the worker threads (updates are rare after the
// first few alignments of a reference).
inline void note_position(bamcols* r, int32_t tid, int32_t pos) {
  int32_t* lo = &r->range_min[(size_t)tid];
  int32_t* hi = &r->range_max[(size_t)tid];
  int32_t cur = __atomic_load_n(lo, __ATOMIC_RELAXED);
  while (pos < cur && !__atomic_compare_exchange_n(lo, &cur, pos, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
  cur = __atomic_load_n(hi, __ATOMIC_RELAXED);
  while (pos > cur && !__atomic_compare_exchange_n(hi, &cur, pos, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
}

template <class F>
void parallel_for(int nt, F fn) {
  if (nt <= 1) {
    fn(0);
    return;
  }
  std::vector<std::thread> pool;
  for (int t = 0; t < nt; ++t) pool.emplace_back(fn, t);
  for (auto& t : pool) t.join();
}

// ---- record boundaries of the inflated window ---------------------------------------------------------
// BAM records are chained by their block_size fields, so finding them is inherently one sequential hop.
// It is done speculatively in parallel: the window is cut into byte segments, every worker GUESSES the
// first record start of its segment (two consecutive plausible record headers) and hops from there; then
// one pass joins the chains: a chain is accepted from the first of its offsets that the already verified
// chain in front of it lands on - from a true record start the hop is deterministic, so everything after
// that offset is exact.  A segment whose guess is not confirmed is hopped again sequentially.  The result
// is always the list the sequential hop would produce.
#define HOP_END 1   // a partial record (or fewer than 4 bytes) at the landing position: end of the whole records
#define HOP_BAD 2   // block_size < 32 at the landing position

int hop_chain(const uint8_t* base, size_t p, size_t limit, size_t wend, std::vector<size_t>& out, size_t* land) {
  while (p < limit) {
    if (p + 4 > wend) {
      *land = p;
      return HOP_END;
    }
    const size_t bs = le32(base + p);
    if (bs < 32) {
      *land = p;
      return HOP_BAD;
    }
    if (p + 4 + bs > wend) {
      *land = p;
      return HOP_END;
    }
    out.push_back(p);
    p += 4 + bs;
  }
  *land = p;
  return 0;
}

// Could a record start at q?  (A heuristic: wrong answers cost time, never correctness.)
inline bool plausible_record(const uint8_t* base, size_t q, size_t wend, int32_t n_ref) {
  if (q + 36 > wend) return false;
  const size_t bs = le32(base + q);
  if (bs < 34 || bs > (1u << 26)) return false;
  const uint8_t* c = base + q + 4;
  const int32_t tid = (int32_t)le32(c), pos = (int32_t)le32(c + 4), ntid = (int32_t)le32(c + 20);
  const size_t l_name = c[8], n_cigar = le16(c + 12);
  const uint32_t l_seq = le32(c + 16);
  if (tid < -1 || tid >= n_ref || ntid < -1 || ntid >= n_ref || pos < -1 || l_name == 0) return false;
  if (l_seq > bs || 32 + l_name + 4 * n_cigar + (size_t)(l_seq + 1) / 2 + l_seq > bs) return false;
  if (q + 36 + l_name > wend) return true;   // the name lies beyond the window: cannot say more
  const uint8_t* nm = c + 32;
  if (nm[l_name - 1] != 0) return false;
  for (size_t i = 0; i + 1 < l_name; ++i)
    if (nm[i] < 0x20 || nm[i] > 0x7e) return false;
  return true;
}

struct HopChain {
  std::vector<size_t> off;
  size_t start = SIZE_MAX, land = 0;
  int state = 0;
};

// Offsets of the whole records in [r->wpos, r->wend) into `off`; *next = where the unread rest begins.
int find_records(bamcols* r, std::vector<size_t>& off, size_t* next) {
  off.clear();
  const uint8_t* base = r->win.data();
  const size_t p0 = r->wpos, wend = r->wend;
  const size_t span = wend - p0;
  const int32_t n_ref = (int32_t)r->ref_names.size();
  const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)r->n_threads, span / (r->grain * 48) + 1));
  size_t cur = p0;
  if (T == 1) {
    const int st = hop_chain(base, cur, wend, wend, off, &cur);
    if (st == HOP_BAD) return fail(r, BAMCOLS_ERR_FORMAT, "BAM record with block_size %zu", (size_t)le32(base + cur));
    *next = cur;
    return 0;
  }
  std::vector<size_t> seg(T + 1);
  for (int t = 0; t <= T; ++t) seg[t] = p0 + span * (size_t)t / (size_t)T;
  std::vector<HopChain> chains(T);
  parallel_for(T, [&](int t) {
    HopChain& c = chains[t];
    if (t == 0) {
      c.start = p0;
    } else {
      const size_t stop = std::min(seg[t + 1], seg[t] + (1u << 16));
      for (size_t q = seg[t]; q < stop; ++q) {
        if (!plausible_record(base, q, wend, n_ref)) continue;
        const size_t nx = q + 4 + le32(base + q);
        if (nx + 36 <= wend && !plausible_record(base, nx, wend, n_ref)) continue;
        c.start = q;
        break;
      }
      if (c.start == SIZE_MAX) return;
    }
    c.off.reserve((seg[t + 1] - seg[t]) / 64 + 16);
    c.state = hop_chain(base, c.start, seg[t + 1], wend, c.off, &c.land);
  });
  size_t total = 0;
  for (const HopChain& c : chains) total += c.off.size();
  off.reserve(total + 64);
  for (int t = 0; t < T; ++t) {
    if (cur >= seg[t + 1]) continue;   // a record reaches over this whole segment
    HopChain& c = chains[t];
    int st = 0;
    bool joined = false;
    if (c.start != SIZE_MAX && !c.off.empty()) {
      st = hop_chain(base, cur, c.start, wend, off, &cur);   // the records in front of the guess (usually none)
      if (st == 0) {
        const auto it = std::lower_bound(c.off.begin(), c.off.end(), cur);
        if (it != c.off.end() && *it == cur) {
          off.insert(off.end(), it, c.off.end());
          cur = c.land;
          st = c.state;
          joined = true;
        }
      }
    }
    if (!joined && st == 0) st = hop_chain(base, cur, seg[t + 1], wend, off, &cur);
    if (st == HOP_BAD) return fail(r, BAMCOLS_ERR_FORMAT, "BAM record with block_size %zu", (size_t)le32(base + cur));
    if (st == HOP_END) break;
  }
  *next = cur;
  return 0;
}

// The reference's filter (bam_utils.py:264-270) with the record checks that come with it, for the record whose
// block_size field is at `rec`.  The one statement of the filter on the host; ecb_bam_validity_kernel is the device's.
enum { REC_FILTERED = 0, REC_VALID = 1, REC_BAD_NAME = 2, REC_BAD_TID = 3 };
inline int record_validity(const uint8_t* rec, int32_t n_ref) {
  const size_t bs = le32(rec);
  const uint8_t* q = rec + 4;
  const int32_t tid = (int32_t)le32(q);
  const size_t l_name = q[8];
  const uint32_t flag = le16(q + 14);
  const int32_t ntid = (int32_t)le32(q + 20), npos = (int32_t)le32(q + 24);
  if (32 + l_name > bs || l_name == 0) return REC_BAD_NAME;
  if (flag & 0x4) return REC_FILTERED;
  if ((flag & 0x1) && ((flag & 0x80) || !(flag & 0x2) || tid != ntid || npos < 0)) return REC_FILTERED;
  if (tid < 0 || tid >= n_ref) return REC_BAD_TID;
  return REC_VALID;
}

// fn(column) for every staged column of the reader's mode, in the order of the caller's buffers:
// read_group or the two key halves, target_idx, hap_idx, and cell_idx in per-cell mode.
template <class F>
void for_staged(bamcols* r, F fn) {
  if (r->mode == 3) {
    fn(r->st_klo);
    fn(r->st_khi);
  } else {
    fn(r->st_rg);
  }
  fn(r->st_tg);
  fn(r->st_hp);
  if (r->mode == 2) fn(r->st_cell);
}

// The whole records of one inflated window after the validity pass.  Worker t of nt takes the records
// [lo(t), lo(t + 1)); their valid ones become rows n_valid[t] ... n_valid[t + 1] - 1 of the window, and in the
// read-group modes they open reads n_start[t] + 1 ... n_start[t + 1], counted from the read that is open when
// the window begins.
struct Window {
  const uint8_t* base;
  const std::vector<size_t>& off;
  std::vector<uint8_t>& fl;   // bit 0 valid, bit 3 starts a read (per-cell: bits 1 and 2 hold its two comparisons)
  size_t n;
  int nt;
  std::vector<size_t> n_valid, n_start;
  size_t lo(int t) const { return n * (size_t)t / (size_t)nt; }
};

// Single-sample read starts (bam_utils.py:301-306): a valid record starts a read iff its trimmed name differs
// from the previous valid record's; the last valid record's trimmed name is remembered for the next window.
void single_starts(bamcols* r, Window& w) {
  const uint8_t* base = w.base;
  std::vector<uint8_t>& fl = w.fl;
  const bool had_prev = r->started;
  const std::string& prev_name = r->current;
  parallel_for(w.nt, [&](int t) {
    const char* pn = nullptr;  // trimmed name of the previous valid record
    size_t pl = 0;
    bool have = false;
    for (size_t j = w.lo(t); j-- > 0;)
      if (fl[j]) {
        const uint8_t* q = base + w.off[j] + 4;
        pn = (const char*)q + 32;
        pl = trimmed_len(pn, (size_t)q[8] - 1);
        have = true;
        break;
      }
    if (!have && had_prev) {
      pn = prev_name.data();
      pl = prev_name.size();
      have = true;
    }
    size_t cnt = 0;
    for (size_t i = w.lo(t); i < w.lo(t + 1); ++i) {
      if (!fl[i]) continue;
      const uint8_t* q = base + w.off[i] + 4;
      const char* nm = (const char*)q + 32;
      const size_t nl = trimmed_len(nm, (size_t)q[8] - 1);
      if (!have || nl != pl || memcmp(nm, pn, nl) != 0) {
        fl[i] |= 8;
        ++cnt;
      }
      pn = nm;
      pl = nl;
      have = true;
    }
    w.n_start[t + 1] = cnt;
  });
  for (int t = 0; t < w.nt; ++t) w.n_start[t + 1] += w.n_start[t];
  for (size_t j = w.n; j-- > 0;)
    if (fl[j]) {
      const uint8_t* q = base + w.off[j] + 4;
      const char* nm = (const char*)q + 32;
      r->current.assign(nm, trimmed_len(nm, (size_t)q[8] - 1));
      break;
    }
}

// Per-cell rules (bam_utils_multisample.py:258-300) over the valid records of the window, in parallel except
// for two cheap sequential passes.  With P the previous valid record, a record B starts a read iff the
// remembered name differs from trim(B), and the remembered name is
//   - trim(first record of the file) until the first switch,
//   - the UNTRIMMED name of the record that made the last switch (:292) afterwards,
// which, because every record inside a read matches the remembered name, is trim(P) if P did not switch and P's
// untrimmed name if it did.  So both outcomes are computed per record in parallel ("differs from trim(P)",
// "differs from P untrimmed") and one pass over two bits per record picks.
// The cell of a read is field 14 of its remembered name, looked up when the NEXT valid alignment arrives
// (dictionary ids follow that order; a read that ends the file alone is never looked up).  Leaves the cell of
// the window's k-th read in sc_group_cell[k] (k = 0: the read open when the window begins).
int cell_starts(bamcols* r, bamcols_cells* cells, Window& w, size_t row0) {
  const uint8_t* base = w.base;
  const std::vector<size_t>& off = w.off;
  std::vector<uint8_t>& fl = w.fl;
  const size_t n = w.n;
  const int nt = w.nt;
  std::vector<size_t>& n_start = w.n_start;
  auto lo = [&](int t) { return w.lo(t); };
  auto name_of = [&](size_t i, const char** nm, size_t* full, size_t* trimmed) {
    const uint8_t* q = base + off[i] + 4;
    *nm = (const char*)q + 32;
    *full = (size_t)q[8] - 1;
    *trimmed = trimmed_len(*nm, *full);
  };

  // both comparison outcomes per valid record, against the previous valid record of the window
  parallel_for(nt, [&](int t) {
    const char* pn = nullptr;
    size_t pf = 0, pt = 0;
    bool have = false;
    for (size_t j = lo(t); j-- > 0;)
      if (fl[j]) {
        name_of(j, &pn, &pf, &pt);
        have = true;
        break;
      }
    for (size_t i = lo(t); i < lo(t + 1); ++i) {
      if (!fl[i]) continue;
      const char* nm;
      size_t nf, ntm;
      name_of(i, &nm, &nf, &ntm);
      if (have) {
        if (ntm != pt || memcmp(nm, pn, ntm) != 0) fl[i] |= 2;   // differs from trim(P)
        if (ntm != pf || memcmp(nm, pn, ntm) != 0) fl[i] |= 4;   // differs from P untrimmed
      }
      pn = nm;
      pf = nf;
      pt = ntm;
      have = true;
    }
  });

  // Which records start a read (bit 3), openers in order.  After the first two valid records of the
  // window (the file's first read is remembered trimmed, :261-262) the rule is a two-state machine:
  // sw(i) = sw(previous valid record) ? bit 2 : bit 1.  Every worker runs its range for both incoming
  // states, the states are chained over the workers, then every worker runs its range again for real.
  std::vector<size_t>& openers = r->sc_openers;
  {
    size_t i0 = n, i1 = n;   // first and second valid record of the window
    for (size_t i = 0; i < n; ++i)
      if (fl[i]) {
        if (i0 == n) {
          i0 = i;
        } else {
          i1 = i;
          break;
        }
      }
    bool sw0, sw1 = false;
    if (!r->started) {
      sw0 = true;                                    // the file's first read
    } else {
      const char* nm;
      size_t nf, ntm;
      name_of(i0, &nm, &nf, &ntm);
      sw0 = r->current.size() != ntm || memcmp(r->current.data(), nm, ntm) != 0;
    }
    if (i1 < n) {
      const bool prev_trimmed_name = sw0 && !r->started;   // only the first read is remembered trimmed
      sw1 = (sw0 && !prev_trimmed_name) ? (fl[i1] & 4) != 0 : (fl[i1] & 2) != 0;
    }
    std::vector<uint8_t> out0(nt, 0), out1(nt, 1), in_state(nt, 0);
    parallel_for(nt, [&](int t) {
      bool s0 = false, s1 = true;
      for (size_t i = std::max(lo(t), i1 == n ? n : i1 + 1); i < lo(t + 1); ++i) {
        const uint8_t f = fl[i];
        if (!f) continue;
        s0 = s0 ? (f & 4) != 0 : (f & 2) != 0;
        s1 = s1 ? (f & 4) != 0 : (f & 2) != 0;
      }
      out0[t] = s0;
      out1[t] = s1;
    });
    {
      bool cur = sw1;
      for (int t = 0; t < nt; ++t) {
        in_state[t] = cur;
        cur = cur ? out1[t] != 0 : out0[t] != 0;
      }
    }
    std::vector<std::vector<size_t>>& mine = r->sc_mine;
    if ((int)mine.size() < nt) mine.resize(nt);
    parallel_for(nt, [&](int t) {
      std::vector<size_t>& op = mine[t];
      op.clear();
      bool st = in_state[t] != 0;
      for (size_t i = lo(t); i < lo(t + 1); ++i) {
        const uint8_t f = fl[i];
        if (!f) continue;
        bool sw;
        if (i == i0) {
          sw = sw0;
        } else if (i == i1) {
          sw = sw1;
        } else if (i < i1) {
          continue;   // unreachable: no valid record lies between i0 and i1
        } else {
          sw = st ? (f & 4) != 0 : (f & 2) != 0;
          st = sw;
        }
        if (sw) {
          fl[i] = f | 8;
          op.push_back(i);
        }
      }
    });
    for (int t = 0; t < nt; ++t) n_start[t + 1] = n_start[t] + mine[t].size();
    openers.resize(n_start[nt]);
    parallel_for(nt, [&](int t) {
      if (!mine[t].empty()) memcpy(openers.data() + n_start[t], mine[t].data(), mine[t].size() * sizeof(size_t));
    });
  }
  size_t last_valid = n;
  for (size_t j = n; j-- > 0;)
    if (fl[j]) {
      last_valid = j;
      break;
    }

  if (r->pending) {   // the read that was open alone at the end of the previous window: this window has a valid record
    const char* cf;
    size_t cl;
    if (!cell_field(r->current, &cf, &cl)) return fail(r, BAMCOLS_ERR_CELL_FIELD, "list index out of range");
    r->cell = cells->id_of(cf, cl);
    r->st_cell[r->pending_row] = r->cell;
    r->pending = false;
  }

  // cell names of the openers (field 14 of the remembered name), in parallel, looked up in the dictionary
  // as it stands now; only cells that are NEW in this window go through the ordered pass below
  const size_t n_open = openers.size();
  std::vector<const char*>& cell_ptr = r->sc_cell_ptr;
  std::vector<size_t>& cell_len = r->sc_cell_len;
  std::vector<uint64_t>& cell_hash = r->sc_cell_hash;
  std::vector<int32_t>& cell_id = r->sc_cell_id;   // -2 no field 14, -1 not in the dictionary yet
  if (cell_ptr.size() < n_open) {
    cell_ptr.resize(n_open);
    cell_len.resize(n_open);
    cell_hash.resize(n_open);
    cell_id.resize(n_open);
  }
  const bamcols_cells* snapshot = cells;
  const bool file_first_here = !r->started;
  {
    const int nto = (int)std::max<size_t>(1, std::min<size_t>((size_t)r->n_threads, n_open / r->grain + 1));
    parallel_for(nto, [&](int t) {
      for (size_t k = n_open * (size_t)t / (size_t)nto; k < n_open * (size_t)(t + 1) / (size_t)nto; ++k) {
        const char* nm;
        size_t nf, ntm;
        name_of(openers[k], &nm, &nf, &ntm);
        const size_t len = (file_first_here && k == 0) ? ntm : nf;   // remembered name of that read
        const char* cf;
        size_t cl;
        cell_id[k] = -2;
        if (!cell_field(nm, len, &cf, &cl)) continue;
        cell_ptr[k] = cf;
        cell_len[k] = cl;
        cell_hash[k] = bamcols_cells::hash_of(cf, cl);
        cell_id[k] = snapshot->find(cf, cl, cell_hash[k]);
      }
    });
  }

  // dictionary pass, in the order the reference resolves cells
  std::vector<int32_t>& group_cell = r->sc_group_cell;
  if (group_cell.size() < n_open + 1) group_cell.resize(n_open + 1);
  group_cell[0] = r->cell;   // the read that is open when the window begins
  bool pending_now = false;
  for (size_t k = 0; k < n_open; ++k) {
    const bool first_of_file = file_first_here && k == 0;
    if (!first_of_file && openers[k] == last_valid) {   // alone at the end of the window: resolved later, or never
      pending_now = true;
      group_cell[k + 1] = 0;
      continue;
    }
    if (cell_id[k] == -2) return fail(r, BAMCOLS_ERR_CELL_FIELD, "list index out of range");
    group_cell[k + 1] = cell_id[k] >= 0 ? cell_id[k] : cells->id_of(cell_ptr[k], cell_len[k], cell_hash[k]);
  }
  if (n_open) {
    const char* nm;
    size_t nf, ntm;
    name_of(openers[n_open - 1], &nm, &nf, &ntm);
    r->current.assign(nm, (file_first_here && n_open == 1) ? ntm : nf);
    r->cell = group_cell[n_open];
    r->pending = pending_now;
    if (pending_now) r->pending_row = row0 + w.n_valid[nt] - 1;   // that read's only row is the window's last row
  }
  return 0;
}

// Rows of the read-group modes, written at their final positions: read_group counts on from the read open
// when the window begins; per-cell mode adds the cell of each read (cell_starts).
template <bool CELLS>
void group_rows(bamcols* r, const Window& w, size_t row0) {
  const int64_t group0 = r->group;
  int32_t* rg = r->st_rg.data() + row0;
  int32_t* tg = r->st_tg.data() + row0;
  int32_t* hp = r->st_hp.data() + row0;
  int32_t* cc = CELLS ? r->st_cell.data() + row0 : nullptr;
  const int32_t* group_cell = r->sc_group_cell.data();
  parallel_for(w.nt, [&](int t) {
    size_t k = w.n_valid[t];
    size_t g = w.n_start[t];
    for (size_t i = w.lo(t); i < w.lo(t + 1); ++i) {
      if (!w.fl[i]) continue;
      if (w.fl[i] & 8) ++g;
      const int32_t tid = (int32_t)le32(w.base + w.off[i] + 4);
      rg[k] = (int32_t)(group0 + (int64_t)g);
      tg[k] = r->tid_target[tid];
      hp[k] = r->tid_hap[tid];
      if (CELLS) cc[k] = group_cell[g];
      ++k;
    }
  });
  r->group = group0 + (int64_t)w.n_start[w.nt];
}

// Rows of name-key mode (bamcols_emit_keys): every valid record gets the 128-bit key of its trimmed name in
// place of a read_group.
void key_rows(bamcols* r, const Window& w, size_t row0) {
  uint64_t* klo = r->st_klo.data() + row0;
  uint64_t* khi = r->st_khi.data() + row0;
  int32_t* tg = r->st_tg.data() + row0;
  int32_t* hp = r->st_hp.data() + row0;
  parallel_for(w.nt, [&](int t) {
    size_t k = w.n_valid[t];
    for (size_t i = w.lo(t); i < w.lo(t + 1); ++i) {
      if (!w.fl[i]) continue;
      const uint8_t* q = w.base + w.off[i] + 4;
      const char* nm = (const char*)q + 32;
      name_key(nm, trimmed_len(nm, (size_t)q[8] - 1), &klo[k], &khi[k]);
      const int32_t tid = (int32_t)le32(q);
      tg[k] = r->tid_target[tid];
      hp[k] = r->tid_hap[tid];
      ++k;
    }
  });
}

// End of the whole reads among the staged rows: everything before the first row of the last read.
size_t whole_reads_end(const bamcols* r) {
  size_t w = r->st_rg.size();
  const int32_t last = r->st_rg[w - 1];
  while (w > 0 && r->st_rg[w - 1] == last) --w;
  return w;
}

// The rules of the reader's mode over every whole record of the inflated window, on all worker threads:
// (1) the record boundaries (find_records), (2) validity per record, (3) per mode: "starts a read" per valid
// record, or nothing in name-key mode, (4) rows written at their final positions (prefix sums over the threads).
// The open last read is held back (st_whole) until the next window or the end of the file closes it; name-key
// mode has no reads to keep whole and hands out every row at once.
int process_window(bamcols* r, bamcols_cells* cells) {
  // rows still waiting from the previous window go to the front
  const size_t left = r->st_tg.size() - r->st_pos;
  for_staged(r, [&](auto& buf) {
    if (r->st_pos > 0) memmove(buf.data(), buf.data() + r->st_pos, left * sizeof(buf[0]));
    buf.resize(left);
  });
  r->st_whole -= r->st_pos;
  if (r->pending) r->pending_row -= r->st_pos;
  r->st_pos = 0;

  // (1) records of the window
  if (r->wend - r->wpos < 4 || r->wend - r->wpos < 4 + (size_t)le32(r->win.data() + r->wpos)) {
    const int rc = refill(r);
    if (rc < 0) return rc;
  }
  PhaseClock clock(r->phase_s);
  std::vector<size_t>& off = r->rec_off;
  size_t p = r->wpos;
  {
    const int rc = find_records(r, off, &p);
    if (rc < 0) return rc;
  }
  r->wpos = p;
  clock.lap(1);
  const size_t n = off.size();
  if (n == 0) {
    if (r->file_done) {
      if (r->wend != r->wpos) return fail(r, BAMCOLS_ERR_FORMAT, "truncated BAM record at the end of the file");
      r->records_done = true;
      r->st_whole = r->st_tg.size();  // the end of the file closes the last read
    }
    return 0;
  }
  r->all_alignments += (int64_t)n;
  r->rec_flag.assign(n, 0);
  const int nt = (int)std::max<size_t>(1, std::min<size_t>((size_t)r->n_threads, n / r->grain + 1));
  Window w{r->win.data(), off, r->rec_flag, n, nt, std::vector<size_t>(nt + 1, 0), std::vector<size_t>(nt + 1, 0)};

  // (2) validity
  const int32_t n_ref = (int32_t)r->tid_target.size();
  std::atomic<int> bad(0);
  parallel_for(nt, [&](int t) {
    size_t cnt = 0;
    for (size_t i = w.lo(t); i < w.lo(t + 1); ++i) {
      const uint8_t* rec = w.base + off[i];
      const int v = record_validity(rec, n_ref);
      if (v != REC_VALID) {
        if (v != REC_FILTERED) bad.store(v);
        continue;
      }
      if (r->track_ranges) note_position(r, (int32_t)le32(rec + 4), (int32_t)le32(rec + 8));
      w.fl[i] = 1;
      ++cnt;
    }
    w.n_valid[t + 1] = cnt;
  });
  if (bad.load() == REC_BAD_NAME) return fail(r, BAMCOLS_ERR_FORMAT, "BAM record with a bad read-name length");
  if (bad.load() == REC_BAD_TID)
    return fail(r, BAMCOLS_ERR_TID, "alignment with a reference id outside the header's %d references", n_ref);
  for (int t = 0; t < nt; ++t) w.n_valid[t + 1] += w.n_valid[t];
  const size_t rows = w.n_valid[nt];
  clock.lap(2);
  if (rows == 0) return 0;
  const size_t row0 = r->st_tg.size();
  for_staged(r, [&](auto& buf) { buf.resize(row0 + rows); });

  if (r->mode == 3) {   // (4) rows: name keys instead of read starts
    key_rows(r, w, row0);
    r->st_whole = r->st_tg.size();
    clock.lap(4);
    return 0;
  }
  // (3) read starts; per-cell mode also resolves the cells here
  if (r->mode == 2) {
    const int rc = cell_starts(r, cells, w, row0);
    if (rc < 0) return rc;
  } else {
    single_starts(r, w);
  }
  clock.lap(3);
  // (4) rows
  if (r->mode == 2) group_rows<true>(r, w, row0); else group_rows<false>(r, w, row0);
  r->started = true;
  r->st_whole = whole_reads_end(r);
  clock.lap(4);
  return 0;
}

// Hands the staged rows of the reader's mode to the caller's buffers dst[] (in for_staged order) until they are
// full or the file ends.  In the read-group modes a call stops at the start of a read, so no read is split
// between two calls.
int64_t emit_rows(bamcols* r, bamcols_cells* cells, void* const* dst, int64_t capacity, int* done) {
  int64_t rows = 0;
  for (;;) {
    const size_t avail = r->st_whole - r->st_pos;
    if (avail > 0) {
      size_t take = std::min<size_t>(avail, (size_t)(capacity - rows));
      if (take < avail && r->mode != 3)  // stop at the start of a read
        while (take > 0 && r->st_rg[r->st_pos + take] == r->st_rg[r->st_pos + take - 1]) --take;
      if (take == 0) {
        if (rows == 0) return fail(r, BAMCOLS_ERR_INVALID, "a read has more alignments than the buffers hold (%lld rows)", (long long)capacity);
        return rows;
      }
      PhaseClock clock(r->phase_s);
      // columns x slices on the worker threads (one memcpy stream does not fill the memory system)
      uint8_t* to[4];
      const uint8_t* from[4];
      size_t width[4];
      int ncol = 0;
      for_staged(r, [&](auto& buf) {
        width[ncol] = sizeof(buf[0]);
        to[ncol] = (uint8_t*)dst[ncol] + (size_t)rows * width[ncol];
        from[ncol] = (const uint8_t*)(buf.data() + r->st_pos);
        ++ncol;
      });
      if (take < (1u << 18)) {   // small: not worth a thread
        for (int c = 0; c < ncol; ++c) memcpy(to[c], from[c], take * width[c]);
      } else {
        const int slices = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(1, r->n_threads / ncol), take / (1u << 18)));
        parallel_for(ncol * slices, [&](int t) {
          const int c = t / slices, k = t % slices;
          const size_t a = take * (size_t)k / (size_t)slices, b = take * (size_t)(k + 1) / (size_t)slices;
          memcpy(to[c] + a * width[c], from[c] + a * width[c], (b - a) * width[c]);
        });
      }
      clock.lap(5);
      rows += (int64_t)take;
      r->st_pos += take;
      if (rows == capacity) return rows;
      continue;
    }
    if (r->records_done) {
      *done = 1;
      return rows;
    }
    const int rc = process_window(r, cells);
    if (rc < 0) return rc;
  }
}

}  // namespace

extern "C" {

const char* bamcols_last_error(const bamcols* r) { return r ? r->err.c_str() : g_open_error.c_str(); }

int bamcols_open(bamcols** out, const char* path, int n_threads) {
  if (!out || !path) return fail(nullptr, BAMCOLS_ERR_INVALID, "NULL argument");
  *out = nullptr;
  bamcols* r = new bamcols();
  auto bail = [&](int code) {
    g_open_error = r->err;
    bamcols_close(r);
    return code;
  };
  r->fd = open(path, O_RDONLY);
  if (r->fd < 0) {
    fail(r, BAMCOLS_ERR_IO, "cannot open %s", path);
    return bail(BAMCOLS_ERR_IO);
  }
  struct stat st;
  if (fstat(r->fd, &st) != 0 || st.st_size <= 0) {
    fail(r, BAMCOLS_ERR_IO, "cannot stat %s (or it is empty)", path);
    return bail(BAMCOLS_ERR_IO);
  }
  r->file_size = (size_t)st.st_size;
  void* m = mmap(nullptr, r->file_size, PROT_READ, MAP_PRIVATE, r->fd, 0);
  if (m == MAP_FAILED) {
    fail(r, BAMCOLS_ERR_IO, "cannot mmap %s", path);
    return bail(BAMCOLS_ERR_IO);
  }
  r->file = (const uint8_t*)m;
  madvise(m, r->file_size, MADV_SEQUENTIAL);
  if (const char* b = getenv("BAMCOLS_BATCH_BLOCKS")) r->batch_blocks = (size_t)std::max(1L, atol(b));  // tests: many small windows
  if (const char* g = getenv("BAMCOLS_GRAIN")) r->grain = (size_t)std::max(1L, atol(g));  // tests: split tiny inputs too
  const unsigned hw = std::thread::hardware_concurrency();
  r->n_threads = n_threads > 0 ? n_threads : (hw ? (int)hw : 1);
  if (r->file_size < 4 || r->file[0] != 0x1f || r->file[1] != 0x8b) {
    fail(r, BAMCOLS_ERR_FORMAT, "File %s is not a BAM file", path);
    return bail(BAMCOLS_ERR_FORMAT);
  }
  // the header rarely needs more than a few blocks: start with a small batch
  const size_t full_batch = r->batch_blocks;
  r->batch_blocks = 16;
  const int rc = read_header(r);
  r->batch_blocks = full_batch;
  if (rc < 0) return bail(rc);
  {
    // virtual offset of the first record: hop over the blocks of the batch that holds the window position
    size_t c = r->last_batch_c0, w = r->last_batch_keep;
    for (;;) {
      BlockJob job;
      size_t bsize = 0;
      const int prc = parse_block(r, c, &job, &bsize);
      if (prc != 0 || w + job.isize > r->wpos || (w + job.isize == r->wpos && c + bsize >= r->cpos)) break;
      w += job.isize;
      c += bsize;
    }
    r->first_voffset = (int64_t)((c << 16) | (r->wpos - w));
  }
  r->prefetch = std::thread([r]() { r->prefetch_rc = refill(r); });
  *out = r;
  return BAMCOLS_OK;
}

void bamcols_close(bamcols* r) {
  if (!r) return;
  if (r->prefetch.joinable()) r->prefetch.join();
  if (r->file) munmap(const_cast<uint8_t*>(r->file), r->file_size);
  if (r->fd >= 0) close(r->fd);
  delete r;
}

int bamcols_n_references(const bamcols* r) { return r ? (int)r->ref_names.size() : (int64_t)BAMCOLS_ERR_INVALID; }

const char* bamcols_reference_name(const bamcols* r, int tid) {
  if (!r || tid < 0 || (size_t)tid >= r->ref_names.size()) return nullptr;
  return r->ref_names[tid].c_str();
}

int64_t bamcols_reference_blob(const bamcols* r, const char** names, const int32_t** lengths) {
  if (!r || !names || !lengths) return BAMCOLS_ERR_INVALID;
  *names = r->ref_blob.data();
  *lengths = r->ref_lengths.data();
  return (int64_t)r->ref_blob.size();
}

int bamcols_reference_length(const bamcols* r, int tid) {
  if (!r || tid < 0 || (size_t)tid >= r->ref_lengths.size()) return BAMCOLS_ERR_INVALID;
  return r->ref_lengths[tid];
}

int bamcols_set_tables(bamcols* r, const int32_t* tid_target, const int32_t* tid_hap, int n_references) {
  if (!r || !tid_target || !tid_hap) return BAMCOLS_ERR_INVALID;
  if ((size_t)n_references != r->ref_names.size())
    return fail(r, BAMCOLS_ERR_INVALID, "tables have %d entries, the header has %zu references", n_references,
                r->ref_names.size());
  r->tid_target.assign(tid_target, tid_target + n_references);
  r->tid_hap.assign(tid_hap, tid_hap + n_references);
  return BAMCOLS_OK;
}

// Header -> tables (alntools/bam_utils.py:561-633; alntools_b200/header.py is the readable statement):
// every @SQ name is split at its LAST '_' (unless that is its first character) into main target and
// haplotype; main targets are numbered target-file ids first, then in header order; haplotypes are
// sorted; lengths[target][haplotype] = reference length.  first_targets: the target file's ids, each
// followed by a NUL (may be empty).
// Distinct strings in order of first appearance -> dense ids.  Open addressing over views into memory the
// caller keeps alive (the reference names, the target list): no per-name allocation.
struct ViewIds {
  std::vector<std::string_view> views;
  std::vector<int32_t> slot;   // -1 = empty
  size_t mask = 0;
  explicit ViewIds(size_t expect) {
    size_t cap = 16;
    while (cap < 2 * expect + 16) cap <<= 1;
    slot.assign(cap, -1);
    mask = cap - 1;
    views.reserve(expect);
  }
  int32_t id_of(std::string_view v) {
    if ((views.size() + 1) * 2 > mask + 1) {   // grow (only when `expect` was too small)
      std::vector<int32_t> bigger((mask + 1) * 2, -1);
      const size_t m2 = bigger.size() - 1;
      for (size_t i = 0; i < views.size(); ++i) {
        size_t j = bamcols_cells::hash_of(views[i].data(), views[i].size()) & m2;
        while (bigger[j] >= 0) j = (j + 1) & m2;
        bigger[j] = (int32_t)i;
      }
      slot.swap(bigger);
      mask = m2;
    }
    size_t j = bamcols_cells::hash_of(v.data(), v.size()) & mask;
    for (; slot[j] >= 0; j = (j + 1) & mask)
      if (views[(size_t)slot[j]] == v) return slot[j];
    slot[j] = (int32_t)views.size();
    views.push_back(v);
    return slot[j];
  }
};

int bamcols_build_tables(bamcols* r, const char* first_targets, int64_t first_len) {
  if (!r || first_len < 0 || (first_len > 0 && !first_targets)) return BAMCOLS_ERR_INVALID;
  const size_t n = r->ref_names.size();
  // main targets: the target list first, then unseen targets in header order (bam_utils.py:571-598)
  ViewIds targets(n);
  for (int64_t p = 0; p < first_len;) {
    const size_t l = strnlen(first_targets + p, (size_t)(first_len - p));
    targets.id_of(std::string_view(first_targets + p, l));
    p += (int64_t)l + 1;
  }
  // target / haplotype of every reference: split at the last '_' unless it is the first character (:584-591)
  ViewIds hap_seen(64);
  std::vector<int32_t> tt(n), hraw(n);
  for (size_t i = 0; i < n; ++i) {
    const std::string& name = r->ref_names[i];
    const size_t cut = name.rfind('_');
    if (cut != std::string::npos && cut > 0) {
      tt[i] = targets.id_of(std::string_view(name.data(), cut));
      hraw[i] = hap_seen.id_of(std::string_view(name.data() + cut + 1, name.size() - cut - 1));
    } else {
      tt[i] = targets.id_of(std::string_view(name));
      hraw[i] = hap_seen.id_of(std::string_view());
    }
  }
  // haplotypes = sorted(set) (:602): ids of the distinct ones in sorted order
  const size_t T = targets.views.size(), H = hap_seen.views.size();
  std::vector<int32_t> order(H), rank(H);
  for (size_t h = 0; h < H; ++h) order[h] = (int32_t)h;
  std::sort(order.begin(), order.end(), [&](int32_t x, int32_t y) { return hap_seen.views[(size_t)x] < hap_seen.views[(size_t)y]; });
  for (size_t k = 0; k < H; ++k) rank[(size_t)order[k]] = (int32_t)k;
  std::vector<int32_t> th(n);
  std::vector<int32_t> owner(T * H, -1);
  r->tb_lengths.assign(T * H, 0);
  for (size_t i = 0; i < n; ++i) {
    th[i] = rank[(size_t)hraw[i]];
    int32_t& o = owner[(size_t)tt[i] * H + (size_t)th[i]];
    if (o >= 0)
      return fail(r, BAMCOLS_ERR_INVALID, "@SQ names '%s' and '%s' map to the same (target, haplotype)",
                  r->ref_names[(size_t)o].c_str(), r->ref_names[i].c_str());
    o = (int32_t)i;
    r->tb_lengths[(size_t)tt[i] * H + (size_t)th[i]] = r->ref_lengths[i];
  }
  r->tb_targets.clear();
  size_t bytes = 0;
  for (const std::string_view& t : targets.views) bytes += t.size() + 1;
  r->tb_targets.reserve(bytes);
  for (const std::string_view& t : targets.views) {
    r->tb_targets.append(t.data(), t.size());
    r->tb_targets.push_back('\0');
  }
  r->tb_haps.clear();
  for (size_t k = 0; k < H; ++k) {
    const std::string_view& h = hap_seen.views[(size_t)order[k]];
    r->tb_haps.append(h.data(), h.size());
    r->tb_haps.push_back('\0');
  }
  r->tb_n_targets = (int32_t)T;
  r->tb_n_haps = (int32_t)H;
  r->tid_target = std::move(tt);
  r->tid_hap = std::move(th);
  return BAMCOLS_OK;
}

int bamcols_tables(const bamcols* r, int32_t* n_targets, int32_t* n_haps, const char** targets, int64_t* targets_len,
                   const char** haps, int64_t* haps_len, const int32_t** tid_target, const int32_t** tid_hap,
                   const int32_t** lengths) {
  if (!r || !n_targets || !n_haps || !targets || !targets_len || !haps || !haps_len || !tid_target || !tid_hap || !lengths)
    return BAMCOLS_ERR_INVALID;
  *n_targets = r->tb_n_targets;
  *n_haps = r->tb_n_haps;
  *targets = r->tb_targets.data();
  *targets_len = (int64_t)r->tb_targets.size();
  *haps = r->tb_haps.data();
  *haps_len = (int64_t)r->tb_haps.size();
  *tid_target = r->tid_target.data();
  *tid_hap = r->tid_hap.data();
  *lengths = r->tb_lengths.data();
  return BAMCOLS_OK;
}

int64_t bamcols_target_section(bamcols* r, const char** bytes) {
  if (!r || !bytes) return BAMCOLS_ERR_INVALID;
  if (r->tb_n_targets == 0 && r->tb_targets.empty()) return fail(r, BAMCOLS_ERR_INVALID, "bamcols_build_tables was not called");
  // T x [len(name), name bytes, H x length], little-endian int32s (alntools/bin_utils.py:153-159)
  std::string& out = r->tb_section;
  out.clear();
  const size_t H = (size_t)r->tb_n_haps;
  out.reserve(r->tb_targets.size() + (size_t)r->tb_n_targets * (4 + 4 * H));
  auto put32 = [&](uint32_t v) {
    const char b[4] = {(char)(v & 0xFF), (char)((v >> 8) & 0xFF), (char)((v >> 16) & 0xFF), (char)((v >> 24) & 0xFF)};
    out.append(b, 4);
  };
  // the reference writes len(name) in CHARACTERS in front of the UTF-8 bytes: only for ASCII names is that the
  // byte count, anything else is left to the caller (who reproduces the reference's bytes in Python)
  for (const char ch : r->tb_targets)
    if ((unsigned char)ch >= 0x80) return 0;
  const char* p = r->tb_targets.data();
  for (int32_t t = 0; t < r->tb_n_targets; ++t) {
    const size_t l = strlen(p);
    put32((uint32_t)l);
    out.append(p, l);
    for (size_t h = 0; h < H; ++h) put32((uint32_t)r->tb_lengths[(size_t)t * H + h]);
    p += l + 1;
  }
  *bytes = out.data();
  return (int64_t)out.size();
}

int bamcols_cells_create(bamcols_cells** out) {
  if (!out) return BAMCOLS_ERR_INVALID;
  *out = new bamcols_cells();
  return BAMCOLS_OK;
}
void bamcols_cells_destroy(bamcols_cells* c) { delete c; }
int64_t bamcols_cells_count(const bamcols_cells* c) { return c ? (int64_t)c->names.size() : (int64_t)BAMCOLS_ERR_INVALID; }
const char* bamcols_cells_name(const bamcols_cells* c, int64_t idx) {
  if (!c || idx < 0 || (size_t)idx >= c->names.size()) return nullptr;
  return c->names[(size_t)idx].c_str();
}

// ---- shards of ONE file (SURVEY 8f N3: what alntools/bam_utils.py:1174-1304 plans and :157-195 copies into
// temporary BAM files is here a list of virtual offsets; nothing is copied) --------------------------------
namespace {

// First BGZF block boundary at or behind `from`: the magic bytes, a header that parses, and two more blocks
// (or the end of the file) chained behind it.
size_t find_block_boundary(bamcols* r, size_t from) {
  const std::string keep_err = r->err;
  for (size_t q = from; q + 18 <= r->file_size; ++q) {
    const uint8_t* p = r->file + q;
    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) continue;
    size_t c = q;
    bool ok = true;
    for (int k = 0; k < 3 && ok && c < r->file_size; ++k) {
      BlockJob job;
      size_t bsize = 0;
      ok = parse_block(r, c, &job, &bsize) == 0;
      c += bsize;
    }
    if (ok) {
      r->err = keep_err;
      return q;
    }
  }
  r->err = keep_err;
  return r->file_size;
}

// Inflated bytes from a block boundary on, with the table that maps them back to virtual offsets.
struct PlanBuf {
  std::vector<uint8_t> data;
  std::vector<size_t> blk_c, blk_off;   // per block: compressed offset, offset of its first byte in `data`
  size_t next_c = 0;
  bool eof = false;
  Inflater inf;
};

int plan_more(bamcols* r, PlanBuf& b, size_t want_blocks) {
  for (size_t k = 0; k < want_blocks && !b.eof; ++k) {
    BlockJob job;
    size_t bsize = 0;
    const int rc = parse_block(r, b.next_c, &job, &bsize);
    if (rc < 0) return rc;
    if (rc == 1) {
      b.eof = true;
      break;
    }
    const size_t at = b.data.size();
    b.data.resize(at + job.isize);
    if (!b.inf.run(job.src, job.src_len, b.data.data() + at, job.isize))
      return fail(r, BAMCOLS_ERR_FORMAT, "corrupt BGZF block (inflate failed) at offset %zu", b.next_c);
    b.blk_c.push_back(b.next_c);
    b.blk_off.push_back(at);
    b.next_c += bsize;
  }
  return 0;
}

int64_t plan_voffset(const PlanBuf& b, size_t pos) {
  // the LAST block that starts at or before pos and is not empty there (a record that begins exactly where a
  // block ends belongs to the next block)
  size_t k = std::upper_bound(b.blk_off.begin(), b.blk_off.end(), pos) - b.blk_off.begin() - 1;
  return (int64_t)((b.blk_c[k] << 16) | (pos - b.blk_off[k]));
}

}  // namespace

int bamcols_plan_shards(bamcols* r, int n_shards, int64_t* voffsets) {
  if (!r || !voffsets || n_shards < 1) return BAMCOLS_ERR_INVALID;
  const int32_t n_ref = (int32_t)r->ref_names.size();
  const size_t c_first = (size_t)(r->first_voffset >> 16);
  voffsets[0] = r->first_voffset;
  voffsets[n_shards] = -1;   // the end of the file
  for (int k = 1; k < n_shards; ++k) {
    voffsets[k] = -1;
    const size_t target = c_first + (size_t)((double)(r->file_size - c_first) * (double)k / (double)n_shards);
    const size_t q = find_block_boundary(r, std::max(target, c_first + 1));
    if (q >= r->file_size) continue;   // nothing behind the target: an empty shard at the end
    PlanBuf b;
    b.next_c = q;
    int rc = plan_more(r, b, 8);
    if (rc < 0) return rc;
    while (b.data.empty() && !b.eof) {   // (empty blocks)
      rc = plan_more(r, b, 8);
      if (rc < 0) return rc;
    }
    if (b.data.empty()) continue;   // only the end-of-file marker lies behind the target: an empty shard
    // a record start: eight plausible records in a row (samtools / htslib start every block with one; a record
    // of a long read can be megabytes, so the search may have to run on for a while)
    size_t p = SIZE_MAX;
    for (size_t cand = 0; cand < ((size_t)1 << 26); ++cand) {
      if (cand + 36 > b.data.size()) {
        if (b.eof) break;
        rc = plan_more(r, b, 16);
        if (rc < 0) return rc;
        if (cand + 36 > b.data.size()) break;
      }
      size_t x = cand;
      int good = 0;
      while (good < 8) {
        if (x + 36 > b.data.size()) {
          if (b.eof) break;
          rc = plan_more(r, b, 8);
          if (rc < 0) return rc;
          continue;
        }
        if (!plausible_record(b.data.data(), x, b.data.size(), n_ref)) break;
        ++good;
        x += 4 + le32(b.data.data() + x);
        if (x == b.data.size() && b.eof) break;   // the chain ends with the file
      }
      if (good >= 8 || (good >= 1 && b.eof && x == b.data.size())) {
        p = cand;
        break;
      }
    }
    if (p == SIZE_MAX) return fail(r, BAMCOLS_ERR_FORMAT, "no record boundary found behind offset %zu while planning shards", q);
    // walk on to the first record whose trimmed name differs from its predecessor's: shards never split a read
    std::string prev;
    bool have_prev = false;
    for (;;) {
      while (p + 4 > b.data.size() || p + 4 + le32(b.data.data() + p) > b.data.size()) {
        if (b.eof) break;
        rc = plan_more(r, b, 16);
        if (rc < 0) return rc;
      }
      if (p + 4 > b.data.size() || p + 4 + le32(b.data.data() + p) > b.data.size()) {
        p = SIZE_MAX;   // the file ends inside this read: the shard is empty
        break;
      }
      const uint8_t* c = b.data.data() + p + 4;
      const size_t l_name = c[8];
      const char* nm = (const char*)c + 32;
      const size_t tl = trimmed_len(nm, l_name ? l_name - 1 : 0);
      if (have_prev && (tl != prev.size() || memcmp(nm, prev.data(), tl) != 0)) break;
      prev.assign(nm, tl);
      have_prev = true;
      p += 4 + le32(b.data.data() + p);
    }
    if (p != SIZE_MAX) voffsets[k] = plan_voffset(b, p);
  }
  // shards are contiguous and in order; a shard that would start before its predecessor's start (one read
  // reaching over several targets) starts where that one does and the predecessor is empty
  for (int k = n_shards - 1; k >= 1; --k)
    if (voffsets[k] < 0) voffsets[k] = k + 1 < n_shards ? voffsets[k + 1] : -1;
  for (int k = 1; k < n_shards; ++k)
    if (voffsets[k] >= 0 && voffsets[k] < voffsets[k - 1]) voffsets[k] = voffsets[k - 1];
  return BAMCOLS_OK;
}

int bamcols_set_range(bamcols* r, int64_t vbegin, int64_t vend) {
  if (!r) return BAMCOLS_ERR_INVALID;
  if (r->mode != 0) return fail(r, BAMCOLS_ERR_INVALID, "bamcols_set_range must come before the first bamcols_emit");
  if (r->prefetch.joinable()) r->prefetch.join();   // whatever it inflated belongs to the unranged reader
  if (vbegin < 0) {   // an empty shard at the end of the file
    r->wpos = r->wend = 0;
    r->file_done = true;
    return BAMCOLS_OK;
  }
  if (vbegin < r->first_voffset) return fail(r, BAMCOLS_ERR_INVALID, "range begins inside the BAM header");
  if (vend >= 0 && vend < vbegin) return fail(r, BAMCOLS_ERR_INVALID, "range ends before it begins");
  r->end_c = vend < 0 ? SIZE_MAX : (size_t)(vend >> 16);
  r->end_u = vend < 0 ? 0u : (uint32_t)(vend & 0xFFFF);
  r->cpos = (size_t)(vbegin >> 16);
  r->wpos = r->wend = 0;
  r->file_done = false;
  r->prefetch_rc = 0;
  if (vend >= 0 && vend == vbegin) {
    r->file_done = true;
    return BAMCOLS_OK;
  }
  const int rc = refill(r);
  if (rc < 0) return rc;
  const size_t skip = (size_t)(vbegin & 0xFFFF);
  if (skip > r->wend) return fail(r, BAMCOLS_ERR_INVALID, "range begins beyond its block");
  r->wpos = skip;
  return BAMCOLS_OK;
}

int bamcols_track_ranges(bamcols* r, int enable) {
  if (!r) return BAMCOLS_ERR_INVALID;
  if (r->mode != 0) return fail(r, BAMCOLS_ERR_INVALID, "bamcols_track_ranges must be called before the first bamcols_emit");
  r->track_ranges = enable != 0;
  if (r->track_ranges) {
    r->range_min.assign(r->ref_names.size(), INT32_MAX);
    r->range_max.assign(r->ref_names.size(), -1);
  }
  return BAMCOLS_OK;
}

int bamcols_ranges(const bamcols* r, const int32_t** min_pos, const int32_t** max_pos) {
  if (!r || !min_pos || !max_pos || !r->track_ranges) return BAMCOLS_ERR_INVALID;
  *min_pos = r->range_min.data();
  *max_pos = r->range_max.data();
  return (int)r->range_min.size();
}

int64_t bamcols_blocks(bamcols* r, int64_t c_begin, int64_t max_bytes, int64_t max_blocks, int64_t* payload_off,
                       int32_t* payload_len, int32_t* isize, int64_t* c_end) {
  if (!r || !payload_off || !payload_len || !isize || !c_end || c_begin < 0 || max_bytes < 1 || max_blocks < 1)
    return BAMCOLS_ERR_INVALID;
  if ((size_t)c_begin > r->file_size) return fail(r, BAMCOLS_ERR_INVALID, "offset %lld beyond the end of the file", (long long)c_begin);
  size_t c = (size_t)c_begin;
  int64_t n = 0;
  while (n < max_blocks) {
    BlockJob job;
    size_t bsize = 0;
    const int rc = parse_block(r, c, &job, &bsize);
    if (rc < 0) return rc;
    if (rc == 1 || (n > 0 && c + bsize - (size_t)c_begin > (size_t)max_bytes)) break;
    payload_off[n] = (int64_t)((size_t)(job.src - r->file) - (size_t)c_begin);
    payload_len[n] = (int32_t)job.src_len;
    isize[n] = (int32_t)job.isize;
    ++n;
    c += bsize;
  }
  *c_end = (int64_t)c;
  return n;
}

int bamcols_inflate_raw(const uint8_t* src, int64_t src_len, uint8_t* dst, int64_t dst_len, int mode) {
  if (!src || (!dst && dst_len) || src_len < 0 || dst_len < 0) return BAMCOLS_ERR_INVALID;
  if (mode == 2) {   // the whole-buffer decoder alone: 1 = decoded, 0 = declined
    std::unique_ptr<Inflater> inf(new Inflater());
    if (dst_len == 0) return 1;
    return fastinflate::fast_inflate(src, (size_t)src_len, dst, (size_t)dst_len, inf->scratch, inf->fixed, inf->fixed_ready) ? 1 : 0;
  }
  std::unique_ptr<Inflater> inf(new Inflater());
  inf->zlib_only = mode == 1;
  return inf->run(src, (size_t)src_len, dst, (size_t)dst_len) ? 1 : 0;
}

int bamcols_phase_seconds(const bamcols* r, double* out6) {
  if (!r || !out6) return BAMCOLS_ERR_INVALID;
  for (int i = 0; i < 6; ++i) out6[i] = r->phase_s[i];
  return BAMCOLS_OK;
}

int64_t bamcols_all_alignments(const bamcols* r) { return r ? r->all_alignments : (int64_t)BAMCOLS_ERR_INVALID; }
int64_t bamcols_n_groups(const bamcols* r) { return r ? r->group + 1 : (int64_t)BAMCOLS_ERR_INVALID; }

int64_t bamcols_emit(bamcols* r, bamcols_cells* cells, int32_t* read_group, int32_t* target_idx, int32_t* hap_idx,
                     int32_t* cell_idx, int64_t capacity, int* done) {
  if (!r || !read_group || !target_idx || !hap_idx || !done || capacity < 1) return BAMCOLS_ERR_INVALID;
  if (cells && !cell_idx) return fail(r, BAMCOLS_ERR_INVALID, "per-cell mode needs a cell_idx buffer");
  if (r->tid_target.empty() && !r->ref_names.empty()) return fail(r, BAMCOLS_ERR_INVALID, "bamcols_set_tables was not called");
  *done = 0;
  if (r->prefetch.joinable()) {
    r->prefetch.join();
    if (r->prefetch_rc < 0) return r->prefetch_rc;
  }
  const int want_mode = cells ? 2 : 1;
  if (r->mode == 0) r->mode = want_mode;
  if (r->mode == 3) return fail(r, BAMCOLS_ERR_INVALID, "a reader that has emitted name keys cannot switch to read groups");
  if (r->mode != want_mode) return fail(r, BAMCOLS_ERR_INVALID, "a reader cannot switch between single-sample and per-cell rules");
  try {   // no exception may cross the C ABI
    void* const dst[4] = {read_group, target_idx, hap_idx, cell_idx};
    return emit_rows(r, cells, dst, capacity, done);
  } catch (const std::bad_alloc&) {
    return fail(r, BAMCOLS_ERR_IO, "out of memory while decoding the window");
  }
}

int64_t bamcols_emit_keys(bamcols* r, uint64_t* key_lo, uint64_t* key_hi, int32_t* target_idx, int32_t* hap_idx,
                          int64_t capacity, int* done) {
  if (!r || !key_lo || !key_hi || !target_idx || !hap_idx || !done || capacity < 1) return BAMCOLS_ERR_INVALID;
  if (r->tid_target.empty() && !r->ref_names.empty()) return fail(r, BAMCOLS_ERR_INVALID, "bamcols_set_tables was not called");
  *done = 0;
  if (r->prefetch.joinable()) {
    r->prefetch.join();
    if (r->prefetch_rc < 0) return r->prefetch_rc;
  }
  if (r->mode == 0) r->mode = 3;
  if (r->mode != 3) return fail(r, BAMCOLS_ERR_INVALID, "a reader that has emitted read groups cannot switch to name keys");
  try {
    void* const dst[4] = {key_lo, key_hi, target_idx, hap_idx};
    return emit_rows(r, nullptr, dst, capacity, done);
  } catch (const std::bad_alloc&) {
    return fail(r, BAMCOLS_ERR_IO, "out of memory while decoding the window");
  }
}

}  // extern "C"
