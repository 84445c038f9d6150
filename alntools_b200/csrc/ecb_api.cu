// ecb_api.cu — context management and the C ABI of libecb200.so (see include/ecb200.h).
#include <algorithm>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/ecb200.h"
#include "ecb_common.cuh"
#include "ecb_scan.cuh"
#include "ecb_group.cuh"
#include "ecb_harvest.cuh"
#include "ecb_finalize.cuh"
#include "ecb_sort.cuh"
#include "ecb_cells.cuh"
#include "ecb_exchange.cuh"
#include "ecb_cells_exchange.cuh"
#include "ecb_bam.cuh"
#include "ecb_sam.cuh"
#include "ecb_collate.cuh"
#include "ecb_longread.cuh"
#include "ecb_samples.cuh"
#include "ecb_ecrows.cuh"

#define ECB_PUSH_LIMIT (0x7FFFFFFFll - 8192)   // alignments of one ecb_push
// Largest ECB_OPT_MAX_READ, and what 0 stands for: the push limit as documented (2^31 - 8192), one more than the
// longest push, so that no read is ever above it.
#define ECB_MAX_READ_LIMIT ((1ll << 31) - 8192)

namespace {

thread_local std::string g_create_error;

struct ecb_timer {
  cudaEvent_t a = nullptr, b = nullptr;
};

}  // namespace

struct ecb_ctx {
  int device = 0;
  int sm_count = 148;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  cudaMemPool_t pool = nullptr;   // private stream-ordered pool: nothing this context does changes the device's default pool
  int n_targets = 0, n_haps = 0, with_cells = 0;
  int64_t hint = 0;
  // options
  int result_on_device = 0;
  int64_t opt_table_slots = 0, opt_pair_slots = 0, opt_grid = 0, opt_chunk_len = 0;
  int use_cache = 1;
  int verify_keys = 0;
  int pageable_results = 0;
  int64_t opt_bam_window = 0;
  int64_t opt_collate_slots = 0, opt_collate_piece = 0, opt_collate_budget = 0;
  int64_t max_read = ECB_MAX_READ_ALIGNMENTS;   // ECB_OPT_MAX_READ (0 stored as the push limit)
  // EC table
  DevBuf table;
  u32 table_slots = 0;
  DevBuf ec_slot, ec_rep, ec_len, row_len, row_off;  // [table_slots] u32 each
  DevBuf spill;
  bool group_attr_set = false;
  DevBuf arena;                              // uint2 pairs
  u64 arena_used = 0;
  DevBuf long_list, mid_list, big_list, count_of;
  // triple table (cells)
  DevBuf ttable;
  u32 ttable_slots = 0;
  u32 n_triples = 0;
  // counters
  EcbCounters* d_ctr = nullptr;
  EcbCounters* h_ctr = nullptr;  // pinned mirror
  u64* h_total = nullptr;        // pinned landing place of a scan total
  u32 n_ec = 0;                  // host copy after the last sync
  // staging
  DevBuf st_rg, st_tg, st_hp, st_cell;
  DevBuf st2_rg, st2_tg, st2_hp, st2_cell;   // second staging set of pipelined host pushes
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_done[2] = {nullptr, nullptr};
  DevBuf overflow_bits;
  // reads longer than ECB_MAX_READ_ALIGNMENTS (ecb_longread.cuh): the grouping kernel's list, the sorted list with
  // the prefix of the lengths, the run ranks and the per-read sums
  DevBuf lr_list, lr_meta, lr_rank, lr_acc;
  DevBuf scan_buf;       // single-pass scan state: ticket, one status word per tile, total
  // push bookkeeping
  u64 min_base = ~0ull, max_end = 0;
  int64_t n_alignments = 0;
  u32 push_count = 0;
  // finalize scratch + results (device)
  DevBuf bitmap, word_rank, first_rel, ecid_of, prov_of, ec_keep;
  DevBuf r_a_indptr, r_a_indices, r_a_data, r_n_indptr, r_n_indices, r_n_data, r_cell_order;
  // cells scratch
  CellScratch cells;
  // host (pinned) results
  void* h_res = nullptr;
  size_t h_res_bytes = 0;
  // stats
  ecb_stats stats{};
  cudaEvent_t ev[8] = {};
  bool long_attr_set = false;
  // arena of the multi-GPU exchange (plain cudaMalloc: must be exportable through CUDA IPC)
  void* xa_base = nullptr;
  int64_t xa_cap_ec = 0;
  int64_t xa_cap_pairs = 0;                  // > 0: a per-cell arena (ecb_cells_arena_create)
  std::vector<void*> xa_opened;
  // per-cell exchange: kept reads per local EC, column of every global cell, entries per column of the slice
  DevBuf cx_kept, cx_col_of_cell, cx_col_counts;
  u32 cx_n_local_cells = 0;
  // samples (ecb_sample_close): every EC's count at the last close (provisional ids below smp_n_ec), the
  // (provisional id, reads) pairs of the closed samples, pairs per sample, the order key where the open sample starts
  // and the alignments pushed into it
  DevBuf smp_last, smp_pairs;
  u32 smp_n_ec = 0;
  u64 smp_n_pairs = 0;
  std::vector<u32> smp_counts;
  u64 smp_base = 0;
  int64_t smp_open = 0;
  // EC rows (ecb_push_ecs, ecb_ecrows.cuh): per row of the last push its key sums, table slot, provisional EC id and
  // arena place; the flags / positions of an append's N entries and its column counts.  ecr_rows: rows of the last
  // push, which await their ecb_sample_append (-1: none); ecr_used: rows were pushed since create/reset; ecr_broken:
  // a push failed after it had changed the EC table (only ecb_reset recovers)
  DevBuf ecr_acc, ecr_slot, ecr_ec, ecr_dst, ecr_flag, ecr_cols;
  DevBuf ecr_seen;           // per provisional id: tag of the last push with a row on the EC (ecr_seen_n set up)
  u32 ecr_seen_n = 0, ecr_tag = 0;
  int64_t ecr_rows = -1;
  bool ecr_used = false, ecr_broken = false;
  std::string err;
};

namespace {

int fail(ecb_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_create_error = buf;
  return code;
}

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(c, ECB_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                  __LINE__);                                                                       \
  } while (0)

#define CKR(expr)            \
  do {                       \
    int r_ = (expr);         \
    if (r_ != ECB_OK) return r_; \
  } while (0)

#define LAUNCH_CHECK(name)                                                                          \
  do {                                                                                              \
    c->stats.kernel_launches++;                                                                     \
    cudaError_t e_ = cudaGetLastError();                                                            \
    if (e_ != cudaSuccess) return fail(c, ECB_ERR_CUDA, "launch of %s failed: %s", name, cudaGetErrorString(e_)); \
  } while (0)

// Device memory comes from the stream-ordered allocator (a private pool per context, on the context's
// stream): growing a buffer costs no device-wide synchronisation, released blocks stay in the pool for the
// next buffer of this context, and ecb_destroy hands everything back to the driver.
int ensure(ecb_ctx* c, DevBuf& b, size_t bytes, bool preserve = false) {
  if (bytes <= b.bytes) return ECB_OK;
  size_t want = std::max(bytes, b.bytes + b.bytes / 2);
  want = (want + 255) & ~(size_t)255;
  void* np = nullptr;
  CK(cudaMallocFromPoolAsync(&np, want, c->pool, c->stream));
  if (preserve && b.p && b.bytes) CK(cudaMemcpyAsync(np, b.p, b.bytes, cudaMemcpyDeviceToDevice, c->stream));
  if (b.p) CK(cudaFreeAsync(b.p, c->stream));
  b.p = np;
  b.bytes = want;
  return ECB_OK;
}

void release(ecb_ctx* c, DevBuf& b) {
  if (b.p) cudaFreeAsync(b.p, c->stream);
  b.p = nullptr;
  b.bytes = 0;
}

u32 pow2_ceil(u64 v) {
  u64 p = 1;
  while (p < v) p <<= 1;
  return (u32)std::min<u64>(p, 1ull << 31);
}

int grid_for(u64 items, int per_block, int cap) {
  u64 g = (items + per_block - 1) / per_block;
  return (int)std::max<u64>(1, std::min<u64>(g, (u64)cap));
}

int sync_counters(ecb_ctx* c) {
  CK(cudaMemcpyAsync(c->h_ctr, c->d_ctr, sizeof(EcbCounters), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->stats.d2h_bytes += sizeof(EcbCounters);
  c->arena_used = c->h_ctr->arena_used;   // rows reserved by the harvest kernels so far
  return ECB_OK;
}

int check_device_error(ecb_ctx* c) {
  const u32 e = c->h_ctr->error;
  if (!e) return ECB_OK;
  if (e & ECB_DEVERR_VALUE_RANGE)
    return fail(c, ECB_ERR_INVALID, "target_idx/hap_idx outside [0,%d) x [0,%d)", c->n_targets, c->n_haps);
  if (e & ECB_DEVERR_READ_TOO_LONG)
    return fail(c, ECB_ERR_LIMIT, "a read has more than %lld alignments%s", (long long)c->max_read,
                c->max_read == ECB_MAX_READ_ALIGNMENTS ? " (ECB_OPT_MAX_READ raises the limit)" : "");
  if (e & ECB_DEVERR_VERIFY) return fail(c, ECB_ERR_LIMIT, "128-bit key collision detected by verification");
  return fail(c, ECB_ERR_LIMIT, "device error bits 0x%x", e);
}

// State of a single-pass scan over n_tiles tiles (ecb_scan.cuh), cleared on the stream: the ticket and the status
// words; the word after them receives the total.
int scan_state(ecb_ctx* c, u64 n_tiles, u64** state) {
  CKR(ensure(c, c->scan_buf, ((size_t)n_tiles + 2) * sizeof(u64)));
  *state = (u64*)c->scan_buf.p;
  CK(cudaMemsetAsync(*state, 0, ((size_t)n_tiles + 1) * sizeof(u64), c->stream));
  return ECB_OK;
}

// Device address of the total of a device_scan over n items, valid until the next scan: a copy of it enqueued
// after the scan reads it without a synchronisation of its own.
const u64* scan_total(const ecb_ctx* c, u64 n) {
  return (const u64*)c->scan_buf.p + (n + SCAN_BLOCK - 1) / SCAN_BLOCK + 1;
}

// Device-wide exclusive scan (in may alias out).  total_out (host) may be NULL.
template <bool POPC>
int device_scan(ecb_ctx* c, const u32* in, u32* out, u64 n, u32 base_offset, u64* total_out) {
  const u64 n_tiles = (n + SCAN_BLOCK - 1) / SCAN_BLOCK;
  if (n_tiles == 0) {
    CKR(ensure(c, c->scan_buf, 2 * sizeof(u64)));
    CK(cudaMemsetAsync((u64*)c->scan_buf.p + 1, 0, sizeof(u64), c->stream));   // scan_total() of an empty scan
    if (total_out) *total_out = 0;
    return ECB_OK;
  }
  if (n_tiles > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "scan of %llu items is too long", (unsigned long long)n);
  u64* state = nullptr;
  CKR(scan_state(c, n_tiles, &state));
  scan_kernel<POPC><<<(unsigned)n_tiles, SCAN_THREADS, 0, c->stream>>>(in, n, out, base_offset, state, (u32)n_tiles);
  LAUNCH_CHECK("scan");
  if (total_out) {
    CK(cudaMemcpyAsync(total_out, state + n_tiles + 1, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += sizeof(u64);
  }
  return ECB_OK;
}

int alloc_ec_arrays(ecb_ctx* c, u32 slots, bool preserve) {
  CKR(ensure(c, c->ec_slot, (size_t)slots * 4, preserve));
  CKR(ensure(c, c->ec_rep, (size_t)slots * 4, preserve));
  CKR(ensure(c, c->ec_len, (size_t)slots * 4, preserve));
  CKR(ensure(c, c->row_len, (size_t)slots * 4, preserve));
  CKR(ensure(c, c->row_off, (size_t)slots * 4, preserve));
  CKR(ensure(c, c->long_list, (size_t)slots * 4, false));
  CKR(ensure(c, c->mid_list, (size_t)slots * 4, false));
  CKR(ensure(c, c->big_list, (size_t)slots * 4, false));
  return ECB_OK;
}

// first_n: alignments of the push that triggers the allocation (0 when unknown).  With a hint the
// table gets hint/8 slots (ECs are a small fraction of the alignments of a whole job); without one
// only the first push is known and a job's early part is EC-rich, so first_n/4.
int init_table(ecb_ctx* c, int64_t first_n = 0) {
  u64 want = c->opt_table_slots > 0 ? (u64)c->opt_table_slots
             : c->hint > 0          ? std::max<u64>(1u << 16, (u64)c->hint / 8)
                                    : std::max<u64>(1u << 16, (u64)first_n / 4);
  c->table_slots = std::max<u32>(1u << 10, pow2_ceil(want));
  CKR(ensure(c, c->table, (size_t)c->table_slots * sizeof(EcbEntry)));
  CK(cudaMemsetAsync(c->table.p, 0xFF, (size_t)c->table_slots * sizeof(EcbEntry), c->stream));
  CKR(alloc_ec_arrays(c, c->table_slots, false));
  if (c->with_cells) {
    u64 tw = c->opt_pair_slots > 0 ? (u64)c->opt_pair_slots : std::max<u64>(1u << 16, (u64)c->hint / 8);
    c->ttable_slots = std::max<u32>(1u << 10, pow2_ceil(tw));
    CKR(ensure(c, c->ttable, (size_t)c->ttable_slots * sizeof(EcbEntry)));
    CK(cudaMemsetAsync(c->ttable.p, 0xFF, (size_t)c->ttable_slots * sizeof(EcbEntry), c->stream));
  }
  CK(cudaMemsetAsync(c->d_ctr, 0, sizeof(EcbCounters), c->stream));
  memset(c->h_ctr, 0, sizeof(EcbCounters));
  c->n_ec = 0;
  c->n_triples = 0;
  c->arena_used = 0;
  return ECB_OK;
}

// Rebuild the (file, EC, cell) table with `new_slots` slots; remap (device, by old EC slot) may be NULL.
int rebuild_triple_table(ecb_ctx* c, u32 new_slots, const u32* remap) {
  DevBuf nt;
  CKR(ensure(c, nt, (size_t)new_slots * sizeof(EcbEntry)));
  CK(cudaMemsetAsync(nt.p, 0xFF, (size_t)new_slots * sizeof(EcbEntry), c->stream));
  ecb_triple_remap_kernel<<<grid_for(c->ttable_slots, 256, c->sm_count * 8), 256, 0, c->stream>>>(
      (const EcbEntry*)c->ttable.p, c->ttable_slots, (EcbEntry*)nt.p, new_slots - 1, remap);
  LAUNCH_CHECK("triple_remap");
  CK(cudaStreamSynchronize(c->stream));
  release(c, c->ttable);
  c->ttable = nt;
  c->ttable_slots = new_slots;
  return ECB_OK;
}

int grow_table(ecb_ctx* c, u32 new_slots) {
  DevBuf nt;
  CKR(ensure(c, nt, (size_t)new_slots * sizeof(EcbEntry)));
  CK(cudaMemsetAsync(nt.p, 0xFF, (size_t)new_slots * sizeof(EcbEntry), c->stream));
  CKR(alloc_ec_arrays(c, new_slots, true));
  DevBuf remap;
  if (c->with_cells) CKR(ensure(c, remap, (size_t)c->table_slots * 4));
  ecb_rehash_kernel<<<grid_for(c->table_slots, 256, c->sm_count * 8), 256, 0, c->stream>>>(
      (const EcbEntry*)c->table.p, c->table_slots, (EcbEntry*)nt.p, new_slots - 1, (u32*)c->ec_slot.p,
      (u32*)remap.p, c->d_ctr);
  LAUNCH_CHECK("rehash");
  CK(cudaStreamSynchronize(c->stream));
  release(c, c->table);
  c->table = nt;
  c->table_slots = new_slots;
  c->stats.table_grows++;
  if (c->with_cells) {
    CKR(rebuild_triple_table(c, c->ttable_slots, (const u32*)remap.p));
    release(c, remap);
  }
  return ECB_OK;
}

GroupParams make_group_params(ecb_ctx* c, const int32_t* rg, const int32_t* tg, const int32_t* hp,
                              const int32_t* cell, int64_t n, int64_t order_base, int drop_last, u32 push_id) {
  GroupParams P{};
  P.rg = rg; P.tg = tg; P.hp = hp; P.cell = cell;
  P.n = (int)n;
  P.order_base = (u64)order_base;
  P.drop_last = drop_last;
  P.use_cache = c->use_cache;
  P.n_targets = c->n_targets;
  P.n_haps = c->n_haps;
  P.table = (EcbEntry*)c->table.p;
  P.mask = c->table_slots - 1;
  P.ec_slot = (u32*)c->ec_slot.p;
  P.ec_rep = (u32*)c->ec_rep.p;
  P.ec_len = (u32*)c->ec_len.p;
  P.ctr = c->d_ctr;
  P.spill = (EcbSpill*)c->spill.p;
  P.overflow_bits = (u32*)c->overflow_bits.p;
  P.ttable = (EcbEntry*)c->ttable.p;
  P.tmask = c->ttable_slots ? c->ttable_slots - 1 : 0;
  P.push_id = push_id;
  P.max_read = (int)c->max_read;
  P.deferred = (uint2*)c->lr_list.p;
  return P;
}

// Opt-in shared memory of the grouping kernels.  The default kernels are prepared once per context; an
// experimental variant is prepared when it is first launched, so that nothing it needs can get in the way
// of the default path.
template <class K>
int allow_group_smem(ecb_ctx* c, K kernel) {
  CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(GroupSmem)));
  return ECB_OK;
}

int group_prepare_launch(ecb_ctx* c) {
  if (!c->group_attr_set) {
    CKR(allow_group_smem(c, ecb_group_insert_kernel<true>));
    CKR(allow_group_smem(c, ecb_group_insert_kernel<false>));
    c->group_attr_set = true;
  }
  return ECB_OK;
}

// Launch geometry of the grouping kernel: one persistent CTA per SM, every warp takes chunks of
// `chunk_len` alignments from a shared counter.
void group_geometry(ecb_ctx* c, int64_t n, int* grid, int* chunk_len) {
  const int wpc = ECB_GWARPS;
  const int64_t warps = (int64_t)c->sm_count * wpc;
  int64_t cl = c->opt_chunk_len > 0 ? c->opt_chunk_len : std::min<int64_t>(4096, std::max<int64_t>(256, n / (warps * 4)));
  cl = (cl + 31) / 32 * 32;
  const int64_t chunks = (n + cl - 1) / cl;
  int64_t g = c->opt_grid > 0 ? c->opt_grid : std::min<int64_t>(c->sm_count, (chunks + wpc - 1) / wpc);
  *grid = (int)std::max<int64_t>(1, g);
  *chunk_len = (int)cl;
}

// Rows of the ECs claimed since provisional id e0, up to the device's EC counter.  No host round trip: the
// range ends where the counter stands when the kernels run, the kernels reserve their rows on the device-side
// arena cursor, the lists of the longer reads are sized on the device, and all four kernels are launched
// whether their range and lists turn out empty or not (an empty one costs a few microseconds).  The arena has
// room for the push (push_one sizes it before the grouping kernel).
int harvest_new_rows(ecb_ctx* c, const int32_t* rg, const int32_t* tg, const int32_t* hp, int64_t n, u32 e0) {
  HarvestParams H{};
  H.rg = rg; H.tg = tg; H.hp = hp; H.n = (int)n;
  H.n_targets = c->n_targets; H.n_haps = c->n_haps;
  H.ec_rep = (const u32*)c->ec_rep.p;
  H.ec_len = (const u32*)c->ec_len.p;
  H.e0 = e0;
  H.row_len = (u32*)c->row_len.p;
  H.row_off = (u32*)c->row_off.p;
  H.long_list = (u32*)c->long_list.p;
  H.mid_list = (u32*)c->mid_list.p;
  H.big_list = (u32*)c->big_list.p;
  H.ctr = c->d_ctr;
  H.arena = (uint2*)c->arena.p;
  ecb_harvest_short_kernel<<<c->sm_count * 16, 256, 0, c->stream>>>(H);
  LAUNCH_CHECK("harvest_short");
  ecb_harvest_warp_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(H);
  LAUNCH_CHECK("harvest_warp");
  ecb_harvest_wsort_kernel<<<c->sm_count * 6, 256, (size_t)8 * HARVEST_WSORT_MAX * 4, c->stream>>>(H);
  LAUNCH_CHECK("harvest_wsort");
  if (!c->long_attr_set) {
    CK(cudaFuncSetAttribute(ecb_harvest_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, HARVEST_LONG_MAX * 4));
    c->long_attr_set = true;
  }
  ecb_harvest_long_kernel<<<c->sm_count * 3, 256, HARVEST_LONG_MAX * 4, c->stream>>>(H);
  LAUNCH_CHECK("harvest_long");
  // the list counters go back to zero for the next push (the kernels above have read them by then)
  CK(cudaMemsetAsync(&c->d_ctr->scratch[1], 0, sizeof(u32), c->stream));
  CK(cudaMemsetAsync(&c->d_ctr->scratch[3], 0, sizeof(u32), c->stream));
  CK(cudaMemsetAsync(&c->d_ctr->n_long, 0, sizeof(u32), c->stream));
  return ECB_OK;
}

// Stable LSD radix sort of n (key, value) pairs on the low `bits` key bits.  Input in sort_k[0]/
// sort_v[0]; returns which ping-pong buffer holds the result.
int radix_sort(ecb_ctx* c, u32 n, int bits, int* result_buf) {
  CellScratch& S = c->cells;
  *result_buf = 0;
  if (n == 0) return ECB_OK;
  const u32 n_tiles = (n + SORT_TILE - 1) / SORT_TILE;
  CKR(ensure(c, S.sort_k[1], (size_t)n * 8));
  CKR(ensure(c, S.sort_v[1], (size_t)n * 4));
  CKR(ensure(c, S.hist, (size_t)n_tiles * 256 * 4));
  int cur = 0;
  for (int shift = 0; shift < bits; shift += 8) {
    sort_hist_kernel<<<n_tiles, SORT_THREADS, 0, c->stream>>>((const u64*)S.sort_k[cur].p, n, shift, (u32*)S.hist.p, n_tiles);
    LAUNCH_CHECK("sort_hist");
    CKR(device_scan<false>(c, (const u32*)S.hist.p, (u32*)S.hist.p, (u64)n_tiles * 256, 0, nullptr));
    sort_scatter_kernel<<<n_tiles, SORT_THREADS, 0, c->stream>>>((const u64*)S.sort_k[cur].p, (const u32*)S.sort_v[cur].p,
                                                                   n, shift, (const u32*)S.hist.p, n_tiles,
                                                                   (u64*)S.sort_k[cur ^ 1].p, (u32*)S.sort_v[cur ^ 1].p);
    LAUNCH_CHECK("sort_scatter");
    cur ^= 1;
  }
  *result_buf = cur;
  return ECB_OK;
}

int bits_for(u64 v) {
  int b = 1;
  while (b < 64 && (v >> b)) ++b;
  return b;
}

// ---- reads longer than ECB_MAX_READ_ALIGNMENTS (ecb_longread.cuh) ----------------------------------------------
// Key pass and insert of the n_def reads the grouping kernel deferred.  One host round trip brings their list back
// (sorted by offset here, so that read indices follow the push order), one copy sends it with the prefix of the
// lengths, and the sort, sums, scan and insert follow on the stream; the caller's sync_counters ends it.
int long_keys(ecb_ctx* c, const GroupParams& P, const int32_t* tg, const int32_t* hp, u32 n_def, LongParams* L) {
  std::vector<uint2> list(n_def);
  CK(cudaMemcpyAsync(list.data(), c->lr_list.p, (size_t)n_def * sizeof(uint2), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->stats.d2h_bytes += (int64_t)n_def * sizeof(uint2);
  std::sort(list.begin(), list.end(), [](const uint2& a, const uint2& b) { return a.x < b.x; });
  // [n_def] (offset, length), then [n_def + 1] u32 starts
  std::vector<u32> meta((size_t)n_def * 2 + n_def + 1);
  memcpy(meta.data(), list.data(), (size_t)n_def * sizeof(uint2));
  u32* start = meta.data() + (size_t)n_def * 2;
  u64 total = 0;
  for (u32 r = 0; r < n_def; ++r) {
    start[r] = (u32)total;
    total += list[r].y;
  }
  start[n_def] = (u32)total;   // total <= alignments of the push < 2^31
  CKR(ensure(c, c->lr_meta, meta.size() * 4));
  CK(cudaMemcpyAsync(c->lr_meta.p, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice, c->stream));
  c->stats.h2d_bytes += (int64_t)meta.size() * 4;
  CellScratch& S = c->cells;
  CKR(ensure(c, S.sort_k[0], (size_t)total * 8));
  CKR(ensure(c, S.sort_v[0], (size_t)total * 4));
  CKR(ensure(c, c->lr_rank, ((size_t)total + 1) * 4));
  CKR(ensure(c, c->lr_acc, (size_t)n_def * sizeof(LongAcc)));
  LongParams& Q = *L;
  Q = LongParams{};
  Q.tg = tg; Q.hp = hp;
  Q.reads = (const uint2*)c->lr_meta.p;
  Q.start = (const u32*)c->lr_meta.p + (size_t)n_def * 2;
  Q.n_reads = n_def;
  Q.total = (u32)total;
  Q.n_targets = c->n_targets; Q.n_haps = c->n_haps;
  Q.keys = (u64*)S.sort_k[0].p;
  Q.vals = (u32*)S.sort_v[0].p;
  Q.rank = (u32*)c->lr_rank.p;
  Q.acc = (LongAcc*)c->lr_acc.p;
  Q.ctr = c->d_ctr;
  ecb_long_gather_kernel<<<grid_for(total, ECB_LONG_THREADS, c->sm_count * 8), ECB_LONG_THREADS, 0, c->stream>>>(Q);
  LAUNCH_CHECK("long_gather");
  int rb = 0;
  CKR(radix_sort(c, (u32)total, 31 + (n_def > 1 ? bits_for(n_def - 1) : 0), &rb));
  Q.sorted = (const u64*)S.sort_k[rb].p;
  ecb_long_sums_kernel<<<grid_for(total, ECB_LONG_THREADS * 16, c->sm_count * 4), ECB_LONG_THREADS, 0, c->stream>>>(Q);
  LAUNCH_CHECK("long_sums");
  CKR(device_scan<false>(c, Q.rank, Q.rank, total + 1, 0, nullptr));
  ecb_long_insert_kernel<<<grid_for(n_def, ECB_LONG_THREADS, c->sm_count), ECB_LONG_THREADS, 0, c->stream>>>(P, Q);
  LAUNCH_CHECK("long_insert");
  return ECB_OK;
}

// Rows of the ECs the deferred reads claimed (after the harvest, which skipped them), and their verification.
int long_rows(ecb_ctx* c, const LongParams& L) {
  const int g_r = grid_for(L.n_reads, ECB_LONG_THREADS, c->sm_count);
  const int g_i = grid_for(L.total, ECB_LONG_THREADS, c->sm_count * 8);
  ecb_long_rows_reserve_kernel<<<g_r, ECB_LONG_THREADS, 0, c->stream>>>(L, (u32*)c->row_len.p, (u32*)c->row_off.p);
  LAUNCH_CHECK("long_rows_reserve");
  ecb_long_rows_kernel<false><<<g_i, ECB_LONG_THREADS, 0, c->stream>>>(L, (uint2*)c->arena.p);
  LAUNCH_CHECK("long_rows");
  ecb_long_rows_kernel<true><<<g_i, ECB_LONG_THREADS, 0, c->stream>>>(L, (uint2*)c->arena.p);
  LAUNCH_CHECK("long_rows_or");
  if (c->verify_keys) {
    ecb_long_verify_kernel<<<std::min<u32>(L.n_reads, (u32)c->sm_count * 4), ECB_LONG_THREADS, 0, c->stream>>>(
        L, (const EcbEntry*)c->table.p, c->table_slots - 1, (const u32*)c->row_len.p, (const u32*)c->row_off.p,
        (const uint2*)c->arena.p);
    LAUNCH_CHECK("long_verify");
  }
  return ECB_OK;
}

CellParams make_cell_params(ecb_ctx* c, const CellResult* cr) {
  CellScratch& S = c->cells;
  CellParams P{};
  P.ttable = (const EcbEntry*)c->ttable.p;
  P.t_slots = c->ttable_slots;
  P.ec_table = (const EcbEntry*)c->table.p;
  P.fe_table = (EcbEntry*)S.fe_table.p;
  P.fe_mask = S.fe_slots - 1;
  P.pair_table = (EcbEntry*)S.pair_table.p;
  P.pair_mask = S.pair_slots - 1;
  P.cell_key = (u64*)S.cell_key.p;
  P.cell_total = (u64*)S.cell_total.p;
  P.cell_new = (int32_t*)S.cell_new.p;
  P.ec_keep = (u32*)c->ec_keep.p;
  P.ecid_of = (const u32*)c->ecid_of.p;
  P.min_base = c->min_base;
  P.n_cells = (u32)cr->n_cells;
  P.ctr = c->d_ctr;
  return P;
}

// The local passes over the (file, EC, cell) table: every cell's sort key and total, the (EC, cell) counts
// summed over files (cr->n_cells = largest cell id + 1).  Needs at least one triple.
int cells_local(ecb_ctx* c, CellResult* cr) {
  CellScratch& S = c->cells;
  if (c->max_end - c->min_base > 0xFFFFFFFFull)
    return fail(c, ECB_ERR_LIMIT, "per-cell mode needs the pushed order range to span less than 2^32 positions");
  S.fe_slots = std::max<u32>(1024u, pow2_ceil((u64)c->n_triples * 2));
  S.pair_slots = S.fe_slots;
  CKR(ensure(c, S.fe_table, (size_t)S.fe_slots * sizeof(EcbEntry)));
  CKR(ensure(c, S.pair_table, (size_t)S.pair_slots * sizeof(EcbEntry)));
  CK(cudaMemsetAsync(S.fe_table.p, 0xFF, (size_t)S.fe_slots * sizeof(EcbEntry), c->stream));
  CK(cudaMemsetAsync(S.pair_table.p, 0xFF, (size_t)S.pair_slots * sizeof(EcbEntry), c->stream));
  CK(cudaMemsetAsync(&c->d_ctr->scratch[0], 0, sizeof(u32), c->stream));
  CKR(ensure(c, c->ec_keep, (size_t)c->n_ec * 4));
  CK(cudaMemsetAsync(c->ec_keep.p, 0, (size_t)c->n_ec * 4, c->stream));

  CellParams P = make_cell_params(c, cr);
  const int g_t = grid_for(c->ttable_slots, 256, c->sm_count * 8);
  cells_pass1_kernel<<<g_t, 256, 0, c->stream>>>(P);
  LAUNCH_CHECK("cells_pass1");
  CKR(sync_counters(c));
  CKR(check_device_error(c));
  const u32 n_cells = c->h_ctr->scratch[0];
  if (n_cells == 0 || n_cells > 0x7FFFFFFFu) return fail(c, ECB_ERR_INVALID, "invalid cell ids (negative?)");
  cr->n_cells = n_cells;
  CKR(ensure(c, S.cell_key, (size_t)n_cells * 8));
  CKR(ensure(c, S.cell_total, (size_t)n_cells * 8 * CELLS_TOTAL_REPLICAS));
  CKR(ensure(c, S.cell_new, (size_t)n_cells * 4));
  CKR(ensure(c, c->r_cell_order, (size_t)n_cells * 4));
  CK(cudaMemsetAsync(S.cell_key.p, 0xFF, (size_t)n_cells * 8, c->stream));
  CK(cudaMemsetAsync(S.cell_total.p, 0, (size_t)n_cells * 8 * CELLS_TOTAL_REPLICAS, c->stream));
  P = make_cell_params(c, cr);
  cells_pass2_kernel<<<g_t, 256, 0, c->stream>>>(P);
  LAUNCH_CHECK("cells_pass2");
  cells_total_reduce_kernel<<<grid_for(n_cells, 256, c->sm_count * 8), 256, 0, c->stream>>>((u64*)S.cell_total.p, n_cells);
  LAUNCH_CHECK("cells_total_reduce");
  return ECB_OK;
}

// Cell order, minimum-count filter and the ec_keep flags (bam_utils_multisample.py:503-636).
int cells_prepare(ecb_ctx* c, int64_t min_cell_count, CellResult* cr) {
  CellScratch& S = c->cells;
  if (c->max_end - c->min_base > 0xFFFFFFFFull)
    return fail(c, ECB_ERR_LIMIT, "per-cell mode needs the pushed order range to span less than 2^32 positions");
  if (c->n_triples == 0) return fail(c, ECB_ERR_EMPTY, "no (EC, cell) counts were recorded");
  const u64 min_count = min_cell_count <= 0 ? 1ull : (u64)min_cell_count;  // :596-597
  CKR(cells_local(c, cr));
  const u32 n_cells = (u32)cr->n_cells;
  CellParams P = make_cell_params(c, cr);

  // order the cells by their nested first-occurrence key
  CKR(ensure(c, S.sort_k[0], (size_t)n_cells * 8));
  CKR(ensure(c, S.sort_v[0], (size_t)n_cells * 4));
  const int g_c = grid_for(n_cells, 256, c->sm_count * 8);
  cells_sort_input_kernel<<<g_c, 256, 0, c->stream>>>((const u64*)S.cell_key.p, n_cells, (u64*)S.sort_k[0].p, (u32*)S.sort_v[0].p);
  LAUNCH_CHECK("cells_sort_input");
  int rb = 0;
  CKR(radix_sort(c, n_cells, 64, &rb));
  CKR(ensure(c, S.flags, (size_t)n_cells * 4));
  CKR(ensure(c, S.offsets, (size_t)n_cells * 4));
  cells_keep_flags_kernel<<<g_c, 256, 0, c->stream>>>((const u64*)S.sort_k[rb].p, (const u32*)S.sort_v[rb].p, n_cells,
                                                      (const u64*)S.cell_total.p, min_count, (u32*)S.flags.p);
  LAUNCH_CHECK("cells_keep_flags");
  u64 n_kept = 0;
  CKR(device_scan<false>(c, (const u32*)S.flags.p, (u32*)S.offsets.p, n_cells, 0, &n_kept));
  CKR(check_device_error(c));
  if (n_kept == 0) return fail(c, ECB_ERR_EMPTY, "no cell reaches the minimum count %llu", (unsigned long long)min_count);
  cr->n_kept_cells = (int64_t)n_kept;
  cells_assign_kernel<<<g_c, 256, 0, c->stream>>>((const u64*)S.sort_k[rb].p, (const u32*)S.sort_v[rb].p, n_cells,
                                                  (const u64*)S.cell_total.p, min_count, (const u32*)S.offsets.p,
                                                  (int32_t*)S.cell_new.p, (int32_t*)c->r_cell_order.p);
  LAUNCH_CHECK("cells_assign");
  cells_ec_keep_kernel<<<grid_for(S.pair_slots, 256, c->sm_count * 8), 256, 0, c->stream>>>(P);
  LAUNCH_CHECK("cells_ec_keep");
  return ECB_OK;
}

// N matrix (CSC) from the kept (EC, cell) pairs (bam_utils_multisample.py:737-747,783-791).
int cells_emit(ecb_ctx* c, CellResult* cr, const u32* ecid_of, u64 n_ec_final) {
  CellScratch& S = c->cells;
  CellParams P = make_cell_params(c, cr);
  P.ecid_of = ecid_of;
  const int g_p = grid_for(S.pair_slots, 256, c->sm_count * 8);
  CKR(ensure(c, S.flags, (size_t)S.pair_slots * 4));
  CKR(ensure(c, S.offsets, (size_t)S.pair_slots * 4));
  cells_pair_flags_kernel<<<g_p, 256, 0, c->stream>>>(P, (u32*)S.flags.p);
  LAUNCH_CHECK("cells_pair_flags");
  u64 nnz = 0;
  CKR(device_scan<false>(c, (const u32*)S.flags.p, (u32*)S.offsets.p, S.pair_slots, 0, &nnz));
  if (nnz == 0 || nnz > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "N matrix has %llu non-zeros", (unsigned long long)nnz);
  cr->nnz_n = (int64_t)nnz;
  CKR(ensure(c, S.sort_k[0], (size_t)nnz * 8));
  CKR(ensure(c, S.sort_v[0], (size_t)nnz * 4));
  cells_pair_emit_kernel<<<g_p, 256, 0, c->stream>>>(P, (const u32*)S.flags.p, (const u32*)S.offsets.p,
                                                     (u64*)S.sort_k[0].p, (u32*)S.sort_v[0].p);
  LAUNCH_CHECK("cells_pair_emit");
  int rb = 0;
  CKR(radix_sort(c, (u32)nnz, 32 + bits_for((u64)cr->n_kept_cells), &rb));
  (void)n_ec_final;
  CKR(ensure(c, c->r_n_indptr, (size_t)(cr->n_kept_cells + 1) * 4));
  CKR(ensure(c, c->r_n_indices, (size_t)nnz * 4));
  CKR(ensure(c, c->r_n_data, (size_t)nnz * 4));
  cells_csc_kernel<<<grid_for(nnz, 256, c->sm_count * 8), 256, 0, c->stream>>>(
      (const u64*)S.sort_k[rb].p, (const u32*)S.sort_v[rb].p, (u32)nnz, (u32)cr->n_kept_cells,
      (int32_t*)c->r_n_indptr.p, (int32_t*)c->r_n_indices.p, (int32_t*)c->r_n_data.p);
  LAUNCH_CHECK("cells_csc");
  return ECB_OK;
}

// N of ecb_finalize_samples (CSC, one column per closed sample) from the pairs and the final EC ids: the pairs per
// sample, uploaded and scanned, are n_indptr; the pairs, keyed by (sample, EC id) and sorted, are the entries.
int samples_emit(ecb_ctx* c, u64 n_ec_final) {
  CellScratch& S = c->cells;
  const u32 n_samples = (u32)c->smp_counts.size();
  const u32 nnz = (u32)c->smp_n_pairs;   // checked against 2^31 - 1 by the caller
  CKR(ensure(c, c->r_n_indptr, ((size_t)n_samples + 1) * 4));
  CKR(ensure(c, c->r_n_indices, std::max<size_t>(nnz, 1) * 4));
  CKR(ensure(c, c->r_n_data, std::max<size_t>(nnz, 1) * 4));
  CK(cudaMemcpyAsync(c->r_n_indptr.p, c->smp_counts.data(), (size_t)n_samples * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemsetAsync((u32*)c->r_n_indptr.p + n_samples, 0, 4, c->stream));
  c->stats.h2d_bytes += (int64_t)n_samples * 4;
  CKR(device_scan<false>(c, (const u32*)c->r_n_indptr.p, (u32*)c->r_n_indptr.p, (u64)n_samples + 1, 0, nullptr));
  if (nnz == 0) return ECB_OK;
  CKR(ensure(c, S.sort_k[0], (size_t)nnz * 8));
  CKR(ensure(c, S.sort_v[0], (size_t)nnz * 4));
  const int ec_bits = bits_for(n_ec_final);
  const int g = grid_for(nnz, 256, c->sm_count * 8);
  ecb_sample_keys_kernel<<<g, 256, 0, c->stream>>>((const uint2*)c->smp_pairs.p, nnz, (const int32_t*)c->r_n_indptr.p,
                                                   n_samples, (const u32*)c->ecid_of.p, ec_bits, (u64*)S.sort_k[0].p,
                                                   (u32*)S.sort_v[0].p);
  LAUNCH_CHECK("sample_keys");
  int rb = 0;
  CKR(radix_sort(c, nnz, ec_bits + bits_for(n_samples), &rb));
  ecb_sample_csc_kernel<<<g, 256, 0, c->stream>>>((const u64*)S.sort_k[rb].p, (const u32*)S.sort_v[rb].p, nnz,
                                                  (1ull << ec_bits) - 1, (int32_t*)c->r_n_indices.p,
                                                  (int32_t*)c->r_n_data.p);
  LAUNCH_CHECK("sample_csc");
  return ECB_OK;
}

void cells_release(ecb_ctx* c) {
  CellScratch& S = c->cells;
  DevBuf* bufs[] = {&S.fe_table, &S.pair_table, &S.cell_key, &S.cell_total, &S.cell_new, &S.sort_k[0], &S.sort_k[1],
                    &S.sort_v[0], &S.sort_v[1], &S.hist, &S.flags, &S.offsets};
  for (DevBuf* b : bufs) release(c, *b);
}

}  // namespace

extern "C" {

int ecb_version(void) { return 2008; }

const char* ecb_last_error(const ecb_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int ecb_create(ecb_ctx** out, int device, int n_targets, int n_haps, int with_cells, int64_t alignments_hint) {
  ecb_ctx* c = nullptr;
  if (!out) return fail(c, ECB_ERR_INVALID, "out is NULL");
  *out = nullptr;
  if (n_targets < 1 || n_targets > ECB_MAX_TARGETS) return fail(c, ECB_ERR_INVALID, "n_targets %d outside [1, 2^26]", n_targets);
  if (n_haps < 1 || n_haps > ECB_MAX_HAPS) return fail(c, ECB_ERR_INVALID, "n_haps %d outside [1, 31]", n_haps);
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
    return fail(c, ECB_ERR_NO_DEVICE, "no CUDA device is visible; libecb200 has no CPU path");
  if (device < 0 || device >= count) return fail(c, ECB_ERR_INVALID, "device %d out of range (%d visible)", device, count);
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(c, ECB_ERR_CUDA, "cudaGetDeviceProperties failed");
  if (prop.major != 10)
    return fail(c, ECB_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
  ecb_ctx* ctx = new ecb_ctx();
  c = ctx;
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  c->n_targets = n_targets;
  c->n_haps = n_haps;
  c->with_cells = with_cells ? 1 : 0;
  c->hint = std::max<int64_t>(alignments_hint, 0);
  auto bail = [&](int code) {
    g_create_error = c->err;
    ecb_destroy(c);
    return code;
  };
  if (cudaSetDevice(device) != cudaSuccess) { fail(c, ECB_ERR_CUDA, "cudaSetDevice failed"); return bail(ECB_ERR_CUDA); }
  {
    // a pool of this context's own, with released memory kept (the default pool would hand it back to the
    // driver at every synchronisation); the device's default pool - which torch and NCCL may share - is
    // left as it is
    cudaMemPoolProps props{};
    props.allocType = cudaMemAllocationTypePinned;
    props.handleTypes = cudaMemHandleTypeNone;
    props.location.type = cudaMemLocationTypeDevice;
    props.location.id = device;
    if (cudaMemPoolCreate(&c->pool, &props) != cudaSuccess) { fail(c, ECB_ERR_CUDA, "cudaMemPoolCreate failed"); return bail(ECB_ERR_CUDA); }
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { fail(c, ECB_ERR_CUDA, "cudaStreamCreate failed"); return bail(ECB_ERR_CUDA); }
  c->stream = c->own_stream;
  for (auto& e : c->ev)
    if (cudaEventCreate(&e) != cudaSuccess) { fail(c, ECB_ERR_CUDA, "cudaEventCreate failed"); return bail(ECB_ERR_CUDA); }
  if (cudaMalloc(&c->d_ctr, sizeof(EcbCounters)) != cudaSuccess || cudaMallocHost(&c->h_ctr, sizeof(EcbCounters)) != cudaSuccess ||
      cudaMallocHost(&c->h_total, 64) != cudaSuccess) {
    fail(c, ECB_ERR_CUDA, "counter allocation failed");
    return bail(ECB_ERR_CUDA);
  }
  *out = c;
  return ECB_OK;
}

int ecb_set_option(ecb_ctx* c, int option, int64_t value) {
  if (!c) return ECB_ERR_INVALID;
  switch (option) {
    case ECB_OPT_RESULT_ON_DEVICE: c->result_on_device = value ? 1 : 0; break;
    case ECB_OPT_TABLE_SLOTS:
      if (c->table_slots) return fail(c, ECB_ERR_STATE, "table already allocated");
      c->opt_table_slots = value; break;
    case ECB_OPT_PAIR_SLOTS:
      if (c->ttable_slots) return fail(c, ECB_ERR_STATE, "table already allocated");
      c->opt_pair_slots = value; break;
    case ECB_OPT_GRID_CTAS: c->opt_grid = value; break;
    case ECB_OPT_HOT_CACHE: c->use_cache = value ? 1 : 0; break;
    case ECB_OPT_VERIFY_KEYS: c->verify_keys = value ? 1 : 0; break;
    case ECB_OPT_CHUNK_LEN: c->opt_chunk_len = value; break;
    case ECB_OPT_PAGEABLE_RESULTS:
      if (c->h_res) return fail(c, ECB_ERR_STATE, "result buffers already allocated");
      c->pageable_results = value ? 1 : 0; break;
    case ECB_OPT_BAM_WINDOW:
      if (value < 0) return fail(c, ECB_ERR_INVALID, "negative window");
      c->opt_bam_window = value; break;
    case ECB_OPT_COLLATE_SLOTS:
      if (value < 0) return fail(c, ECB_ERR_INVALID, "negative slot count");
      c->opt_collate_slots = value; break;
    case ECB_OPT_COLLATE_PIECE:
      if (value < 0 || value > ECB_PUSH_LIMIT) return fail(c, ECB_ERR_INVALID, "collate piece %lld outside [0, %lld]", (long long)value, (long long)ECB_PUSH_LIMIT);
      c->opt_collate_piece = value; break;
    case ECB_OPT_COLLATE_BUDGET:
      if (value < 0) return fail(c, ECB_ERR_INVALID, "negative collate budget");
      c->opt_collate_budget = value; break;
    case ECB_OPT_MAX_READ:
      if (value != 0 && (value < ECB_MAX_READ_ALIGNMENTS || value > ECB_MAX_READ_LIMIT))
        return fail(c, ECB_ERR_INVALID, "max_read %lld is neither 0 nor in [%d, %lld]", (long long)value,
                    ECB_MAX_READ_ALIGNMENTS, (long long)ECB_MAX_READ_LIMIT);
      c->max_read = value ? value : ECB_MAX_READ_LIMIT; break;
    default: return fail(c, ECB_ERR_INVALID, "unknown option %d", option);
  }
  return ECB_OK;
}

int ecb_set_stream(ecb_ctx* c, void* cuda_stream) {
  if (!c) return ECB_ERR_INVALID;
  CK(cudaSetDevice(c->device));
  CK(cudaStreamSynchronize(c->stream));
  c->stream = cuda_stream ? (cudaStream_t)cuda_stream : c->own_stream;
  return ECB_OK;
}

// One launch sequence over one contiguous piece of columns (the whole push, or one piece of a
// pipelined host push).
static int push_one(ecb_ctx* c, const int32_t* read_group, const int32_t* target_idx, const int32_t* hap_idx,
                    const int32_t* cell_idx, int64_t n, int64_t order_base, int drop_last_group, int on_device,
                    u32 push_id) {
  CK(cudaEventRecord(c->ev[0], c->stream));
  const int32_t *rg = read_group, *tg = target_idx, *hp = hap_idx, *cell = cell_idx;
  const size_t col_bytes = (size_t)n * 4;
  auto misaligned = [](const void* p) { return ((uintptr_t)p & 15) != 0; };
  const bool stage = !on_device || misaligned(rg) || misaligned(tg) || misaligned(hp);
  if (stage) {
    const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    CKR(ensure(c, c->st_rg, col_bytes));
    CKR(ensure(c, c->st_tg, col_bytes));
    CKR(ensure(c, c->st_hp, col_bytes));
    CK(cudaMemcpyAsync(c->st_rg.p, rg, col_bytes, kind, c->stream));
    CK(cudaMemcpyAsync(c->st_tg.p, tg, col_bytes, kind, c->stream));
    CK(cudaMemcpyAsync(c->st_hp.p, hp, col_bytes, kind, c->stream));
    rg = (const int32_t*)c->st_rg.p; tg = (const int32_t*)c->st_tg.p; hp = (const int32_t*)c->st_hp.p;
    if (cell) {
      CKR(ensure(c, c->st_cell, col_bytes));
      CK(cudaMemcpyAsync(c->st_cell.p, cell, col_bytes, kind, c->stream));
      cell = (const int32_t*)c->st_cell.p;
    }
    if (!on_device) c->stats.h2d_bytes += (int64_t)col_bytes * (cell ? 4 : 3);
  }

  // capacity: at most half full before the push starts, and - going by the ECs per alignment seen so
  // far - at most about 60 % full after it (a growth in the middle of a push costs a replay)
  while ((u64)c->n_ec * 2 > c->table_slots) CKR(grow_table(c, c->table_slots * 2));
  if (c->n_alignments > 0 && !c->opt_table_slots) {
    const double rate = (double)c->n_ec / (double)c->n_alignments;
    const u64 projected = (u64)c->n_ec + (u64)(rate * (double)n);
    if (projected * 5 > (u64)c->table_slots * 3 && c->table_slots < (1u << 31)) CKR(grow_table(c, pow2_ceil(projected * 2)));
  }
  if (c->with_cells) {
    // the triple table must be able to absorb one new entry per READ of this push without filling up
    // (it has no replay path): count the reads first - one pass over read_group, 4 bytes per alignment
    CK(cudaMemsetAsync(&c->d_ctr->scratch[4], 0, sizeof(u32), c->stream));
    ecb_count_reads_kernel<<<grid_for((u64)n, 1024, c->sm_count * 4), 256, 0, c->stream>>>(rg, (int)n, &c->d_ctr->scratch[4]);
    LAUNCH_CHECK("count_reads");
    CKR(sync_counters(c));
    const u64 reads = c->h_ctr->scratch[4];
    u64 need = ((u64)c->n_triples + reads) * 2;
    if (need > c->ttable_slots) CKR(rebuild_triple_table(c, pow2_ceil(need), nullptr));
  }
  const size_t ov_words = ((size_t)n + 31) / 32;
  CKR(ensure(c, c->overflow_bits, ov_words * 4));
  CK(cudaMemsetAsync(c->overflow_bits.p, 0, ov_words * 4, c->stream));
  CKR(ensure(c, c->lr_list, ((size_t)n / (ECB_MAX_READ_ALIGNMENTS + 1) + 1) * sizeof(uint2)));

  // room for one row entry per alignment of this push: the rows of its new ECs come from distinct reads
  const u64 arena_bound = c->arena_used + (u64)n;
  if (arena_bound > 0xFFFFFFFFull) return fail(c, ECB_ERR_LIMIT, "row arena exceeds 2^32 entries");
  CKR(ensure(c, c->arena, (size_t)arena_bound * sizeof(uint2), true));

  const u32 e_before = c->n_ec;
  CKR(group_prepare_launch(c));
  int grid = 1, chunk_len = 32;
  group_geometry(c, n, &grid, &chunk_len);
  CKR(ensure(c, c->spill, (size_t)grid * ECB_CACHE * sizeof(EcbSpill)));
  GroupParams P = make_group_params(c, rg, tg, hp, cell, n, order_base, drop_last_group, push_id);
  P.chunk_len = chunk_len;
  CK(cudaMemsetAsync(&c->d_ctr->chunk_next, 0, sizeof(u32), c->stream));
  CK(cudaEventRecord(c->ev[1], c->stream));
  if (c->with_cells) ecb_group_insert_kernel<true><<<grid, ECB_GTHREADS, sizeof(GroupSmem), c->stream>>>(P);
  else ecb_group_insert_kernel<false><<<grid, ECB_GTHREADS, sizeof(GroupSmem), c->stream>>>(P);
  LAUNCH_CHECK("group_insert");
  CK(cudaEventRecord(c->ev[2], c->stream));
  // the rows of the ECs the grouping kernel claimed, before the host has seen the counters: the harvest reads only
  // ec_rep / ec_len of claimed ECs, which lie inside this push, also when the kernel set a device error
  CK(cudaEventRecord(c->ev[3], c->stream));
  CKR(harvest_new_rows(c, rg, tg, hp, n, e_before));
  CK(cudaEventRecord(c->ev[4], c->stream));
  CK(cudaEventRecord(c->ev[7], c->stream));   // the end of the push, unless more work follows below
  // the push's round trip: new-EC count, table overflow, deferred reads, device errors, the arena cursor
  CKR(sync_counters(c));
  CKR(check_device_error(c));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev[1], c->ev[2])); c->stats.group_ms = ms;
  CK(cudaEventElapsedTime(&ms, c->ev[3], c->ev[4])); c->stats.harvest_ms = ms;
  const u32 e_harvested = c->h_ctr->n_ec;   // where the harvest's range ended
  // reads longer than ECB_MAX_READ_ALIGNMENTS: the sort-based pass (only when the grouping kernel deferred some)
  const u32 n_def = c->h_ctr->n_deferred;
  LongParams L{};
  float long_ms = 0;
  if (n_def) {
    CK(cudaEventRecord(c->ev[5], c->stream));
    CKR(long_keys(c, P, tg, hp, n_def, &L));
    CK(cudaEventRecord(c->ev[6], c->stream));
    CKR(sync_counters(c));
    CKR(check_device_error(c));
    CK(cudaEventElapsedTime(&long_ms, c->ev[5], c->ev[6]));
  }
  DevBuf spill_in;
  // table too full: grow, then replay just what did not fit
  while (c->h_ctr->n_overflow || c->h_ctr->n_spill || c->h_ctr->n_deferred_fail) {
    c->stats.overflow_reads += c->h_ctr->n_overflow;
    const u32 n_spill = c->h_ctr->n_spill;
    if (c->table_slots >= (1u << 31)) return fail(c, ECB_ERR_LIMIT, "EC table cannot grow beyond 2^31 slots");
    if (n_spill) {
      CKR(ensure(c, spill_in, (size_t)n_spill * sizeof(EcbSpill)));
      CK(cudaMemcpyAsync(spill_in.p, c->spill.p, (size_t)n_spill * sizeof(EcbSpill), cudaMemcpyDeviceToDevice, c->stream));
    }
    CKR(grow_table(c, c->table_slots * 4u > c->table_slots ? c->table_slots * 4u : (1u << 31)));
    CK(cudaMemsetAsync(&c->d_ctr->n_overflow, 0, sizeof(u32), c->stream));
    CK(cudaMemsetAsync(&c->d_ctr->n_spill, 0, sizeof(u32), c->stream));
    P = make_group_params(c, rg, tg, hp, cell, n, order_base, drop_last_group, push_id);
    const int rg_grid = grid_for(ov_words, 256, c->sm_count * 8);
    if (c->with_cells) ecb_replay_kernel<true><<<rg_grid, 256, 0, c->stream>>>(P);
    else ecb_replay_kernel<false><<<rg_grid, 256, 0, c->stream>>>(P);
    LAUNCH_CHECK("replay");
    if (n_spill) {
      ecb_spill_replay_kernel<<<grid_for(n_spill, 256, c->sm_count * 8), 256, 0, c->stream>>>(
          P, (const EcbSpill*)spill_in.p, n_spill);
      LAUNCH_CHECK("spill_replay");
    }
    if (c->h_ctr->n_deferred_fail) {   // the deferred reads still pending go in again; their keys are kept
      CK(cudaMemsetAsync(&c->d_ctr->n_deferred_fail, 0, sizeof(u32), c->stream));
      ecb_long_insert_kernel<<<grid_for(n_def, ECB_LONG_THREADS, c->sm_count), ECB_LONG_THREADS, 0, c->stream>>>(P, L);
      LAUNCH_CHECK("long_insert");
    }
    CKR(sync_counters(c));
    CKR(check_device_error(c));
  }
  release(c, spill_in);
  if (c->h_ctr->n_triple_overflow) return fail(c, ECB_ERR_LIMIT, "(file, EC, cell) table ran out of probes");
  c->n_ec = c->h_ctr->n_ec;
  c->n_triples = c->h_ctr->n_triples;
  // a push without replay, long reads or verification ends here: nothing was enqueued after the round trip above,
  // so the caller's buffers are free and the counters are current
  const bool more = c->n_ec > e_harvested || n_def || c->verify_keys;
  float replay_harvest_ms = 0;
  if (c->n_ec > e_harvested) {   // ECs claimed by the replay or the deferred long-read pass
    CK(cudaEventRecord(c->ev[3], c->stream));
    CKR(harvest_new_rows(c, rg, tg, hp, n, e_harvested));
    CK(cudaEventRecord(c->ev[4], c->stream));
  }
  if (n_def) {
    CK(cudaEventRecord(c->ev[5], c->stream));
    CKR(long_rows(c, L));
    CK(cudaEventRecord(c->ev[6], c->stream));
    CK(cudaMemsetAsync(&c->d_ctr->n_deferred, 0, sizeof(u32), c->stream));   // the list is empty for the next push
  }
  if (more) CK(cudaEventRecord(c->ev[7], c->stream));
  if (c->verify_keys) {
    VerifyParams V{};
    V.rg = rg; V.tg = tg; V.hp = hp; V.n = (int)n; V.drop_last = drop_last_group;
    V.table = (const EcbEntry*)c->table.p;
    V.mask = c->table_slots - 1;
    V.row_len = (const u32*)c->row_len.p;
    V.row_off = (const u32*)c->row_off.p;
    V.arena = (const uint2*)c->arena.p;
    V.ctr = c->d_ctr;
    ecb_verify_kernel<<<grid_for((u64)n, 256, c->sm_count * 16), 256, 0, c->stream>>>(V);
    LAUNCH_CHECK("verify");
  }
  if (more) {   // a second round trip: the caller's buffers are free again, the counters (arena cursor, device-side
                // errors of the replay's harvest, the long-read rows and the verification) are current on the host
    CKR(sync_counters(c));
    CKR(check_device_error(c));
  }
  if (c->n_ec > e_harvested) {
    CK(cudaEventElapsedTime(&replay_harvest_ms, c->ev[3], c->ev[4]));
    c->stats.harvest_ms += replay_harvest_ms;
  }
  CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[7])); c->stats.push_ms = ms;
  if (n_def) {
    CK(cudaEventElapsedTime(&ms, c->ev[5], c->ev[6]));
    c->stats.long_reads += n_def;
    c->stats.long_ms += long_ms + ms;
  }

  c->min_base = std::min<u64>(c->min_base, (u64)order_base);
  c->max_end = std::max<u64>(c->max_end, (u64)order_base + (u64)n);
  c->n_alignments += n;
  c->stats.table_slots = c->table_slots;
  c->stats.table_used = c->n_ec;
  return ECB_OK;
}

// Host columns of a large push are sent in read-aligned pieces on a second stream, two staging sets
// deep, so that the copy of piece i+1 runs while piece i is grouped and harvested.  The pieces share
// the push id (the "file" of the per-cell path) and only the last one drops the last read.
#define ECB_PIPE_PIECE (8ll << 20)   // alignments per piece (96 MB of columns)

static int push_pipelined(ecb_ctx* c, const int32_t* rg, const int32_t* tg, const int32_t* hp, const int32_t* cell,
                          int64_t n, int64_t order_base, int drop_last_group, u32 push_id) {
  std::vector<int64_t> cut{0};
  while (cut.back() < n) {
    int64_t b = std::min<int64_t>(n, cut.back() + ECB_PIPE_PIECE);
    while (b < n && rg[b] == rg[b - 1]) ++b;   // never split a read
    cut.push_back(b);
  }
  const int pieces = (int)cut.size() - 1;
  int64_t longest = 0;
  for (int i = 0; i < pieces; ++i) longest = std::max(longest, cut[i + 1] - cut[i]);
  if (!c->copy_stream) {
    CK(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&c->copy_done[0], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->copy_done[1], cudaEventDisableTiming));
  }
  DevBuf* set[2][4] = {{&c->st_rg, &c->st_tg, &c->st_hp, &c->st_cell}, {&c->st2_rg, &c->st2_tg, &c->st2_hp, &c->st2_cell}};
  const int ncols = cell ? 4 : 3;
  for (int k = 0; k < 2; ++k)
    for (int j = 0; j < ncols; ++j) CKR(ensure(c, *set[k][j], (size_t)longest * 4));
  CK(cudaStreamSynchronize(c->stream));   // the staging sets exist before the copy stream touches them
  const int32_t* src[4] = {rg, tg, hp, cell};
  auto send = [&](int i) -> int {
    const size_t bytes = (size_t)(cut[i + 1] - cut[i]) * 4;
    for (int j = 0; j < ncols; ++j)
      CK(cudaMemcpyAsync(set[i & 1][j]->p, src[j] + cut[i], bytes, cudaMemcpyHostToDevice, c->copy_stream));
    CK(cudaEventRecord(c->copy_done[i & 1], c->copy_stream));
    c->stats.h2d_bytes += (int64_t)bytes * ncols;
    return ECB_OK;
  };
  CKR(send(0));
  for (int i = 0; i < pieces; ++i) {
    if (i + 1 < pieces) CKR(send(i + 1));   // its staging set was last read by piece i-1, which has completed
    CK(cudaStreamWaitEvent(c->stream, c->copy_done[i & 1], 0));
    const int rc = push_one(c, (const int32_t*)set[i & 1][0]->p, (const int32_t*)set[i & 1][1]->p,
                            (const int32_t*)set[i & 1][2]->p, cell ? (const int32_t*)set[i & 1][3]->p : nullptr,
                            cut[i + 1] - cut[i], order_base + cut[i], drop_last_group && i + 1 == pieces, 1, push_id);
    if (rc != ECB_OK) {
      cudaStreamSynchronize(c->copy_stream);
      return rc;
    }
  }
  return ECB_OK;
}

int ecb_push(ecb_ctx* c, const int32_t* read_group, const int32_t* target_idx, const int32_t* hap_idx,
             const int32_t* cell_idx, int64_t n, int64_t order_base, int drop_last_group, int on_device) {
  if (!c) return ECB_ERR_INVALID;
  if (n < 0 || order_base < 0) return fail(c, ECB_ERR_INVALID, "negative n or order_base");
  if (n > ECB_PUSH_LIMIT) return fail(c, ECB_ERR_LIMIT, "a push is limited to 2^31-8192 alignments; split it");
  if (n > 0 && (!read_group || !target_idx || !hap_idx)) return fail(c, ECB_ERR_INVALID, "NULL column");
  if (c->with_cells && n > 0 && !cell_idx) return fail(c, ECB_ERR_INVALID, "context has cells but cell_idx is NULL");
  if (!c->with_cells && cell_idx) return fail(c, ECB_ERR_INVALID, "cell_idx given but context was created without cells");
  if (c->ecr_broken || c->ecr_rows >= 0)
    return fail(c, ECB_ERR_STATE, c->ecr_broken ? "an ecb_push_ecs failed after it changed the EC table: ecb_reset first"
                                                : "the EC rows of the last ecb_push_ecs await ecb_sample_append");
  CK(cudaSetDevice(c->device));
  if (!c->table_slots) CKR(init_table(c, n));
  const u32 push_id = c->push_count++;
  c->stats.long_reads = 0;   // "the last push": summed over the pieces of a pipelined push
  c->stats.long_ms = 0;
  if (n == 0) return ECB_OK;
  c->smp_open += n;
  order_base += (int64_t)c->smp_base;   // 0 until a sample is closed
  if (!on_device && n >= 2 * ECB_PIPE_PIECE)
    return push_pipelined(c, read_group, target_idx, hap_idx, cell_idx, n, order_base, drop_last_group, push_id);
  return push_one(c, read_group, target_idx, hap_idx, cell_idx, n, order_base, drop_last_group, on_device, push_id);
}

// ecb_finalize, and with samples ecb_finalize_samples: the same A and EC ids, N from the closed samples' pairs.
static int finalize(ecb_ctx* c, int64_t min_cell_count, bool samples, ecb_result* out) {
  memset(out, 0, sizeof *out);
  CK(cudaSetDevice(c->device));
  if (!c->table_slots || c->n_ec == 0) return fail(c, ECB_ERR_EMPTY, "no equivalence classes (nothing pushed)");
  CK(cudaEventRecord(c->ev[0], c->stream));
  const u32 n_prov = c->n_ec;   // the host mirror of the counters is current: every push ends with a sync
  const u64 span = c->max_end - c->min_base;
  if (span > (1ull << 34)) return fail(c, ECB_ERR_LIMIT, "order_base range spans more than 2^34 positions");
  const size_t words = (size_t)((span + 31) / 32) + 1;

  CKR(ensure(c, c->bitmap, words * 4));
  CKR(ensure(c, c->word_rank, words * 4));
  CKR(ensure(c, c->first_rel, (size_t)n_prov * 8));
  CKR(ensure(c, c->ecid_of, (size_t)n_prov * 4));
  CK(cudaMemsetAsync(c->bitmap.p, 0, words * 4, c->stream));

  FinalizeParams F{};
  F.table = (const EcbEntry*)c->table.p;
  F.ec_slot = (const u32*)c->ec_slot.p;
  F.row_len = (const u32*)c->row_len.p;
  F.row_off = (const u32*)c->row_off.p;
  F.arena = (const uint2*)c->arena.p;
  F.n_ec = n_prov;
  F.min_base = c->min_base;
  F.bitmap = (u32*)c->bitmap.p;
  F.word_rank = (const u32*)c->word_rank.p;
  F.first_rel = (u64*)c->first_rel.p;
  F.ecid_of = (u32*)c->ecid_of.p;
  CKR(ensure(c, c->count_of, (size_t)n_prov * 4));
  F.count_of = (u32*)c->count_of.p;

  CellResult cr{};
  if (c->with_cells) {
    CKR(cells_prepare(c, min_cell_count, &cr));   // cell order, kept cells, ec_keep flags
    F.ec_keep = (const u32*)c->ec_keep.p;
  }

  const int g_ec = grid_for(n_prov, 256, c->sm_count * 8);
  ecb_fin_mark_kernel<<<g_ec, 256, 0, c->stream>>>(F);
  LAUNCH_CHECK("fin_mark");
  u64 n_kept = n_prov;
  if (c->with_cells) {
    CKR(device_scan<true>(c, F.bitmap, (u32*)c->word_rank.p, words, 0, &n_kept));   // the cell filter decides: host round trip
    if (n_kept == 0) return fail(c, ECB_ERR_EMPTY, "no equivalence class survives the cell filter");
  } else {
    // single sample: every EC is kept, so E is known; the count of first-occurrence bits is checked against it
    // when the one round trip of this call brings it back (it differs when order_base ranges overlapped)
    CKR(device_scan<true>(c, F.bitmap, (u32*)c->word_rank.p, words, 0, nullptr));
    CK(cudaMemcpyAsync(c->h_total + 1, scan_total(c, words), sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
  }
  const u64 E = n_kept;
  if (E + 1 > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "more than 2^31 equivalence classes");

  CKR(ensure(c, c->r_a_indptr, (E + 1) * 4));
  CKR(ensure(c, c->prov_of, E * 4));
  F.a_indptr = (int32_t*)c->r_a_indptr.p;
  F.prov_of = (u32*)c->prov_of.p;
  F.n_final = (u32)E;
  const bool single = !c->with_cells && !samples;
  if (single) {
    CKR(ensure(c, c->r_n_indptr, 2 * 4));
    CKR(ensure(c, c->r_n_indices, E * 4));
    CKR(ensure(c, c->r_n_data, E * 4));
    F.n_indptr = (int32_t*)c->r_n_indptr.p;
    F.n_indices = (int32_t*)c->r_n_indices.p;
    F.n_data = (int32_t*)c->r_n_data.p;
  }
  ecb_fin_rank_kernel<<<g_ec, 256, 0, c->stream>>>(F);
  LAUNCH_CHECK("fin_rank");
  // rows in id order, indptr scanned in the same pass; the arena's fill (known on the host since the last push)
  // bounds the number of non-zeros, so the result arrays need not wait for the exact figure
  const u64 z_bound = std::max<u64>(c->arena_used, 1);
  if (z_bound > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "A matrix may have more than 2^31-1 non-zeros");
  CKR(ensure(c, c->r_a_indices, z_bound * 4));
  CKR(ensure(c, c->r_a_data, z_bound * 4));
  F.a_indices = (int32_t*)c->r_a_indices.p;
  F.a_data = (int32_t*)c->r_a_data.p;
  F.z_cap = z_bound;
  F.n_tiles = (u32)((E + FIN_EMIT_TILE - 1) / FIN_EMIT_TILE);
  CKR(scan_state(c, F.n_tiles, &F.scan_state));
  if (single) ecb_fin_emit_kernel<true><<<F.n_tiles, FIN_EMIT_THREADS, 0, c->stream>>>(F);
  else ecb_fin_emit_kernel<false><<<F.n_tiles, FIN_EMIT_THREADS, 0, c->stream>>>(F);
  LAUNCH_CHECK("fin_emit");
  CK(cudaMemcpyAsync(c->h_total, F.scan_state + F.n_tiles + 1, sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
  c->stats.d2h_bytes += 2 * sizeof(u64);
  CellResult cr2 = cr;
  if (c->with_cells) CKR(cells_emit(c, &cr2, (const u32*)c->ecid_of.p, E));   // N matrix as CSC
  else if (samples) CKR(samples_emit(c, E));
  CKR(sync_counters(c));   // the round trip of this call: non-zeros, first-occurrence bits, device-side errors
  CKR(check_device_error(c));
  const u64 Z = *c->h_total;
  if (!c->with_cells && c->h_total[1] != n_prov)
    return fail(c, ECB_ERR_INVALID, "order_base ranges of different pushes overlap (%llu first positions for %u ECs)",
                (unsigned long long)c->h_total[1], n_prov);
  if (Z > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "A matrix has more than 2^31-1 non-zeros");

  int64_t n_samples = 1, nnz_n = (int64_t)E;
  if (c->with_cells) {
    n_samples = cr2.n_kept_cells;
    nnz_n = cr2.nnz_n;
  } else if (samples) {
    n_samples = (int64_t)c->smp_counts.size();
    nnz_n = (int64_t)c->smp_n_pairs;
  }

  out->n_ec = (int64_t)E;
  out->nnz_a = (int64_t)Z;
  out->n_samples = n_samples;
  out->nnz_n = nnz_n;
  out->n_reads = (int64_t)c->h_ctr->n_reads;
  out->n_alignments = c->n_alignments;
  if (c->result_on_device) {
    out->a_indptr = (const int32_t*)c->r_a_indptr.p;
    out->a_indices = (const int32_t*)c->r_a_indices.p;
    out->a_data = (const int32_t*)c->r_a_data.p;
    out->n_indptr = (const int32_t*)c->r_n_indptr.p;
    out->n_indices = (const int32_t*)c->r_n_indices.p;
    out->n_data = (const int32_t*)c->r_n_data.p;
    out->cell_order = c->with_cells ? (const int32_t*)c->r_cell_order.p : nullptr;
  } else {
    const size_t sizes[7] = {(size_t)(E + 1) * 4, (size_t)Z * 4, (size_t)Z * 4, (size_t)(n_samples + 1) * 4,
                             (size_t)nnz_n * 4, (size_t)nnz_n * 4, c->with_cells ? (size_t)n_samples * 4 : 0};
    const void* src[7] = {c->r_a_indptr.p, c->r_a_indices.p, c->r_a_data.p, c->r_n_indptr.p,
                          c->r_n_indices.p, c->r_n_data.p, c->r_cell_order.p};
    size_t total = 0, offs[7];
    for (int i = 0; i < 7; ++i) { offs[i] = total; total += (sizes[i] + 63) & ~(size_t)63; }
    if (total > c->h_res_bytes) {
      if (c->h_res) {
        if (c->pageable_results) free(c->h_res); else CK(cudaFreeHost(c->h_res));
      }
      c->h_res = nullptr;
      c->h_res_bytes = 0;
      if (c->pageable_results) {
        c->h_res = malloc(total + total / 4);
        if (!c->h_res) return fail(c, ECB_ERR_CUDA, "out of host memory for %zu result bytes", total);
      } else {
        CK(cudaMallocHost(&c->h_res, total + total / 4));
      }
      c->h_res_bytes = total + total / 4;
    }
    char* base = (char*)c->h_res;
    for (int i = 0; i < 7; ++i)
      if (sizes[i]) {
        CK(cudaMemcpyAsync(base + offs[i], src[i], sizes[i], cudaMemcpyDeviceToHost, c->stream));
        c->stats.d2h_bytes += (int64_t)sizes[i];
      }
    out->a_indptr = (const int32_t*)(base + offs[0]);
    out->a_indices = (const int32_t*)(base + offs[1]);
    out->a_data = (const int32_t*)(base + offs[2]);
    out->n_indptr = (const int32_t*)(base + offs[3]);
    out->n_indices = (const int32_t*)(base + offs[4]);
    out->n_data = (const int32_t*)(base + offs[5]);
    out->cell_order = c->with_cells ? (const int32_t*)(base + offs[6]) : nullptr;
  }
  CK(cudaEventRecord(c->ev[1], c->stream));
  CK(cudaStreamSynchronize(c->stream));
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  c->stats.finalize_ms = ms;
  return ECB_OK;
}

int ecb_finalize(ecb_ctx* c, int64_t min_cell_count, ecb_result* out) {
  if (!c || !out) return ECB_ERR_INVALID;
  if (c->ecr_used) {
    memset(out, 0, sizeof *out);
    return fail(c, ECB_ERR_STATE, "the context holds ECs given as EC rows (ecb_push_ecs), which carry no reads: "
                                  "ecb_finalize_samples gives their counts");
  }
  return finalize(c, min_cell_count, false, out);
}

int ecb_sample_close(ecb_ctx* c, int64_t* nonzeros) {
  if (!c) return ECB_ERR_INVALID;
  if (nonzeros) *nonzeros = 0;
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "samples are closed on single-sample contexts only");
  if (c->ecr_broken || c->ecr_rows >= 0)
    return fail(c, ECB_ERR_STATE, c->ecr_broken ? "an ecb_push_ecs failed after it changed the EC table: ecb_reset first"
                                                : "the EC rows of the last ecb_push_ecs await ecb_sample_append");
  CK(cudaSetDevice(c->device));
  const u32 n = c->table_slots ? c->n_ec : 0;   // current on the host: every push ends with a sync
  u32 added = 0;
  float ms = 0;
  if (n) {
    CKR(ensure(c, c->smp_last, (size_t)n * 4, true));
    CKR(ensure(c, c->smp_pairs, (size_t)(c->smp_n_pairs + n) * sizeof(uint2), true));
    CK(cudaEventRecord(c->ev[0], c->stream));
    CK(cudaMemsetAsync(&c->d_ctr->scratch[6], 0, sizeof(u32), c->stream));
    ecb_sample_close_kernel<<<grid_for(n, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        (const EcbEntry*)c->table.p, (const u32*)c->ec_slot.p, n, c->smp_n_ec, (u32*)c->smp_last.p,
        (uint2*)c->smp_pairs.p + c->smp_n_pairs, &c->d_ctr->scratch[6]);
    LAUNCH_CHECK("sample_close");
    CK(cudaEventRecord(c->ev[1], c->stream));
    CKR(sync_counters(c));   // the call's one round trip brings the pair count back
    added = c->h_ctr->scratch[6];
    CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  }
  c->smp_n_ec = n;
  c->smp_n_pairs += added;
  c->smp_counts.push_back(added);
  c->smp_base = c->max_end;   // the next sample's order keys follow this one's
  c->smp_open = 0;
  c->stats.samples++;
  c->stats.sample_pairs += added;
  c->stats.sample_ms += ms;
  if (nonzeros) *nonzeros = added;
  return ECB_OK;
}

int ecb_finalize_samples(ecb_ctx* c, ecb_result* out) {
  if (!c || !out) return ECB_ERR_INVALID;
  memset(out, 0, sizeof *out);
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "samples are closed on single-sample contexts only");
  if (c->smp_open) return fail(c, ECB_ERR_INVALID, "%lld alignments were pushed after the last ecb_sample_close",
                               (long long)c->smp_open);
  if (c->ecr_broken) return fail(c, ECB_ERR_STATE, "an ecb_push_ecs failed after it changed the EC table: ecb_reset first");
  if (c->ecr_rows >= 0)
    return fail(c, ECB_ERR_INVALID, "the %lld EC rows of the last ecb_push_ecs await ecb_sample_append",
                (long long)c->ecr_rows);
  if (c->smp_n_pairs > 0x7FFFFFFFull)
    return fail(c, ECB_ERR_LIMIT, "N matrix has %llu non-zeros (more than 2^31-1)", (unsigned long long)c->smp_n_pairs);
  return finalize(c, 0, true, out);
}

// ---- ECs given as EC-file rows (ecb_push_ecs / ecb_sample_append; kernels in ecb_ecrows.cuh) --------------------
// A host copy of an index pointer of n + 1 entries (copied back when it is device memory), checked before any kernel
// indexes with it: it runs from 0 to nnz and never decreases; with rows (A) no two entries are equal either, since an
// empty row is no set of elements.
static int host_indptr(ecb_ctx* c, const int32_t* p, int64_t n, int64_t nnz, int on_device, bool rows, const char* what,
                       std::vector<int32_t>& copy, const int32_t** out) {
  if (on_device) {
    copy.resize((size_t)n + 1);
    CK(cudaMemcpyAsync(copy.data(), p, ((size_t)n + 1) * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->stats.d2h_bytes += (n + 1) * 4;
    p = copy.data();
  }
  if (p[0] != 0 || p[n] != nnz)
    return fail(c, ECB_ERR_FORMAT, "%s: %s runs from %d to %d, not from 0 to nnz = %lld", what, rows ? "a_indptr" : "n_indptr",
                p[0], p[n], (long long)nnz);
  for (int64_t i = 0; i < n; ++i) {
    if (p[i + 1] < p[i])
      return fail(c, ECB_ERR_FORMAT, "%s: %s decreases at %lld (%d after %d)", what, rows ? "a_indptr" : "n_indptr",
                  (long long)i + 1, p[i + 1], p[i]);
    if (rows && p[i + 1] == p[i]) return fail(c, ECB_ERR_FORMAT, "%s: row %lld is empty", what, (long long)i);
  }
  *out = p;
  return ECB_OK;
}

// Device columns of an EC-file array: the caller's when they are device memory, else staged with one copy each.
static const int32_t* ecr_upload(ecb_ctx* c, DevBuf& st, const int32_t* p, int64_t n, int on_device, int* rc) {
  *rc = ECB_OK;
  if (on_device || n == 0) return p;
  if ((*rc = ensure(c, st, (size_t)n * 4)) != ECB_OK) return nullptr;
  if (cudaMemcpyAsync(st.p, p, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream) != cudaSuccess) {
    *rc = fail(c, ECB_ERR_CUDA, "cudaMemcpyAsync of an EC-file array failed");
    return nullptr;
  }
  c->stats.h2d_bytes += n * 4;
  return (const int32_t*)st.p;
}

static int ecr_state(ecb_ctx* c) {
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "EC rows go into single-sample contexts only");
  if (c->ecr_broken) return fail(c, ECB_ERR_STATE, "an ecb_push_ecs failed after it changed the EC table: ecb_reset first");
  return ECB_OK;
}

int ecb_push_ecs(ecb_ctx* c, const int32_t* a_indptr, const int32_t* a_indices, const int32_t* a_data, int64_t n_ec,
                 int64_t nnz, int64_t order_base, int on_device) {
  if (!c) return ECB_ERR_INVALID;
  CKR(ecr_state(c));
  if (n_ec < 0 || nnz < 0 || order_base < 0) return fail(c, ECB_ERR_INVALID, "negative n_ec, nnz or order_base");
  if (n_ec > (1ll << 30) || nnz > 0x7FFFFFFFll)
    return fail(c, ECB_ERR_LIMIT, "one push of EC rows takes at most 2^30 rows and 2^31 - 1 entries");
  if (!a_indptr || (nnz > 0 && (!a_indices || !a_data))) return fail(c, ECB_ERR_INVALID, "NULL array");
  if (c->smp_open)
    return fail(c, ECB_ERR_STATE, "%lld alignments were pushed after the last ecb_sample_close: close that sample first",
                (long long)c->smp_open);
  CK(cudaSetDevice(c->device));
  std::vector<int32_t> ip_copy;
  const int32_t* ip = nullptr;
  CKR(host_indptr(c, a_indptr, n_ec, nnz, on_device, true, "EC rows", ip_copy, &ip));
  if (!c->table_slots) CKR(init_table(c, n_ec * 8));
  const u64 base = c->smp_base + (u64)order_base;
  if (n_ec == 0) {
    c->ecr_rows = 0;
    c->ecr_used = true;
    c->stats.ec_pushes++;
    return ECB_OK;
  }
  CK(cudaEventRecord(c->ev[0], c->stream));
  int rc = ECB_OK;
  EcrParams R{};
  R.indptr = ecr_upload(c, c->st_rg, a_indptr, n_ec + 1, on_device, &rc);
  CKR(rc);
  R.indices = ecr_upload(c, c->st_tg, a_indices, nnz, on_device, &rc);
  CKR(rc);
  R.data = ecr_upload(c, c->st_hp, a_data, nnz, on_device, &rc);
  CKR(rc);
  const u32 n = (u32)n_ec;
  CKR(ensure(c, c->ecr_acc, (size_t)n * sizeof(Mix4)));
  CKR(ensure(c, c->ecr_slot, (size_t)n * 4));
  CKR(ensure(c, c->ecr_ec, (size_t)n * 4));
  CKR(ensure(c, c->ecr_dst, (size_t)n * 4));
  CK(cudaMemsetAsync(c->ecr_acc.p, 0, (size_t)n * sizeof(Mix4), c->stream));
  CK(cudaMemsetAsync(c->d_ctr->ecr_bad, 0xFF, sizeof c->d_ctr->ecr_bad, c->stream));
  R.n_rows = n;
  R.nnz = (u32)nnz;
  R.n_targets = c->n_targets;
  R.n_haps = c->n_haps;
  R.base = base;
  R.acc = (Mix4*)c->ecr_acc.p;
  R.row_slot = (u32*)c->ecr_slot.p;
  R.row_ec = (u32*)c->ecr_ec.p;
  R.row_dst = (u32*)c->ecr_dst.p;
  R.ctr = c->d_ctr;
  const int g_z = grid_for(nnz, ECR_THREADS, c->sm_count * 16), g_r = grid_for(n, ECR_THREADS, c->sm_count * 16);
  ecb_ecr_keys_kernel<<<g_z, ECR_THREADS, 0, c->stream>>>(R);
  LAUNCH_CHECK("ecr_keys");
  CKR(sync_counters(c));   // the value checks come back before anything is inserted
  const u32* bad = c->h_ctr->ecr_bad;
  auto row_of = [&](u32 i) { return (long long)(std::upper_bound(ip, ip + n_ec + 1, (int32_t)i) - ip) - 1; };
  if (bad[ECR_BAD_TARGET] != ECB_NONE)
    return fail(c, ECB_ERR_FORMAT, "EC rows: target outside [0, %d) at entry %u (row %lld)", c->n_targets,
                bad[ECR_BAD_TARGET], row_of(bad[ECR_BAD_TARGET]));
  if (bad[ECR_BAD_ORDER] != ECB_NONE)
    return fail(c, ECB_ERR_FORMAT, "EC rows: targets not strictly ascending at entry %u (row %lld)", bad[ECR_BAD_ORDER],
                row_of(bad[ECR_BAD_ORDER]));
  if (bad[ECR_BAD_MASK] != ECB_NONE)
    return fail(c, ECB_ERR_FORMAT, "EC rows: haplotype mask 0 or with a bit at or above n_haps = %d at entry %u (row %lld)",
                c->n_haps, bad[ECR_BAD_MASK], row_of(bad[ECR_BAD_MASK]));

  // from here on the table changes: the rows of an earlier push can no longer be appended
  c->ecr_rows = -1;
  while ((u64)(c->n_ec + n) * 2 > c->table_slots) {   // at most half full after the insert: no replay path
    if (c->table_slots >= (1u << 31)) return fail(c, ECB_ERR_LIMIT, "EC table cannot grow beyond 2^31 slots");
    CKR(grow_table(c, c->table_slots * 2));
  }
  const u64 bound = c->arena_used + (u64)nnz;
  if (bound > 0xFFFFFFFFull) return fail(c, ECB_ERR_LIMIT, "row arena exceeds 2^32 entries");
  CKR(ensure(c, c->arena, (size_t)bound * sizeof(uint2), true));
  const u32 ids_bound = c->n_ec + n;
  if (ids_bound > c->ecr_seen_n) {
    CKR(ensure(c, c->ecr_seen, (size_t)ids_bound * 4, true));
    CK(cudaMemsetAsync((u32*)c->ecr_seen.p + c->ecr_seen_n, 0, (size_t)(ids_bound - c->ecr_seen_n) * 4, c->stream));
    c->ecr_seen_n = ids_bound;
  }
  R.seen = (u32*)c->ecr_seen.p;
  R.tag = ++c->ecr_tag;
  c->ecr_broken = true;   // until the rows are in
  const GroupParams P = make_group_params(c, nullptr, nullptr, nullptr, nullptr, 0, 0, 0, 0);
  ecb_ecr_insert_kernel<<<g_r, ECR_THREADS, 0, c->stream>>>(P, R);
  LAUNCH_CHECK("ecr_insert");
  ecb_ecr_reserve_kernel<<<g_r, ECR_THREADS, 0, c->stream>>>(R, (const EcbEntry*)c->table.p, (u32*)c->row_len.p,
                                                             (u32*)c->row_off.p);
  LAUNCH_CHECK("ecr_reserve");
  ecb_ecr_copy_kernel<<<g_z, ECR_THREADS, 0, c->stream>>>(R, (uint2*)c->arena.p);
  LAUNCH_CHECK("ecr_copy");
  CK(cudaEventRecord(c->ev[2], c->stream));
  ecb_ecr_check_kernel<<<g_z, ECR_THREADS, 0, c->stream>>>(R, (const u32*)c->row_len.p, (const u32*)c->row_off.p,
                                                           (const uint2*)c->arena.p);
  LAUNCH_CHECK("ecr_check");
  CK(cudaEventRecord(c->ev[3], c->stream));
  CK(cudaEventRecord(c->ev[1], c->stream));
  CKR(sync_counters(c));
  if (bad[ECR_BAD_DUPLICATE] != ECB_NONE)
    return fail(c, ECB_ERR_FORMAT, "EC rows: row %u holds the set of another row of the same push (duplicate rows)",
                bad[ECR_BAD_DUPLICATE]);
  if (bad[ECR_BAD_PROBE] != ECB_NONE) return fail(c, ECB_ERR_LIMIT, "EC rows: the EC table ran out of probes at row %u",
                                                  bad[ECR_BAD_PROBE]);
  if (bad[ECR_BAD_COLLISION] != ECB_NONE)
    return fail(c, ECB_ERR_LIMIT, "EC rows: row %u and a different set share one 128-bit key (key collision)",
                bad[ECR_BAD_COLLISION]);
  CKR(check_device_error(c));
  c->ecr_broken = false;
  const u32 claimed = c->h_ctr->n_ec - c->n_ec;
  c->n_ec = c->h_ctr->n_ec;
  c->min_base = std::min<u64>(c->min_base, base);
  c->max_end = std::max<u64>(c->max_end, base + n);
  c->smp_base = c->max_end;   // a later push of rows follows these, whether they get their counts or not
  c->ecr_rows = n_ec;
  c->ecr_used = true;
  float ms = 0, check_ms = 0;
  CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  CK(cudaEventElapsedTime(&check_ms, c->ev[2], c->ev[3]));
  c->stats.ec_pushes++;
  c->stats.ec_rows += n_ec;
  c->stats.ec_claimed += claimed;
  c->stats.ec_ms += ms;
  c->stats.ec_check_ms += check_ms;
  c->stats.table_slots = c->table_slots;
  c->stats.table_used = c->n_ec;
  return ECB_OK;
}

int ecb_sample_append(ecb_ctx* c, const int32_t* n_indptr, const int32_t* n_indices, const int32_t* n_data,
                      int64_t n_samples, int64_t nnz, int on_device, int64_t* nonzeros) {
  if (!c) return ECB_ERR_INVALID;
  if (nonzeros) *nonzeros = 0;
  CKR(ecr_state(c));
  if (n_samples < 0 || nnz < 0) return fail(c, ECB_ERR_INVALID, "negative n_samples or nnz");
  if (n_samples > 0x7FFFFFFFll || nnz > 0x7FFFFFFFll)
    return fail(c, ECB_ERR_LIMIT, "one append takes at most 2^31 - 1 samples and 2^31 - 1 entries");
  if (!n_indptr || (nnz > 0 && (!n_indices || !n_data))) return fail(c, ECB_ERR_INVALID, "NULL array");
  if (c->ecr_rows < 0) return fail(c, ECB_ERR_STATE, "no EC rows await their samples: ecb_push_ecs first");
  CK(cudaSetDevice(c->device));
  std::vector<int32_t> ip_copy;
  const int32_t* ip = nullptr;
  CKR(host_indptr(c, n_indptr, n_samples, nnz, on_device, false, "N", ip_copy, &ip));
  const u32 S = (u32)n_samples, z = (u32)nnz;
  std::vector<u32> cols(S, 0u);
  float ms = 0;
  if (z) {
    CK(cudaEventRecord(c->ev[0], c->stream));
    int rc = ECB_OK;
    const int32_t* d_ip = ecr_upload(c, c->st_rg, n_indptr, n_samples + 1, on_device, &rc);
    CKR(rc);
    const int32_t* d_ix = ecr_upload(c, c->st_tg, n_indices, nnz, on_device, &rc);
    CKR(rc);
    const int32_t* d_v = ecr_upload(c, c->st_hp, n_data, nnz, on_device, &rc);
    CKR(rc);
    CKR(ensure(c, c->ecr_flag, ((size_t)z + 1) * 4));
    CKR(ensure(c, c->ecr_cols, std::max<size_t>(S, 1) * 4));
    CKR(ensure(c, c->smp_pairs, (size_t)(c->smp_n_pairs + z) * sizeof(uint2), true));
    CK(cudaMemsetAsync((u32*)c->ecr_flag.p + z, 0, 4, c->stream));
    CK(cudaMemsetAsync(c->d_ctr->ecr_bad, 0xFF, sizeof c->d_ctr->ecr_bad, c->stream));
    const int g = grid_for(z, ECR_THREADS, c->sm_count * 16);
    ecb_ecr_append_flags_kernel<<<g, ECR_THREADS, 0, c->stream>>>(d_ix, d_v, z, (u32)c->ecr_rows, (u32*)c->ecr_flag.p,
                                                                   c->d_ctr);
    LAUNCH_CHECK("ecr_append_flags");
    CKR(device_scan<false>(c, (const u32*)c->ecr_flag.p, (u32*)c->ecr_flag.p, (u64)z + 1, 0, nullptr));
    ecb_ecr_append_pairs_kernel<<<g, ECR_THREADS, 0, c->stream>>>(
        d_ip, S, d_ix, d_v, z, (u32)c->ecr_rows, (const u32*)c->ecr_flag.p, (const u32*)c->ecr_ec.p,
        (uint2*)c->smp_pairs.p + c->smp_n_pairs, (u32*)c->ecr_cols.p);
    LAUNCH_CHECK("ecr_append_pairs");
    if (S) CK(cudaMemcpyAsync(cols.data(), c->ecr_cols.p, (size_t)S * 4, cudaMemcpyDeviceToHost, c->stream));
    c->stats.d2h_bytes += (int64_t)S * 4;
    CK(cudaEventRecord(c->ev[1], c->stream));
    CKR(sync_counters(c));   // the call's one round trip: the column counts and the value checks
    const u32* bad = c->h_ctr->ecr_bad;
    if (bad[ECR_BAD_N_INDEX] != ECB_NONE)
      return fail(c, ECB_ERR_FORMAT, "N: EC index outside [0, %lld) at entry %u", (long long)c->ecr_rows,
                  bad[ECR_BAD_N_INDEX]);
    if (bad[ECR_BAD_N_COUNT] != ECB_NONE)
      return fail(c, ECB_ERR_FORMAT, "N: negative count at entry %u", bad[ECR_BAD_N_COUNT]);
    CK(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
  }
  u64 added = 0;
  for (u32 v : cols) added += v;
  // the ECs the rows claimed hold no reads: their count at this "close" is 0
  const u32 n = c->n_ec;
  if (n > c->smp_n_ec) {
    CKR(ensure(c, c->smp_last, (size_t)n * 4, true));
    CK(cudaMemsetAsync((u32*)c->smp_last.p + c->smp_n_ec, 0, (size_t)(n - c->smp_n_ec) * 4, c->stream));
  }
  c->smp_n_ec = n;
  c->smp_n_pairs += added;
  c->smp_counts.insert(c->smp_counts.end(), cols.begin(), cols.end());
  c->ecr_rows = -1;
  c->stats.samples += n_samples;
  c->stats.sample_pairs += (int64_t)added;
  c->stats.sample_ms += ms;
  if (nonzeros) *nonzeros = (int64_t)added;
  return ECB_OK;
}

int ecb_reset(ecb_ctx* c) {
  if (!c) return ECB_ERR_INVALID;
  CK(cudaSetDevice(c->device));
  if (c->table_slots) {
    CK(cudaMemsetAsync(c->table.p, 0xFF, (size_t)c->table_slots * sizeof(EcbEntry), c->stream));
    if (c->ttable_slots) CK(cudaMemsetAsync(c->ttable.p, 0xFF, (size_t)c->ttable_slots * sizeof(EcbEntry), c->stream));
    CK(cudaMemsetAsync(c->d_ctr, 0, sizeof(EcbCounters), c->stream));   // stream-ordered: no host sync needed
  }
  memset(c->h_ctr, 0, sizeof(EcbCounters));
  c->n_ec = 0;
  c->n_triples = 0;
  c->arena_used = 0;
  c->min_base = ~0ull;
  c->max_end = 0;
  c->n_alignments = 0;
  c->push_count = 0;
  c->smp_n_ec = 0;
  c->smp_n_pairs = 0;
  c->smp_counts.clear();
  c->smp_base = 0;
  c->smp_open = 0;
  c->ecr_rows = -1;
  c->ecr_used = c->ecr_broken = false;
  const int64_t slots = c->stats.table_slots;
  c->stats = ecb_stats{};
  c->stats.table_slots = slots;
  return ECB_OK;
}

int ecb_get_stats(const ecb_ctx* c, ecb_stats* out) {
  if (!c || !out) return ECB_ERR_INVALID;
  *out = c->stats;
  out->table_slots = c->table_slots;
  out->table_used = c->n_ec;
  out->row_entries = (int64_t)c->arena_used;
  return ECB_OK;
}

int ecb_rebase(ecb_ctx* c, int64_t delta) {
  if (!c) return ECB_ERR_INVALID;
  if (delta < 0) return fail(c, ECB_ERR_INVALID, "negative delta");
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "ecb_rebase covers the single-sample path only");
  CK(cudaSetDevice(c->device));
  if (delta == 0 || !c->table_slots || c->n_ec == 0) return ECB_OK;
  ecb_rebase_kernel<<<grid_for(c->n_ec, 256, c->sm_count * 8), 256, 0, c->stream>>>(
      (EcbEntry*)c->table.p, (const u32*)c->ec_slot.p, c->n_ec, (u64)delta);
  LAUNCH_CHECK("rebase");
  c->min_base += (u64)delta;
  c->max_end += (u64)delta;
  return ECB_OK;
}

// ---- the exchange over peer memory (see include/ecb200.h and ecb_exchange.cuh) ------------------------------

// An exchange arena: [header | cap_ec EC records | header | cap_pairs pair records], each header {records, unused,
// overflow}.  A single-sample arena (ecb_arena_create) has no pair part.  Its capacity counts 32-byte dispatch-1
// records, and the 24-byte records of dispatch 2 share that space; the per-cell capacities count the records of the
// dispatch at hand (the caller sizes them from exact counts).
struct ArenaLayout {
  char* base;
  int64_t cap_ec, cap_pairs;
  unsigned long long* ec_hdr() const { return (unsigned long long*)base; }
  unsigned long long* ec_rec() const { return (unsigned long long*)(base + ECB_ARENA_HEADER_BYTES); }
  unsigned long long* pair_hdr() const { return ec_rec() + (size_t)cap_ec * ECB_KEYREC_WORDS; }
  unsigned long long* pair_rec() const { return pair_hdr() + ECB_ARENA_HEADER_BYTES / 8; }
  size_t bytes() const {
    return ECB_ARENA_HEADER_BYTES + (size_t)cap_ec * ECB_KEYREC_WORDS * 8 +
           (cap_pairs ? ECB_ARENA_HEADER_BYTES + (size_t)cap_pairs * ECB_CPAIR1_WORDS * 8 : 0);
  }
  // 8-byte words of each record area, as the dispatch kernels' overflow test counts them (order: dispatch 2)
  u64 ec_words(bool order) const { return (u64)cap_ec * (order && cap_pairs ? ECB_ORDREC_WORDS : ECB_KEYREC_WORDS); }
  u64 pair_words(bool order) const { return (u64)cap_pairs * (order ? ECB_CPAIR2_WORDS : ECB_CPAIR1_WORDS); }
};

static ArenaLayout arena_of(const ecb_ctx* c) { return ArenaLayout{(char*)c->xa_base, c->xa_cap_ec, c->xa_cap_pairs}; }

// The arena of an owner context: plain cudaMalloc (exportable through CUDA IPC), headers cleared.
static int arena_alloc(ecb_ctx* c, int64_t cap_ec, int64_t cap_pairs, void* ipc_handle_out, void** base_out) {
  CK(cudaMalloc(&c->xa_base, ArenaLayout{nullptr, cap_ec, cap_pairs}.bytes()));
  c->xa_cap_ec = cap_ec;
  c->xa_cap_pairs = cap_pairs;
  const ArenaLayout L = arena_of(c);
  CK(cudaMemset(L.ec_hdr(), 0, ECB_ARENA_HEADER_BYTES));
  if (L.cap_pairs) CK(cudaMemset(L.pair_hdr(), 0, ECB_ARENA_HEADER_BYTES));
  if (ipc_handle_out) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handles are documented as 64 bytes");
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, c->xa_base));
    memcpy(ipc_handle_out, &h, sizeof h);
  }
  *base_out = c->xa_base;
  return ECB_OK;
}

// Both headers of this context's arena in one round trip: the records that arrived (n_pair = 0 without a pair
// part), ECB_ERR_LIMIT when the last dispatch (order: dispatch 2) found the arena too small.
static int arena_headers(ecb_ctx* c, bool order, u64* n_ec, u64* n_pair) {
  const ArenaLayout L = arena_of(c);
  unsigned long long h[6] = {0, 0, 0, 0, 0, 0};
  CK(cudaMemcpyAsync(h, L.ec_hdr(), 3 * 8, cudaMemcpyDeviceToHost, c->stream));
  if (L.cap_pairs) CK(cudaMemcpyAsync(h + 3, L.pair_hdr(), 3 * 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  *n_ec = h[0];
  *n_pair = h[3];
  const u64 rec_words = order ? ECB_ORDREC_WORDS : ECB_KEYREC_WORDS;
  if (!h[2] && !h[5] && h[0] * rec_words <= L.ec_words(order) && h[3] <= (u64)L.cap_pairs) return ECB_OK;
  if (L.cap_pairs)
    return fail(c, ECB_ERR_LIMIT, "exchange arena too small: %llu ECs and %llu pairs arrived, capacity %lld and %lld", h[0],
                h[3], (long long)L.cap_ec, (long long)L.cap_pairs);
  if (order) return fail(c, ECB_ERR_LIMIT, "exchange arena too small for the second dispatch");
  return fail(c, ECB_ERR_LIMIT, "exchange arena too small: %llu records arrived, capacity %lld", h[0], (long long)L.cap_ec);
}

// Every rank's arena as seen from this process, as targets of a dispatch (order: dispatch 2): the EC areas, and the
// pair areas of per-cell arenas (cap_pairs > 0) when P is given.
static int arena_targets(ecb_ctx* c, int world, void* const* bases, int64_t cap_ec, int64_t cap_pairs, bool order,
                         ArenaTargets* E, ArenaTargets* P = nullptr) {
  for (int r = 0; r < world; ++r) {
    if (!bases[r]) return fail(c, ECB_ERR_INVALID, "arena base of rank %d is NULL", r);
    const ArenaLayout L{(char*)bases[r], cap_ec, cap_pairs};
    E->hdr[r] = L.ec_hdr();
    E->rec[r] = L.ec_rec();
    if (P) {
      P->hdr[r] = L.pair_hdr();
      P->rec[r] = L.pair_rec();
    }
  }
  const ArenaLayout L{nullptr, cap_ec, cap_pairs};
  E->cap_words = L.ec_words(order);
  if (P) P->cap_words = L.pair_words(order);
  return ECB_OK;
}

// Shards with alignments, by position, and the rank that holds each (dispatch 2); they must not overlap (one
// read order over all ranks).
static int shard_routes(ecb_ctx* c, int world, const int64_t* shard_lo, const int64_t* shard_hi, u64* lo, u32* dest,
                        u32* n_shards) {
  std::vector<int> order;
  for (int r = 0; r < world; ++r)
    if (shard_hi[r] > shard_lo[r]) order.push_back(r);
  std::sort(order.begin(), order.end(), [&](int a, int b) { return shard_lo[a] < shard_lo[b]; });
  if (order.empty()) return fail(c, ECB_ERR_STATE, "no rank has pushed alignments");
  for (size_t k = 0; k < order.size(); ++k) {
    if (k && shard_lo[order[k]] < shard_hi[order[k - 1]])
      return fail(c, ECB_ERR_INVALID, "the ranks' order_base ranges overlap");
    if (shard_hi[order[k]] - shard_lo[order[k]] > 0xFFFFFFFEll)
      return fail(c, ECB_ERR_LIMIT, "a rank's alignments span more than 2^32 positions");
    lo[k] = (u64)shard_lo[order[k]];
    dest[k] = (u32)order[k];
  }
  *n_shards = (u32)order.size();
  return ECB_OK;
}

// The ECs of this context as a dispatch sends them: dispatch 1 (shard_lo NULL), or dispatch 2 with the routes of
// the shards (when there is an EC to route).
static int key_dispatch_params(ecb_ctx* c, int world, const int64_t* shard_lo, const int64_t* shard_hi,
                               KeyDispatchParams* K) {
  K->table = (const EcbEntry*)c->table.p;
  K->ec_slot = (const u32*)c->ec_slot.p;
  K->n_ec = c->table_slots ? c->n_ec : 0;
  K->world = (u32)world;
  if (shard_lo && K->n_ec) CKR(shard_routes(c, world, shard_lo, shard_hi, K->lo, K->dest, &K->n_shards));
  return ECB_OK;
}

// The EC records of a dispatch into the EC areas E (order: dispatch 2; kept_only: the per-cell dispatch 2, where
// ECs without reads in kept cells stay behind).
static int key_dispatch(ecb_ctx* c, const KeyDispatchParams& K, const ArenaTargets& E, bool order, bool kept_only,
                        const char* name) {
  const int g = grid_for(K.n_ec, 256, c->sm_count * 8);
  if (!order) ecb_key_dispatch_kernel<false><<<g, 256, 0, c->stream>>>(K, E);
  else if (!kept_only) ecb_key_dispatch_kernel<true><<<g, 256, 0, c->stream>>>(K, E);
  else ecb_key_dispatch_kernel<true, true><<<g, 256, 0, c->stream>>>(K, E);
  LAUNCH_CHECK(name);
  return ECB_OK;
}

// Owner merge of n_rec dispatch-1 EC records (ecb_import_arena, ecb_cells_import_arena).
static int import_keys(ecb_ctx* c, const unsigned long long* rec, u64 n_rec) {
  if (n_rec == 0) return ECB_OK;
  if (n_rec > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "too many records in one import");
  if (!c->table_slots) CKR(init_table(c));
  // the owner table must be able to take every incoming record as a new EC without filling up
  const u64 need = ((u64)c->n_ec + n_rec) * 2;
  if (need > c->table_slots) CKR(grow_table(c, pow2_ceil(need)));
  KeyImportParams P{};
  P.rec = rec;
  P.n_rec = (u32)n_rec;
  P.table = (EcbEntry*)c->table.p;
  P.mask = c->table_slots - 1;
  P.ec_slot = (u32*)c->ec_slot.p;
  P.ctr = c->d_ctr;
  ecb_import_keys_kernel<<<grid_for(n_rec, 256, c->sm_count * 8), 256, 0, c->stream>>>(P);
  LAUNCH_CHECK("import_keys");
  CKR(sync_counters(c));   // the one round trip of the merge: the number of merged ECs is known to the host again
  CKR(check_device_error(c));
  c->n_ec = c->h_ctr->n_ec;
  return ECB_OK;
}

// The flags of the second dispatch's slice build (ecb_order_mark_kernel, cells_pair_slice_kernel), after a
// sync_counters.
static int check_slice_flags(ecb_ctx* c) {
  const u32 bad = c->h_ctr->scratch[5];
  if (!bad) return ECB_OK;
  return fail(c, ECB_ERR_INVALID, "second dispatch: %s",
              (bad & 4u) ? "an EC arrived that the local context has never seen" : (bad & 2u) ? "two ECs share a first read"
              : (bad & 1u) ? "a record outside the shard's positions arrived" : (bad & 8u) ? "a pair arrived without its EC"
                           : "a pair's column is out of range");
}

// The A part of a slice (ecb_order_build, ecb_cells_order_build) from the n_rec dispatch-2 records at `rec`: an EC's
// id in the slice is the rank of its bit in a bitmap over the shard's `span` positions, its row comes from the
// LOCAL context.  Row lengths -> r_a_indptr, merged counts -> counts, rows -> r_a_indices / r_a_data, and *nnz.
// The lens pass skips every record the mark pass flags; the rows kernel, which indexes with what the lens pass
// wrote, runs only after one round trip has shown the flags clear and the non-zeros within int32.
static int build_a_slice(ecb_ctx* c, const ecb_ctx* local, const unsigned long long* rec, u64 n_rec, u64 span,
                         DevBuf& counts, u64* nnz) {
  const u32 local_n_ec = local->table_slots ? local->n_ec : 0;
  if (span > 0xFFFFFFFEull) return fail(c, ECB_ERR_LIMIT, "a rank's alignments span more than 2^32 positions");
  if (n_rec > span) return fail(c, ECB_ERR_INVALID, "%llu ECs arrived for a shard of %llu positions", n_rec, span);
  if (n_rec > local_n_ec) return fail(c, ECB_ERR_INVALID, "%llu ECs arrived but the local context holds %u", n_rec, local_n_ec);
  if (n_rec + 1 > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "slice exceeds the int32 fields of the EC file");
  const size_t words = (size_t)(span / 32) + 1;
  CKR(ensure(c, c->bitmap, words * 4));
  CKR(ensure(c, c->word_rank, words * 4));
  CKR(ensure(c, c->r_a_indptr, (n_rec + 1) * 4));
  CKR(ensure(c, counts, std::max<u64>(n_rec, 1) * 4));
  CKR(ensure(c, c->first_rel, std::max<u64>(n_rec, 1) * 8));   // scratch: local id per record, then per slice id
  // every row of the slice is a row of the local context: its arena fill bounds the non-zeros
  const u64 z_bound = std::max<u64>(local->arena_used, 1);
  CKR(ensure(c, c->r_a_indices, z_bound * 4));
  CKR(ensure(c, c->r_a_data, z_bound * 4));
  u32* lid_of_rec = (u32*)c->first_rel.p;
  u32* lid_of_id = lid_of_rec + n_rec;
  CK(cudaMemsetAsync(c->bitmap.p, 0, words * 4, c->stream));
  CK(cudaMemsetAsync(c->r_a_indptr.p, 0, (n_rec + 1) * 4, c->stream));
  CK(cudaMemsetAsync(&c->d_ctr->scratch[5], 0, sizeof(u32), c->stream));
  *nnz = 0;
  if (n_rec == 0) return ECB_OK;
  const int g = grid_for(n_rec, 256, c->sm_count * 8);
  ecb_order_mark_kernel<<<g, 256, 0, c->stream>>>(rec, (u32)n_rec, (u32)span, (const EcbEntry*)local->table.p,
                                                  local->table_slots - 1, (u32*)c->bitmap.p, lid_of_rec, &c->d_ctr->scratch[5]);
  LAUNCH_CHECK("order_mark");
  CKR(device_scan<true>(c, (const u32*)c->bitmap.p, (u32*)c->word_rank.p, words, 0, nullptr));
  ecb_order_lens_kernel<<<g, 256, 0, c->stream>>>(rec, (u32)n_rec, (u32)span, (const u32*)c->bitmap.p,
                                                  (const u32*)c->word_rank.p, lid_of_rec, (const u32*)local->row_len.p,
                                                  (int32_t*)c->r_a_indptr.p, (int32_t*)counts.p, lid_of_id);
  LAUNCH_CHECK("order_lens");
  CKR(device_scan<false>(c, (const u32*)c->r_a_indptr.p, (u32*)c->r_a_indptr.p, n_rec + 1, 0, nullptr));
  CK(cudaMemcpyAsync(c->h_total, scan_total(c, n_rec + 1), sizeof(u64), cudaMemcpyDeviceToHost, c->stream));
  c->stats.d2h_bytes += sizeof(u64);
  CKR(sync_counters(c));
  CKR(check_slice_flags(c));
  *nnz = *c->h_total;
  if (*nnz > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "slice exceeds the int32 fields of the EC file");
  ecb_order_rows_kernel<<<grid_for(n_rec, 256, c->sm_count * 16), 256, 0, c->stream>>>(
      lid_of_id, (const u32*)local->row_len.p, (const u32*)local->row_off.p, (const uint2*)local->arena.p,
      (const int32_t*)c->r_a_indptr.p, (u32)n_rec, (int32_t*)c->r_a_indices.p, (int32_t*)c->r_a_data.p);
  LAUNCH_CHECK("order_rows");
  return ECB_OK;
}

int ecb_arena_create(ecb_ctx* c, int64_t cap_records, void* ipc_handle_out, void** base_out) {
  if (!c || cap_records < 1 || !base_out) return ECB_ERR_INVALID;
  if (c->xa_base) return fail(c, ECB_ERR_STATE, "this context already has an arena");
  CK(cudaSetDevice(c->device));
  return arena_alloc(c, cap_records, 0, ipc_handle_out, base_out);
}

int ecb_arena_open_peer(ecb_ctx* c, const void* ipc_handle, void** base_out) {
  if (!c || !ipc_handle || !base_out) return ECB_ERR_INVALID;
  CK(cudaSetDevice(c->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle, sizeof h);
  void* p = nullptr;
  CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  c->xa_opened.push_back(p);
  *base_out = p;
  return ECB_OK;
}

int ecb_arena_reset(ecb_ctx* c) {
  if (!c || !c->xa_base) return ECB_ERR_INVALID;
  CK(cudaSetDevice(c->device));
  const ArenaLayout L = arena_of(c);
  CK(cudaMemsetAsync(L.ec_hdr(), 0, ECB_ARENA_HEADER_BYTES, c->stream));
  if (L.cap_pairs) CK(cudaMemsetAsync(L.pair_hdr(), 0, ECB_ARENA_HEADER_BYTES, c->stream));
  // on a caller-provided stream (ecb_set_stream) the call is stream-ordered - a collective on that stream is the
  // barrier in front of the peers' stores; a context on its own stream synchronises
  if (c->stream == c->own_stream) CK(cudaStreamSynchronize(c->stream));
  return ECB_OK;
}

int ecb_export_to_arenas(ecb_ctx* c, int world, void* const* arena_bases, int64_t cap_records, int64_t* min_base,
                         int64_t* max_end) {
  if (!c || !arena_bases || cap_records < 1) return ECB_ERR_INVALID;
  if (world < 1 || world > ECB_MAX_WORLD) return fail(c, ECB_ERR_INVALID, "world %d outside [1, %d]", world, ECB_MAX_WORLD);
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "the multi-GPU exchange covers the single-sample path only");
  if (c->ecr_used) return fail(c, ECB_ERR_STATE, "the multi-GPU exchange covers reads; this context holds EC rows");
  CK(cudaSetDevice(c->device));
  if (!c->table_slots) CKR(init_table(c));
  if (min_base) *min_base = c->n_ec ? (int64_t)c->min_base : 0;
  if (max_end) *max_end = c->n_ec ? (int64_t)c->max_end : 0;
  if (c->n_ec == 0) return ECB_OK;
  KeyDispatchParams K{};
  ArenaTargets E{};
  CKR(key_dispatch_params(c, world, nullptr, nullptr, &K));
  CKR(arena_targets(c, world, arena_bases, cap_records, 0, false, &E));
  CKR(key_dispatch(c, K, E, false, false, "export_to_arenas"));
  // remote stores are complete (and visible to the owner) when the kernel is.  On a caller-provided stream the
  // caller's next collective on that stream is the barrier between the stores and the owner's merge - no host
  // round trip here; a context on its own stream synchronises
  if (c->stream == c->own_stream) CK(cudaStreamSynchronize(c->stream));
  return ECB_OK;
}

int ecb_import_arena(ecb_ctx* c) {
  if (!c || !c->xa_base) return ECB_ERR_INVALID;
  CK(cudaSetDevice(c->device));
  u64 n_ec = 0, n_pair = 0;
  CKR(arena_headers(c, false, &n_ec, &n_pair));
  return import_keys(c, arena_of(c).ec_rec(), n_ec);
}

int ecb_order_dispatch(ecb_ctx* c, int world, void* const* arena_bases, int64_t cap_records, const int64_t* shard_lo,
                       const int64_t* shard_hi) {
  if (!c || !arena_bases || !shard_lo || !shard_hi || cap_records < 1) return ECB_ERR_INVALID;
  if (world < 1 || world > ECB_MAX_WORLD) return fail(c, ECB_ERR_INVALID, "world %d outside [1, %d]", world, ECB_MAX_WORLD);
  CK(cudaSetDevice(c->device));
  KeyDispatchParams K{};
  CKR(key_dispatch_params(c, world, shard_lo, shard_hi, &K));
  if (K.n_ec == 0) return ECB_OK;
  ArenaTargets E{};
  CKR(arena_targets(c, world, arena_bases, cap_records, 0, true, &E));
  CKR(key_dispatch(c, K, E, true, false, "order_dispatch"));
  if (c->stream == c->own_stream) CK(cudaStreamSynchronize(c->stream));   // (as ecb_export_to_arenas)
  return ECB_OK;
}

int ecb_order_build(ecb_ctx* c, const ecb_ctx* local, int64_t shard_lo, int64_t shard_hi, ecb_slice* out) {
  if (!c || !local || !out || !c->xa_base || shard_hi < shard_lo) return ECB_ERR_INVALID;
  if (local->device != c->device) return fail(c, ECB_ERR_INVALID, "the local context lives on another device");
  memset(out, 0, sizeof *out);
  CK(cudaSetDevice(c->device));
  u64 n_ec = 0, n_pair = 0, nnz = 0;
  CKR(arena_headers(c, true, &n_ec, &n_pair));
  CKR(build_a_slice(c, local, arena_of(c).ec_rec(), n_ec, (u64)(shard_hi - shard_lo), c->r_n_data, &nnz));
  CK(cudaStreamSynchronize(c->stream));
  out->id_base = 0;   // the caller knows where this rank's id range starts (the ECs of the shards in front)
  out->n_ec = (int64_t)n_ec;
  out->nnz = (int64_t)nnz;
  out->a_indptr = (const int32_t*)c->r_a_indptr.p;
  out->a_indices = (const int32_t*)c->r_a_indices.p;
  out->a_data = (const int32_t*)c->r_a_data.p;
  out->n_data = (const int32_t*)c->r_n_data.p;
  return ECB_OK;
}

// ---- the per-cell exchange (see include/ecb200.h and ecb_cells_exchange.cuh) ------------------------------

int ecb_cells_summary(ecb_ctx* c, const int32_t* cell_map, int64_t map_len, int64_t n_cells, uint64_t* cell_key,
                      uint64_t* cell_total) {
  if (!c || !cell_key || !cell_total || n_cells < 1 || n_cells > 0x7FFFFFFFll || (cell_map && map_len < 0))
    return ECB_ERR_INVALID;
  if (!c->with_cells) return fail(c, ECB_ERR_INVALID, "the per-cell exchange needs a context created with cells");
  CK(cudaSetDevice(c->device));
  CK(cudaMemsetAsync(cell_key, 0xFF, (size_t)n_cells * 8, c->stream));
  CK(cudaMemsetAsync(cell_total, 0, (size_t)n_cells * 8, c->stream));
  c->cx_n_local_cells = 0;
  if (!c->table_slots || c->n_triples == 0) return ECB_OK;   // a rank without reads takes part with an empty summary
  CellResult cr{};
  CKR(cells_local(c, &cr));
  const u32 n_local = (u32)cr.n_cells;
  if (cell_map && (int64_t)n_local > map_len)
    return fail(c, ECB_ERR_INVALID, "local cell id %u outside the cell map of %lld entries", n_local - 1, (long long)map_len);
  c->cx_n_local_cells = n_local;
  CK(cudaMemsetAsync(&c->d_ctr->scratch[5], 0, sizeof(u32), c->stream));
  cells_summary_kernel<<<grid_for(n_local, 256, c->sm_count * 8), 256, 0, c->stream>>>(
      (const u64*)c->cells.cell_key.p, (const u64*)c->cells.cell_total.p, n_local, cell_map, (u32)n_cells, (u64*)cell_key,
      (u64*)cell_total, &c->d_ctr->scratch[5]);
  LAUNCH_CHECK("cells_summary");
  CKR(sync_counters(c));
  if (c->h_ctr->scratch[5]) return fail(c, ECB_ERR_INVALID, "a cell id lies outside the %lld global cells", (long long)n_cells);
  return ECB_OK;
}

int ecb_cells_order(ecb_ctx* c, int world, const uint64_t* cell_keys, const uint64_t* cell_totals, int64_t n_cells,
                    int64_t min_cell_count, const int32_t* cell_map, int64_t* n_samples, const int32_t** cell_order) {
  if (!c || !cell_keys || !cell_totals || !n_samples || !cell_order || n_cells < 1 || n_cells > 0x7FFFFFFFll)
    return ECB_ERR_INVALID;
  if (world < 1 || world > ECB_MAX_WORLD) return fail(c, ECB_ERR_INVALID, "world %d outside [1, %d]", world, ECB_MAX_WORLD);
  if (!c->with_cells) return fail(c, ECB_ERR_INVALID, "the per-cell exchange needs a context created with cells");
  CK(cudaSetDevice(c->device));
  *n_samples = 0;
  *cell_order = nullptr;
  CellScratch& S = c->cells;
  const u32 C = (u32)n_cells;
  const u64 min_count = min_cell_count <= 0 ? 1ull : (u64)min_cell_count;  // bam_utils_multisample.py:596-597
  // sort by (first rank that holds the cell, its key there): on the key, then stably on the rank
  CKR(ensure(c, S.sort_k[0], (size_t)C * 8));
  CKR(ensure(c, S.sort_v[0], (size_t)C * 4));
  const int g_c = grid_for(C, 256, c->sm_count * 8);
  cells_first_key_kernel<<<g_c, 256, 0, c->stream>>>((const u64*)cell_keys, (u32)world, C, (u64*)S.sort_k[0].p, (u32*)S.sort_v[0].p);
  LAUNCH_CHECK("cells_first_key");
  int rb = 0;
  CKR(radix_sort(c, C, 64, &rb));
  cells_first_rank_kernel<<<g_c, 256, 0, c->stream>>>((const u64*)cell_keys, (u32)world, C, (const u32*)S.sort_v[rb].p,
                                                      (u64*)S.sort_k[0].p, (u32*)S.sort_v[0].p);
  LAUNCH_CHECK("cells_first_rank");
  CKR(radix_sort(c, C, 8, &rb));
  CKR(ensure(c, S.flags, (size_t)C * 4));
  CKR(ensure(c, S.offsets, (size_t)C * 4));
  cells_keep_flags_kernel<<<g_c, 256, 0, c->stream>>>((const u64*)S.sort_k[rb].p, (const u32*)S.sort_v[rb].p, C,
                                                      (const u64*)cell_totals, min_count, (u32*)S.flags.p);
  LAUNCH_CHECK("cells_keep_flags");
  u64 n_kept = 0;
  CKR(device_scan<false>(c, (const u32*)S.flags.p, (u32*)S.offsets.p, C, 0, &n_kept));
  if (n_kept == 0) return fail(c, ECB_ERR_EMPTY, "no cell reaches the minimum count %llu", (unsigned long long)min_count);
  CKR(ensure(c, c->cx_col_of_cell, (size_t)C * 4));
  CKR(ensure(c, c->r_cell_order, (size_t)C * 4));
  cells_assign_kernel<<<g_c, 256, 0, c->stream>>>((const u64*)S.sort_k[rb].p, (const u32*)S.sort_v[rb].p, C,
                                                  (const u64*)cell_totals, min_count, (const u32*)S.offsets.p,
                                                  (int32_t*)c->cx_col_of_cell.p, (int32_t*)c->r_cell_order.p);
  LAUNCH_CHECK("cells_assign");
  // this rank's side: the column of every local cell, and the reads of every local EC in kept cells
  CKR(ensure(c, c->cx_kept, (size_t)std::max<u32>(c->n_ec, 1) * 4));
  CK(cudaMemsetAsync(c->cx_kept.p, 0, (size_t)std::max<u32>(c->n_ec, 1) * 4, c->stream));
  if (c->cx_n_local_cells) {
    cells_local_columns_kernel<<<grid_for(c->cx_n_local_cells, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        cell_map, c->cx_n_local_cells, (const int32_t*)c->cx_col_of_cell.p, C, (int32_t*)S.cell_new.p);
    LAUNCH_CHECK("cells_local_columns");
    cells_kept_reads_kernel<<<grid_for(S.pair_slots, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        (const EcbEntry*)S.pair_table.p, S.pair_slots - 1, (const EcbEntry*)c->table.p, (const int32_t*)S.cell_new.p,
        (u32*)c->cx_kept.p);
    LAUNCH_CHECK("cells_kept_reads");
  }
  if (c->stream == c->own_stream) CK(cudaStreamSynchronize(c->stream));
  *n_samples = (int64_t)n_kept;
  *cell_order = (const int32_t*)c->r_cell_order.p;
  return ECB_OK;
}

int ecb_cells_dispatch_counts(ecb_ctx* c, int world, const int64_t* shard_lo, const int64_t* shard_hi, int64_t* counts) {
  if (!c || !counts || (!shard_lo) != (!shard_hi)) return ECB_ERR_INVALID;
  if (world < 1 || world > ECB_MAX_WORLD) return fail(c, ECB_ERR_INVALID, "world %d outside [1, %d]", world, ECB_MAX_WORLD);
  CK(cudaSetDevice(c->device));
  CK(cudaMemsetAsync(counts, 0, (size_t)world * 2 * 8, c->stream));
  KeyDispatchParams K{};
  CKR(key_dispatch_params(c, world, shard_lo, shard_hi, &K));
  CellPairDispatchParams P{};
  P.ec_table = K.table;
  P.ec_slot = K.ec_slot;
  P.world = (u32)world;
  if (shard_lo) {   // dispatch 2, an owner context
    if (K.n_ec == 0) return ECB_OK;
    memcpy(P.lo, K.lo, sizeof P.lo);
    memcpy(P.dest, K.dest, sizeof P.dest);
    P.n_shards = K.n_shards;
    P.pair_table = (const EcbEntry*)c->cells.pair_table.p;
    P.pair_slots = c->xa_cap_pairs ? c->cells.pair_slots : 0;
    cells_dispatch_count_kernel<true><<<c->sm_count * 4, 256, 0, c->stream>>>(K, P, (unsigned long long*)counts);
  } else {          // dispatch 1, a local context after ecb_cells_order
    if (K.n_ec && !c->cx_kept.p) return fail(c, ECB_ERR_STATE, "ecb_cells_order has not run on this context");
    P.pair_table = (const EcbEntry*)c->cells.pair_table.p;
    P.pair_slots = c->cx_n_local_cells ? c->cells.pair_slots : 0;
    P.cell_new = (const int32_t*)c->cells.cell_new.p;
    if (K.n_ec == 0 && P.pair_slots == 0) return ECB_OK;
    cells_dispatch_count_kernel<false><<<c->sm_count * 4, 256, 0, c->stream>>>(K, P, (unsigned long long*)counts);
  }
  LAUNCH_CHECK("cells_dispatch_count");
  if (c->stream == c->own_stream) CK(cudaStreamSynchronize(c->stream));   // counts are read on another stream
  return ECB_OK;
}

int ecb_cells_arena_create(ecb_ctx* c, int64_t cap_ec, int64_t cap_pairs, void* ipc_handle_out, void** base_out) {
  if (!c || cap_ec < 1 || cap_pairs < 1 || !base_out) return ECB_ERR_INVALID;
  CK(cudaSetDevice(c->device));
  // a smaller arena of an earlier call is replaced: nothing in flight may still use it or the peers' old ones
  CK(cudaStreamSynchronize(c->stream));
  for (void* p : c->xa_opened) CK(cudaIpcCloseMemHandle(p));
  c->xa_opened.clear();
  if (c->xa_base) CK(cudaFree(c->xa_base));
  c->xa_base = nullptr;
  c->xa_cap_ec = c->xa_cap_pairs = 0;
  return arena_alloc(c, cap_ec, cap_pairs, ipc_handle_out, base_out);
}

int ecb_cells_export_to_arenas(ecb_ctx* c, int world, void* const* arena_bases, int64_t cap_ec, int64_t cap_pairs,
                               int64_t* min_base, int64_t* max_end) {
  if (!c || !arena_bases || cap_ec < 1 || cap_pairs < 1) return ECB_ERR_INVALID;
  if (world < 1 || world > ECB_MAX_WORLD) return fail(c, ECB_ERR_INVALID, "world %d outside [1, %d]", world, ECB_MAX_WORLD);
  if (!c->with_cells) return fail(c, ECB_ERR_INVALID, "the per-cell exchange needs a context created with cells");
  CK(cudaSetDevice(c->device));
  const u32 n_ec = c->table_slots ? c->n_ec : 0;
  if (min_base) *min_base = n_ec ? (int64_t)c->min_base : 0;
  if (max_end) *max_end = n_ec ? (int64_t)c->max_end : 0;
  if (n_ec == 0) return ECB_OK;
  if (!c->cx_kept.p) return fail(c, ECB_ERR_STATE, "ecb_cells_order has not run on this context");
  ArenaTargets E{}, A{};
  CKR(arena_targets(c, world, arena_bases, cap_ec, cap_pairs, false, &E, &A));
  // EVERY local EC goes, with the reads it has in kept cells (0 too: this rank may hold its first occurrence)
  KeyDispatchParams K{};
  CKR(key_dispatch_params(c, world, nullptr, nullptr, &K));
  K.count_of = (const u32*)c->cx_kept.p;
  CKR(key_dispatch(c, K, E, false, false, "cells_export_ecs"));
  if (c->cx_n_local_cells) {
    CellPairDispatchParams P{};
    P.pair_table = (const EcbEntry*)c->cells.pair_table.p;
    P.pair_slots = c->cells.pair_slots;
    P.ec_table = K.table;
    P.cell_new = (const int32_t*)c->cells.cell_new.p;
    P.world = (u32)world;
    cells_pair_dispatch_kernel<false><<<grid_for(P.pair_slots, 256, c->sm_count * 8), 256, 0, c->stream>>>(P, A);
    LAUNCH_CHECK("cells_export_pairs");
  }
  if (c->stream == c->own_stream) CK(cudaStreamSynchronize(c->stream));   // (as ecb_export_to_arenas)
  return ECB_OK;
}

int ecb_cells_import_arena(ecb_ctx* c) {
  if (!c || !c->xa_base || !c->xa_cap_pairs) return ECB_ERR_INVALID;
  CK(cudaSetDevice(c->device));
  const ArenaLayout L = arena_of(c);
  u64 n_ec = 0, n_pair = 0;
  CKR(arena_headers(c, false, &n_ec, &n_pair));
  CKR(import_keys(c, L.ec_rec(), n_ec));
  if (n_pair > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "too many records in one import");
  if (n_pair && !c->table_slots) return fail(c, ECB_ERR_INVALID, "pairs arrived without their ECs");
  CellScratch& S = c->cells;
  S.pair_slots = std::max<u32>(1024u, pow2_ceil(n_pair * 2));
  CKR(ensure(c, S.pair_table, (size_t)S.pair_slots * sizeof(EcbEntry)));
  CK(cudaMemsetAsync(S.pair_table.p, 0xFF, (size_t)S.pair_slots * sizeof(EcbEntry), c->stream));
  if (n_pair) {
    cells_pair_import_kernel<<<grid_for(n_pair, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        L.pair_rec(), (u32)n_pair, (const EcbEntry*)c->table.p, c->table_slots - 1, (EcbEntry*)S.pair_table.p,
        S.pair_slots - 1, c->d_ctr);
    LAUNCH_CHECK("cells_import_pairs");
    CKR(sync_counters(c));
    CKR(check_device_error(c));
  }
  return ECB_OK;
}

int ecb_cells_order_dispatch(ecb_ctx* c, int world, void* const* arena_bases, int64_t cap_ec, int64_t cap_pairs,
                             const int64_t* shard_lo, const int64_t* shard_hi) {
  if (!c || !arena_bases || !shard_lo || !shard_hi || cap_ec < 1 || cap_pairs < 1 || !c->xa_cap_pairs) return ECB_ERR_INVALID;
  if (world < 1 || world > ECB_MAX_WORLD) return fail(c, ECB_ERR_INVALID, "world %d outside [1, %d]", world, ECB_MAX_WORLD);
  CK(cudaSetDevice(c->device));
  KeyDispatchParams K{};
  CKR(key_dispatch_params(c, world, shard_lo, shard_hi, &K));
  if (K.n_ec == 0) return ECB_OK;
  ArenaTargets E{}, A{};
  CKR(arena_targets(c, world, arena_bases, cap_ec, cap_pairs, true, &E, &A));
  CKR(key_dispatch(c, K, E, true, true, "cells_order_dispatch_ecs"));
  CellPairDispatchParams P{};
  P.pair_table = (const EcbEntry*)c->cells.pair_table.p;
  P.pair_slots = c->cells.pair_slots;
  P.ec_table = K.table;
  P.ec_slot = K.ec_slot;
  P.world = (u32)world;
  memcpy(P.lo, K.lo, sizeof P.lo);
  memcpy(P.dest, K.dest, sizeof P.dest);
  P.n_shards = K.n_shards;
  cells_pair_dispatch_kernel<true><<<grid_for(P.pair_slots, 256, c->sm_count * 8), 256, 0, c->stream>>>(P, A);
  LAUNCH_CHECK("cells_order_dispatch_pairs");
  if (c->stream == c->own_stream) CK(cudaStreamSynchronize(c->stream));
  return ECB_OK;
}

int ecb_cells_order_build(ecb_ctx* c, const ecb_ctx* local, int64_t shard_lo, int64_t shard_hi, int64_t n_samples,
                          ecb_cells_slice* out) {
  if (!c || !local || !out || !c->xa_base || !c->xa_cap_pairs || shard_hi < shard_lo || n_samples < 1 ||
      n_samples > 0x7FFFFFFFll)
    return ECB_ERR_INVALID;
  if (local->device != c->device) return fail(c, ECB_ERR_INVALID, "the local context lives on another device");
  memset(out, 0, sizeof *out);
  CK(cudaSetDevice(c->device));
  const ArenaLayout L = arena_of(c);
  u64 n_ec = 0, n_pair = 0, nnz = 0;
  CKR(arena_headers(c, true, &n_ec, &n_pair));
  if (n_pair > 0x7FFFFFFFull) return fail(c, ECB_ERR_LIMIT, "slice exceeds the int32 fields of the EC file");
  const u64 span = (u64)(shard_hi - shard_lo);
  CKR(ensure(c, c->cx_col_counts, (size_t)n_samples * 4));
  CK(cudaMemsetAsync(c->cx_col_counts.p, 0, (size_t)n_samples * 4, c->stream));
  CKR(build_a_slice(c, local, L.ec_rec(), n_ec, span, c->count_of, &nnz));   // merged counts: not part of the slice
  CKR(ensure(c, c->r_n_indices, std::max<u64>(n_pair, 1) * 4));
  CKR(ensure(c, c->r_n_data, std::max<u64>(n_pair, 1) * 4));
  if (n_pair) {
    CellScratch& S = c->cells;
    CKR(ensure(c, S.sort_k[0], (size_t)n_pair * 8));
    CKR(ensure(c, S.sort_v[0], (size_t)n_pair * 4));
    cells_pair_slice_kernel<<<grid_for(n_pair, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        L.pair_rec(), (u32)n_pair, (u32)span, (u32)n_samples, (const u32*)c->bitmap.p, (const u32*)c->word_rank.p,
        (u64*)S.sort_k[0].p, (u32*)S.sort_v[0].p, &c->d_ctr->scratch[5]);
    LAUNCH_CHECK("cells_pair_slice");
    CKR(sync_counters(c));   // the sort and the column counts below index with what the pair pass produced
    CKR(check_slice_flags(c));
    int rb = 0;
    CKR(radix_sort(c, (u32)n_pair, 32 + bits_for((u64)n_samples), &rb));
    cells_slice_csc_kernel<<<grid_for(n_pair, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        (const u64*)S.sort_k[rb].p, (const u32*)S.sort_v[rb].p, (u32)n_pair, (int32_t*)c->cx_col_counts.p,
        (int32_t*)c->r_n_indices.p, (int32_t*)c->r_n_data.p);
    LAUNCH_CHECK("cells_slice_csc");
  }
  CKR(sync_counters(c));
  CKR(check_device_error(c));
  out->n_ec = (int64_t)n_ec;
  out->nnz = (int64_t)nnz;
  out->a_indptr = (const int32_t*)c->r_a_indptr.p;
  out->a_indices = (const int32_t*)c->r_a_indices.p;
  out->a_data = (const int32_t*)c->r_a_data.p;
  out->n_samples = n_samples;
  out->nnz_n = (int64_t)n_pair;
  out->n_col_counts = (const int32_t*)c->cx_col_counts.p;
  out->n_indices = (const int32_t*)c->r_n_indices.p;
  out->n_data = (const int32_t*)c->r_n_data.p;
  return ECB_OK;
}

int ecb_destroy(ecb_ctx* c) {
  if (!c) return ECB_OK;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  DevBuf* bufs[] = {&c->table, &c->ec_slot, &c->ec_rep, &c->ec_len, &c->spill, &c->row_len, &c->row_off, &c->arena, &c->long_list, &c->mid_list, &c->big_list, &c->count_of,
                    &c->ttable, &c->st_rg, &c->st_tg, &c->st_hp, &c->st_cell, &c->st2_rg, &c->st2_tg, &c->st2_hp, &c->st2_cell,
                    &c->overflow_bits, &c->lr_list, &c->lr_meta, &c->lr_rank, &c->lr_acc,
                    &c->scan_buf, &c->bitmap, &c->word_rank, &c->first_rel, &c->ecid_of, &c->prov_of, &c->ec_keep,
                    &c->r_a_indptr, &c->r_a_indices, &c->r_a_data, &c->r_n_indptr, &c->r_n_indices,
                    &c->r_n_data, &c->r_cell_order, &c->cx_kept, &c->cx_col_of_cell, &c->cx_col_counts,
                    &c->smp_last, &c->smp_pairs, &c->ecr_acc, &c->ecr_slot, &c->ecr_ec, &c->ecr_dst, &c->ecr_flag,
                    &c->ecr_cols, &c->ecr_seen};
  for (DevBuf* b : bufs) release(c, *b);
  cells_release(c);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->copy_stream) {
    cudaStreamSynchronize(c->copy_stream);
    cudaStreamDestroy(c->copy_stream);
    cudaEventDestroy(c->copy_done[0]);
    cudaEventDestroy(c->copy_done[1]);
  }
  for (void* p : c->xa_opened) cudaIpcCloseMemHandle(p);
  if (c->xa_base) cudaFree(c->xa_base);
  if (c->d_ctr) cudaFree(c->d_ctr);
  if (c->h_ctr) cudaFreeHost(c->h_ctr);
  if (c->h_total) cudaFreeHost(c->h_total);
  if (c->h_res) {
    if (c->pageable_results) free(c->h_res); else cudaFreeHost(c->h_res);
  }
  for (auto& e : c->ev)
    if (e) cudaEventDestroy(e);
  if (c->own_stream) {
    cudaStreamSynchronize(c->own_stream);
    cudaStreamDestroy(c->own_stream);
  }
  if (c->pool) cudaMemPoolDestroy(c->pool);
  delete c;
  return ECB_OK;
}

}  // extern "C"

// ---- device decode of single-sample BAM files (kernels in ecb_bam.cuh) ----------------------------------------
struct ecb_bam {
  ecb_ctx* c = nullptr;
  int32_t n_ref = 0;
  bool track = false;
  DevBuf tid_target, tid_hap, range_min, range_max;
  DevBuf comp, blocks;
  DevBuf win[2];                  // inflated window; the bytes left after its last whole record move to the other one
  int cur = 0;
  u64 carry = 0;                  // bytes at the front of win[cur]: the start of a record that continues
  DevBuf seg_start, seg_cnt, seg_state, seg_land[2];
  DevBuf off, valid, rowpos, vrec, starts, starts_x;
  DevBuf rows[2][3];              // read_group, target_idx, hap_idx; the open read moves to the other set
  int rcur = 0;
  u64 n_rows = 0, open_row = 0;   // rows held in rows[rcur]; first row of the read that is still open
  int64_t all_alignments = 0, group = -1;
  bool failed = false, finished = false;
  BamDevState* d_st = nullptr;
  BamDevState* h_st = nullptr;    // pinned mirror
  std::vector<BamBlock> h_blocks;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  ecb_bam_stats stats{};
};

namespace {

#define ECB_BAM_AUTO_WINDOW (1ll << 30)

int bam_sync_state(ecb_bam* d) {
  ecb_ctx* c = d->c;
  CK(cudaMemcpyAsync(d->h_st, d->d_st, sizeof(BamDevState), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return ECB_OK;
}

double bam_ms(cudaEvent_t a, cudaEvent_t b) {
  float ms = 0;
  cudaEventElapsedTime(&ms, a, b);
  return ms;
}

void bam_release(ecb_bam* d) {
  ecb_ctx* c = d->c;
  DevBuf* bufs[] = {&d->tid_target, &d->tid_hap, &d->range_min, &d->range_max, &d->comp, &d->blocks, &d->win[0], &d->win[1],
                    &d->seg_start, &d->seg_cnt, &d->seg_state, &d->seg_land[0], &d->seg_land[1], &d->off, &d->valid,
                    &d->rowpos, &d->vrec, &d->starts, &d->starts_x};
  for (DevBuf* b : bufs) release(c, *b);
  for (auto& set : d->rows)
    for (DevBuf& b : set) release(c, b);
  cudaStreamSynchronize(c->stream);
  if (d->d_st) cudaFree(d->d_st);
  if (d->h_st) cudaFreeHost(d->h_st);
  for (auto& e : d->ev)
    if (e) cudaEventDestroy(e);
  delete d;
}

// The records of win[cur][p0, carry + wbytes) after blocks [b0, b1) of the call were inflated behind the carry.
int bam_window(ecb_bam* d, long long b0, long long b1, u64 wbytes, u32 p0) {
  ecb_ctx* c = d->c;
  const u64 wend64 = d->carry + wbytes;
  if (wend64 >= (u64)ECB_BAM_NONE) return fail(c, ECB_ERR_LIMIT, "a BAM window of %llu inflated bytes (a record longer than 4 GiB?)", wend64);
  const u32 wend = (u32)wend64;
  CKR(ensure(c, d->win[d->cur], wend64 + 16, true));   // keeps the carried bytes
  uint8_t* win = (uint8_t*)d->win[d->cur].p;
  CK(cudaEventRecord(d->ev[2], c->stream));
  if (b1 > b0) {
    ecb_bam_inflate_kernel<<<(unsigned)((b1 - b0 + ECB_BAM_INFLATE_THREADS - 1) / ECB_BAM_INFLATE_THREADS), ECB_BAM_INFLATE_THREADS,
                             0, c->stream>>>((const uint8_t*)d->comp.p, (const BamBlock*)d->blocks.p, b0, b1, win + d->carry, d->d_st);
    LAUNCH_CHECK("bam_inflate");
  }
  CK(cudaEventRecord(d->ev[3], c->stream));
  // a rejected block leaves its output range partly unwritten: report it before anything hops over that range
  CKR(bam_sync_state(d));
  if (d->h_st->error & BAM_ERR_INFLATE)
    return fail(c, ECB_ERR_FORMAT, "corrupt BGZF block (inflate failed): block %lld of this call", d->h_st->bad_block);

  // record hop: guesses, join rounds, offsets
  const u32 n_seg = wend > p0 ? (wend - p0 + ECB_BAM_SEG - 1) / ECB_BAM_SEG : 1u;
  CKR(ensure(c, d->seg_start, (size_t)n_seg * 4));
  CKR(ensure(c, d->seg_cnt, (size_t)n_seg * 4));
  CKR(ensure(c, d->seg_state, (size_t)n_seg * 4));
  CKR(ensure(c, d->seg_land[0], (size_t)n_seg * 4));
  CKR(ensure(c, d->seg_land[1], (size_t)n_seg * 4));
  BamHop H{win, p0, wend, n_seg, d->n_ref, (u32*)d->seg_start.p, (u32*)d->seg_cnt.p, (u32*)d->seg_state.p};
  u32* land[2] = {(u32*)d->seg_land[0].p, (u32*)d->seg_land[1].p};
  const int grid = (int)((n_seg + 127) / 128);
  ecb_bam_guess_kernel<<<grid, 128, 0, c->stream>>>(H, land[0]);
  LAUNCH_CHECK("bam_guess");
  int a = 0;
  for (;;) {
    CK(cudaMemsetAsync(&d->d_st->changed, 0, sizeof(u32), c->stream));
    ecb_bam_round_kernel<<<grid, 128, 0, c->stream>>>(H, land[a], land[1 - a], &d->d_st->changed);
    LAUNCH_CHECK("bam_round");
    a = 1 - a;
    d->stats.hop_rounds++;
    CKR(bam_sync_state(d));
    if (d->h_st->changed == 0) break;
  }
  u64 n_rec64 = 0;
  CKR(device_scan<false>(c, H.cnt, H.cnt, n_seg, 0, &n_rec64));
  const u32 n_rec = (u32)n_rec64;
  CKR(ensure(c, d->off, (size_t)n_rec * 4 + 4));
  ecb_bam_offsets_kernel<<<grid, 128, 0, c->stream>>>(H, H.cnt, land[a], (u32*)d->off.p, d->d_st);
  LAUNCH_CHECK("bam_offsets");
  CK(cudaEventRecord(d->ev[4], c->stream));
  CKR(bam_sync_state(d));
  if (d->h_st->hop_state == BAM_HOP_BAD) return fail(c, ECB_ERR_FORMAT, "BAM record with block_size %u", d->h_st->hop_bs);
  const u32 land_at = d->h_st->hop_land;

  // rules and rows
  if (n_rec) {
    BamRules R{win, (const u32*)d->off.p, n_rec, d->n_ref, (const int32_t*)d->tid_target.p, (const int32_t*)d->tid_hap.p,
               d->track ? (int32_t*)d->range_min.p : nullptr, d->track ? (int32_t*)d->range_max.p : nullptr, d->d_st};
    CKR(ensure(c, d->valid, (size_t)n_rec * 4));
    CKR(ensure(c, d->rowpos, (size_t)n_rec * 4));
    const int rgrid = (int)((n_rec + 255) / 256);
    ecb_bam_validity_kernel<<<rgrid, 256, 0, c->stream>>>(R, (u32*)d->valid.p);
    LAUNCH_CHECK("bam_validity");
    u64 n_valid64 = 0;
    CKR(device_scan<false>(c, (const u32*)d->valid.p, (u32*)d->rowpos.p, n_rec, 0, &n_valid64));
    CKR(bam_sync_state(d));
    if (d->h_st->error & BAM_ERR_NAME) return fail(c, ECB_ERR_FORMAT, "BAM record with a bad read-name length");
    if (d->h_st->error & BAM_ERR_TID)
      return fail(c, ECB_ERR_FORMAT, "alignment with reference id %d outside the header's %d references", d->h_st->bad_tid, d->n_ref);
    const u32 n_valid = (u32)n_valid64;
    if (n_valid) {
      CKR(ensure(c, d->vrec, (size_t)n_valid * 4));
      CKR(ensure(c, d->starts, (size_t)n_valid * 4));
      CKR(ensure(c, d->starts_x, (size_t)n_valid * 4));
      for (DevBuf& b : d->rows[d->rcur]) CKR(ensure(c, b, (size_t)(d->n_rows + n_valid) * 4, true));
      ecb_bam_compact_kernel<<<rgrid, 256, 0, c->stream>>>(R, (const u32*)d->valid.p, (const u32*)d->rowpos.p, (u32*)d->vrec.p);
      LAUNCH_CHECK("bam_compact");
      const int vgrid = (int)((n_valid + 255) / 256);
      const BamRecordAt A{win, (const u32*)d->vrec.p};
      ecb_read_starts_kernel<<<vgrid, 256, 0, c->stream>>>(A, n_valid, &d->d_st->carry, (u32*)d->starts.p);
      LAUNCH_CHECK("bam_starts");
      u64 n_starts = 0;
      CKR(device_scan<false>(c, (const u32*)d->starts.p, (u32*)d->starts_x.p, n_valid, 0, &n_starts));
      ecb_read_rows_kernel<<<vgrid, 256, 0, c->stream>>>(A, n_valid, (const u32*)d->starts.p, (const u32*)d->starts_x.p,
                                                          d->group, d->n_rows, R.tid_target, R.tid_hap, &d->d_st->carry,
                                                          (int32_t*)d->rows[d->rcur][0].p, (int32_t*)d->rows[d->rcur][1].p,
                                                          (int32_t*)d->rows[d->rcur][2].p);
      LAUNCH_CHECK("bam_rows");
      d->n_rows += n_valid;
      d->group += (int64_t)n_starts;
    }
    d->all_alignments += n_rec;
    d->stats.records += n_rec;
  }
  CK(cudaEventRecord(d->ev[5], c->stream));

  // what follows the last whole record starts the next window
  const u64 keep = wend - land_at;
  if (keep) {
    CKR(ensure(c, d->win[1 - d->cur], keep + 16));
    CK(cudaMemcpyAsync(d->win[1 - d->cur].p, win + land_at, keep, cudaMemcpyDeviceToDevice, c->stream));
    d->cur = 1 - d->cur;
  }
  d->carry = keep;
  CK(cudaEventSynchronize(d->ev[5]));
  d->stats.inflate_ms += bam_ms(d->ev[2], d->ev[3]);
  d->stats.hop_ms += bam_ms(d->ev[3], d->ev[4]);
  d->stats.rules_ms += bam_ms(d->ev[4], d->ev[5]);
  d->stats.windows++;
  return ECB_OK;
}

int bam_decode(ecb_bam* d, const uint8_t* bytes, int64_t n_bytes, const int64_t* block_off, const int32_t* block_len,
               const int32_t* block_isize, int64_t n_blocks, int64_t skip, int last, const int32_t** read_group,
               const int32_t** target_idx, const int32_t** hap_idx, int64_t* rows) {
  ecb_ctx* c = d->c;
  if (n_bytes < 0 || n_blocks < 0 || skip < 0) return fail(c, ECB_ERR_INVALID, "negative size");
  if ((n_blocks > 0 && (!block_off || !block_len || !block_isize)) || (n_bytes > 0 && !bytes))
    return fail(c, ECB_ERR_INVALID, "NULL block table or bytes");
  if (skip > 0 && d->carry) return fail(c, ECB_ERR_INVALID, "skip is only meaningful before the first record");
  // the block table comes from outside the library: every block must lie inside `bytes`
  d->h_blocks.resize((size_t)n_blocks);
  int64_t total = 0;
  for (int64_t i = 0; i < n_blocks; ++i) {
    if (block_off[i] < 0 || block_len[i] < 0 || block_off[i] > n_bytes || block_len[i] > n_bytes - block_off[i])
      return fail(c, ECB_ERR_INVALID, "block %lld lies outside the %lld bytes given", (long long)i, (long long)n_bytes);
    if (block_isize[i] < 0 || block_isize[i] > 65536)
      return fail(c, ECB_ERR_FORMAT, "BGZF block %lld of this call claims %u inflated bytes; the device decoder takes at most 65536",
                  (long long)i, (unsigned)block_isize[i]);
    d->h_blocks[(size_t)i] = BamBlock{(u64)block_off[i], (u32)block_len[i], (u32)block_isize[i], 0};
    total += block_isize[i];
  }
  if (skip > total) return fail(c, ECB_ERR_INVALID, "skip %lld beyond the %lld inflated bytes of the call", (long long)skip, (long long)total);
  CK(cudaSetDevice(c->device));

  // rows of the read the previous call left open go to the front
  if (d->open_row > 0) {
    const u64 keep = d->n_rows - d->open_row;
    const int other = 1 - d->rcur;
    for (int j = 0; j < 3; ++j) {
      CKR(ensure(c, d->rows[other][j], (size_t)keep * 4 + 4));
      if (keep)
        CK(cudaMemcpyAsync(d->rows[other][j].p, (const int32_t*)d->rows[d->rcur][j].p + d->open_row, (size_t)keep * 4,
                           cudaMemcpyDeviceToDevice, c->stream));
    }
    d->rcur = other;
    d->n_rows = keep;
    d->open_row = 0;
    CK(cudaMemsetAsync(&d->d_st->carry.open_row, 0, sizeof(unsigned long long), c->stream));
  }

  // windows of whole blocks, at most ECB_OPT_BAM_WINDOW inflated bytes each (at least one block)
  const int64_t wmax = c->opt_bam_window > 0 ? c->opt_bam_window : ECB_BAM_AUTO_WINDOW;
  std::vector<int64_t> cut{0};
  std::vector<u64> wbytes;
  {
    u64 acc = 0;
    for (int64_t i = 0; i < n_blocks; ++i) {
      const u64 sz = d->h_blocks[(size_t)i].isize;
      if (i > cut.back() && acc + sz > (u64)wmax) {
        cut.push_back(i);
        wbytes.push_back(acc);
        acc = 0;
      }
      d->h_blocks[(size_t)i].dst_off = acc;
      acc += sz;
    }
    if (n_blocks > 0) {
      cut.push_back(n_blocks);
      wbytes.push_back(acc);
    }
  }
  if (!wbytes.empty() && (u64)skip > wbytes[0]) return fail(c, ECB_ERR_INVALID, "skip %lld beyond the first window", (long long)skip);

  CK(cudaEventRecord(d->ev[0], c->stream));
  if (n_blocks > 0) {
    CKR(ensure(c, d->comp, (size_t)n_bytes + 16));
    CKR(ensure(c, d->blocks, (size_t)n_blocks * sizeof(BamBlock)));
    CK(cudaMemcpyAsync(d->comp.p, bytes, (size_t)n_bytes, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(d->blocks.p, d->h_blocks.data(), (size_t)n_blocks * sizeof(BamBlock), cudaMemcpyHostToDevice, c->stream));
    d->stats.h2d_bytes += n_bytes;
    d->stats.blocks += n_blocks;
    d->stats.inflated_bytes += total;
  }
  CK(cudaEventRecord(d->ev[1], c->stream));
  for (size_t w = 0; w < wbytes.size(); ++w)
    CKR(bam_window(d, cut[w], cut[w + 1], wbytes[w], w == 0 ? (u32)skip : 0u));
  CKR(bam_sync_state(d));
  d->stats.h2d_ms += bam_ms(d->ev[0], d->ev[1]);
  if (last) {
    if (d->carry) return fail(c, ECB_ERR_FORMAT, "truncated BAM record at the end of the file");
    d->finished = true;
    d->open_row = d->n_rows;   // the end of the file closes the last read
  } else {
    d->open_row = d->h_st->carry.open_row;
  }
  *read_group = (const int32_t*)d->rows[d->rcur][0].p;
  *target_idx = (const int32_t*)d->rows[d->rcur][1].p;
  *hap_idx = (const int32_t*)d->rows[d->rcur][2].p;
  *rows = (int64_t)d->open_row;
  return ECB_OK;
}

}  // namespace

extern "C" {

int ecb_bam_create(ecb_ctx* c, const int32_t* tid_target, const int32_t* tid_hap, int32_t n_references, int track_ranges,
                   ecb_bam** out) {
  if (!c || !out) return ECB_ERR_INVALID;
  *out = nullptr;
  if (n_references < 0 || (n_references > 0 && (!tid_target || !tid_hap))) return fail(c, ECB_ERR_INVALID, "bad reference tables");
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "the device BAM decoder covers the single-sample path only");
  CK(cudaSetDevice(c->device));
  ecb_bam* d = new ecb_bam();
  d->c = c;
  d->n_ref = n_references;
  d->track = track_ranges != 0;
  auto bail = [&](int code) {
    bam_release(d);
    return code;
  };
  const size_t tb = (size_t)n_references * 4 + 4;
  int rc = ECB_OK;
  for (DevBuf* b : {&d->tid_target, &d->tid_hap, &d->range_min, &d->range_max})
    if (rc == ECB_OK) rc = ensure(c, *b, tb);
  if (rc != ECB_OK) return bail(rc);
  std::vector<int32_t> lo((size_t)n_references + 1, INT32_MAX);
  if (cudaMalloc(&d->d_st, sizeof(BamDevState)) != cudaSuccess || cudaMallocHost(&d->h_st, sizeof(BamDevState)) != cudaSuccess)
    return bail(fail(c, ECB_ERR_CUDA, "decoder state allocation failed"));
  for (auto& e : d->ev)
    if (cudaEventCreate(&e) != cudaSuccess) return bail(fail(c, ECB_ERR_CUDA, "cudaEventCreate failed"));
  memset(d->h_st, 0, sizeof(BamDevState));
  d->h_st->bad_block = 0x7FFFFFFFFFFFFFFFll;
  const cudaMemcpyKind h2d = cudaMemcpyHostToDevice;
  if (n_references > 0 &&
      (cudaMemcpyAsync(d->tid_target.p, tid_target, (size_t)n_references * 4, h2d, c->stream) != cudaSuccess ||
       cudaMemcpyAsync(d->tid_hap.p, tid_hap, (size_t)n_references * 4, h2d, c->stream) != cudaSuccess))
    return bail(fail(c, ECB_ERR_CUDA, "table copy failed"));
  if (cudaMemcpyAsync(d->range_min.p, lo.data(), tb, h2d, c->stream) != cudaSuccess ||
      cudaMemsetAsync(d->range_max.p, 0xFF, tb, c->stream) != cudaSuccess ||
      cudaMemcpyAsync(d->d_st, d->h_st, sizeof(BamDevState), h2d, c->stream) != cudaSuccess ||
      cudaStreamSynchronize(c->stream) != cudaSuccess)
    return bail(fail(c, ECB_ERR_CUDA, "decoder initialisation failed"));
  *out = d;
  return ECB_OK;
}

int ecb_bam_decode(ecb_bam* d, const uint8_t* bytes, int64_t n_bytes, const int64_t* block_off, const int32_t* block_len,
                   const int32_t* block_isize, int64_t n_blocks, int64_t skip, int last, const int32_t** read_group,
                   const int32_t** target_idx, const int32_t** hap_idx, int64_t* rows) {
  if (!d || !read_group || !target_idx || !hap_idx || !rows) return ECB_ERR_INVALID;
  if (d->failed) return fail(d->c, ECB_ERR_STATE, "this decoder failed earlier; create a new one");
  if (d->finished) return fail(d->c, ECB_ERR_STATE, "this decoder has had its last call");
  const int rc = bam_decode(d, bytes, n_bytes, block_off, block_len, block_isize, n_blocks, skip, last, read_group,
                            target_idx, hap_idx, rows);
  if (rc != ECB_OK) d->failed = true;
  return rc;
}

int ecb_bam_counters(const ecb_bam* d, int64_t* all_alignments, int64_t* n_groups) {
  if (!d || !all_alignments || !n_groups) return ECB_ERR_INVALID;
  *all_alignments = d->all_alignments;
  *n_groups = d->group + 1;
  return ECB_OK;
}

int ecb_bam_ranges(ecb_bam* d, int32_t* range_min, int32_t* range_max) {
  if (!d || (d->n_ref > 0 && (!range_min || !range_max))) return ECB_ERR_INVALID;
  ecb_ctx* c = d->c;
  if (!d->track) return fail(c, ECB_ERR_STATE, "ranges were not tracked");
  if (d->n_ref == 0) return ECB_OK;
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(range_min, d->range_min.p, (size_t)d->n_ref * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(range_max, d->range_max.p, (size_t)d->n_ref * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return ECB_OK;
}

int ecb_bam_get_stats(const ecb_bam* d, ecb_bam_stats* out) {
  if (!d || !out) return ECB_ERR_INVALID;
  *out = d->stats;
  return ECB_OK;
}

int ecb_bam_destroy(ecb_bam* d) {
  if (!d) return ECB_OK;
  cudaSetDevice(d->c->device);
  bam_release(d);
  return ECB_OK;
}

}  // extern "C"

// ---- device parse of single-sample SAM text (kernels in ecb_sam.cuh) --------------------------------------------
struct ecb_sam {
  ecb_ctx* c = nullptr;
  int32_t n_ref = 0;
  bool track = false;
  int64_t next_line = 1;          // line number of the next call's first byte
  DevBuf tid_target, tid_hap, range_min, range_max;
  DevBuf slots, blob, name_off;   // the @SQ name table
  u32 mask = 0;
  DevBuf text, seg_nl, seg_tab, line_end, tabs_end, lines, valid, rowpos, vline, starts, starts_x;
  DevBuf rows[2][3];              // read_group, target_idx, hap_idx; the open read moves to the other set
  int rcur = 0;
  u64 n_rows = 0, open_row = 0;
  int64_t all_alignments = 0, group = -1;
  bool failed = false, finished = false;
  SamDevState* d_st = nullptr;
  SamDevState* h_st = nullptr;    // pinned mirror
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  ecb_sam_stats stats{};
};

namespace {

int sam_sync_state(ecb_sam* d) {
  ecb_ctx* c = d->c;
  CK(cudaMemcpyAsync(d->h_st, d->d_st, sizeof(SamDevState), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return ECB_OK;
}

void sam_release(ecb_sam* d) {
  ecb_ctx* c = d->c;
  DevBuf* bufs[] = {&d->tid_target, &d->tid_hap, &d->range_min, &d->range_max, &d->slots, &d->blob, &d->name_off,
                    &d->text, &d->seg_nl, &d->seg_tab, &d->line_end, &d->tabs_end, &d->lines, &d->valid, &d->rowpos,
                    &d->vline, &d->starts, &d->starts_x};
  for (DevBuf* b : bufs) release(c, *b);
  for (auto& set : d->rows)
    for (DevBuf& b : set) release(c, b);
  cudaStreamSynchronize(c->stream);
  if (d->d_st) cudaFree(d->d_st);
  if (d->h_st) cudaFreeHost(d->h_st);
  for (auto& e : d->ev)
    if (e) cudaEventDestroy(e);
  delete d;
}

// The messages of the SAM_BAD_* kinds; alntools_b200/sam_utils.py raises the same ones.
int sam_bad_line(ecb_sam* d, int64_t line, u32 kind) {
  static const char* what[] = {"", "a header line (starting with '@') after the first alignment line",
                               "fewer than 11 tab-separated fields", "QNAME empty or longer than 254 bytes",
                               "FLAG not a decimal integer in [0, 65535]", "RNAME not '*' and not an @SQ name",
                               "POS not a decimal integer in [0, 2147483647]", "RNEXT not '*', '=' or an @SQ name",
                               "PNEXT not a decimal integer in [0, 2147483647]"};
  if (kind == SAM_BAD_TID)
    return fail(d->c, ECB_ERR_FORMAT, "line %lld: alignment with reference id -1 outside the header's %d references",
                (long long)line, d->n_ref);
  return fail(d->c, ECB_ERR_FORMAT, "line %lld: %s", (long long)line, kind < SAM_BAD_TID ? what[kind] : "bad line");
}

int sam_parse(ecb_sam* d, const uint8_t* text, int64_t n_bytes, int last, const int32_t** read_group,
              const int32_t** target_idx, const int32_t** hap_idx, int64_t* rows) {
  ecb_ctx* c = d->c;
  if (n_bytes < 0 || n_bytes > (1ll << 31)) return fail(c, ECB_ERR_INVALID, "a call takes 0 to 2 GiB of text, not %lld bytes", (long long)n_bytes);
  if (n_bytes > 0 && !text) return fail(c, ECB_ERR_INVALID, "NULL text");
  const bool open_end = n_bytes > 0 && text[n_bytes - 1] != '\n';
  if (open_end && !last) return fail(c, ECB_ERR_INVALID, "a call that is not the last must end with a whole line");
  CK(cudaSetDevice(c->device));

  // rows of the read the previous call left open go to the front
  if (d->open_row > 0) {
    const u64 keep = d->n_rows - d->open_row;
    const int other = 1 - d->rcur;
    for (int j = 0; j < 3; ++j) {
      CKR(ensure(c, d->rows[other][j], (size_t)keep * 4 + 4));
      if (keep)
        CK(cudaMemcpyAsync(d->rows[other][j].p, (const int32_t*)d->rows[d->rcur][j].p + d->open_row, (size_t)keep * 4,
                           cudaMemcpyDeviceToDevice, c->stream));
    }
    d->rcur = other;
    d->n_rows = keep;
    d->open_row = 0;
    CK(cudaMemsetAsync(&d->d_st->carry.open_row, 0, sizeof(unsigned long long), c->stream));
  }

  // the text, a '\n' after an open last line, zeros up to a whole segment
  const u64 n = (u64)n_bytes + (open_end ? 1 : 0);
  const u32 n_seg = (u32)((n + SAM_SEG - 1) / SAM_SEG);
  CKR(ensure(c, d->text, (size_t)n_seg * SAM_SEG + 16));
  uint8_t* txt = (uint8_t*)d->text.p;
  CK(cudaEventRecord(d->ev[0], c->stream));
  if (n_bytes > 0) CK(cudaMemcpyAsync(txt, text, (size_t)n_bytes, cudaMemcpyHostToDevice, c->stream));
  if (open_end) CK(cudaMemsetAsync(txt + n_bytes, '\n', 1, c->stream));
  if ((u64)n_seg * SAM_SEG > n) CK(cudaMemsetAsync(txt + n, 0, (size_t)n_seg * SAM_SEG - n, c->stream));
  CK(cudaEventRecord(d->ev[1], c->stream));

  // lines
  u64 n_lines64 = 0;
  if (n_seg) {
    CKR(ensure(c, d->seg_nl, (size_t)n_seg * 4));
    CKR(ensure(c, d->seg_tab, (size_t)n_seg * 4));
    const int wgrid = (int)(((u64)n_seg * 32 + 255) / 256);
    ecb_sam_count_kernel<<<wgrid, 256, 0, c->stream>>>((const uint4*)txt, n_seg, (u32*)d->seg_nl.p, (u32*)d->seg_tab.p);
    LAUNCH_CHECK("sam_count");
    CKR(device_scan<false>(c, (const u32*)d->seg_tab.p, (u32*)d->seg_tab.p, n_seg, 0, nullptr));
    CKR(device_scan<false>(c, (const u32*)d->seg_nl.p, (u32*)d->seg_nl.p, n_seg, 0, &n_lines64));
    CKR(ensure(c, d->line_end, (size_t)n_lines64 * 4 + 4));
    CKR(ensure(c, d->tabs_end, (size_t)n_lines64 * 4 + 4));
    ecb_sam_lines_kernel<<<wgrid, 256, 0, c->stream>>>((const uint4*)txt, n_seg, (const u32*)d->seg_nl.p,
                                                       (const u32*)d->seg_tab.p, (u32*)d->line_end.p, (u32*)d->tabs_end.p);
    LAUNCH_CHECK("sam_lines");
  }
  const u32 n_lines = (u32)n_lines64;
  CK(cudaEventRecord(d->ev[2], c->stream));

  // fields, checks and the filter
  u64 n_valid64 = 0;
  if (n_lines) {
    CKR(ensure(c, d->lines, (size_t)n_lines * sizeof(SamLine)));
    CKR(ensure(c, d->valid, (size_t)n_lines * 4));
    CKR(ensure(c, d->rowpos, (size_t)n_lines * 4));
    SamFields F{txt, (const u32*)d->line_end.p, (const u32*)d->tabs_end.p, n_lines,
                SamNames{(const SamNameSlot*)d->slots.p, d->mask, (const char*)d->blob.p, (const int64_t*)d->name_off.p},
                d->n_ref, d->track ? (int32_t*)d->range_min.p : nullptr, d->track ? (int32_t*)d->range_max.p : nullptr,
                d->d_st};
    ecb_sam_fields_kernel<<<(n_lines + 255) / 256, 256, 0, c->stream>>>(F, (SamLine*)d->lines.p, (u32*)d->valid.p);
    LAUNCH_CHECK("sam_fields");
    CKR(device_scan<false>(c, (const u32*)d->valid.p, (u32*)d->rowpos.p, n_lines, 0, &n_valid64));
    CKR(sam_sync_state(d));
    if (d->h_st->bad != SAM_NO_ERROR)
      return sam_bad_line(d, d->next_line + (int64_t)(d->h_st->bad >> 4), (u32)(d->h_st->bad & 15u));
  }
  CK(cudaEventRecord(d->ev[3], c->stream));

  // rules and rows
  const u32 n_valid = (u32)n_valid64;
  if (n_valid) {
    CKR(ensure(c, d->vline, (size_t)n_valid * 4));
    CKR(ensure(c, d->starts, (size_t)n_valid * 4));
    CKR(ensure(c, d->starts_x, (size_t)n_valid * 4));
    for (DevBuf& b : d->rows[d->rcur]) CKR(ensure(c, b, (size_t)(d->n_rows + n_valid) * 4, true));
    ecb_sam_compact_kernel<<<(n_lines + 255) / 256, 256, 0, c->stream>>>((const u32*)d->valid.p, (const u32*)d->rowpos.p,
                                                                         n_lines, (u32*)d->vline.p);
    LAUNCH_CHECK("sam_compact");
    const SamRecordAt A{txt, (const SamLine*)d->lines.p, (const u32*)d->vline.p};
    const int vgrid = (int)((n_valid + 255) / 256);
    ecb_read_starts_kernel<<<vgrid, 256, 0, c->stream>>>(A, n_valid, &d->d_st->carry, (u32*)d->starts.p);
    LAUNCH_CHECK("sam_starts");
    u64 n_starts = 0;
    CKR(device_scan<false>(c, (const u32*)d->starts.p, (u32*)d->starts_x.p, n_valid, 0, &n_starts));
    ecb_read_rows_kernel<<<vgrid, 256, 0, c->stream>>>(A, n_valid, (const u32*)d->starts.p, (const u32*)d->starts_x.p,
                                                        d->group, d->n_rows, (const int32_t*)d->tid_target.p,
                                                        (const int32_t*)d->tid_hap.p, &d->d_st->carry,
                                                        (int32_t*)d->rows[d->rcur][0].p, (int32_t*)d->rows[d->rcur][1].p,
                                                        (int32_t*)d->rows[d->rcur][2].p);
    LAUNCH_CHECK("sam_rows");
    d->n_rows += n_valid;
    d->group += (int64_t)n_starts;
  }
  CK(cudaEventRecord(d->ev[4], c->stream));
  CKR(sam_sync_state(d));
  d->all_alignments += n_lines;
  d->next_line += n_lines;
  d->stats.bytes += n_bytes;
  d->stats.lines += n_lines;
  d->stats.calls++;
  d->stats.h2d_ms += bam_ms(d->ev[0], d->ev[1]);
  d->stats.lines_ms += bam_ms(d->ev[1], d->ev[2]);
  d->stats.fields_ms += bam_ms(d->ev[2], d->ev[3]);
  d->stats.rules_ms += bam_ms(d->ev[3], d->ev[4]);
  if (last) {
    d->finished = true;
    d->open_row = d->n_rows;   // the end of the text closes the last read
  } else {
    d->open_row = d->h_st->carry.open_row;
  }
  *read_group = (const int32_t*)d->rows[d->rcur][0].p;
  *target_idx = (const int32_t*)d->rows[d->rcur][1].p;
  *hap_idx = (const int32_t*)d->rows[d->rcur][2].p;
  *rows = (int64_t)d->open_row;
  return ECB_OK;
}

}  // namespace

extern "C" {

int ecb_sam_create(ecb_ctx* c, const char* ref_names, const int64_t* ref_name_off, int32_t n_references,
                   const int32_t* tid_target, const int32_t* tid_hap, int64_t first_line, int track_ranges, ecb_sam** out) {
  if (!c || !out) return ECB_ERR_INVALID;
  *out = nullptr;
  if (n_references < 0 || !ref_name_off || (n_references > 0 && (!tid_target || !tid_hap)))
    return fail(c, ECB_ERR_INVALID, "bad reference tables");
  if (first_line < 1) return fail(c, ECB_ERR_INVALID, "first_line must be at least 1");
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "the device SAM decoder covers the single-sample path only");
  if (ref_name_off[0] != 0) return fail(c, ECB_ERR_INVALID, "ref_name_off[0] must be 0");
  for (int32_t i = 0; i < n_references; ++i)
    if (ref_name_off[i + 1] < ref_name_off[i] || ref_name_off[i + 1] - ref_name_off[i] > 0xFFFFFFFFll)
      return fail(c, ECB_ERR_INVALID, "ref_name_off is not a list of offsets");
  const int64_t blob_bytes = ref_name_off[n_references];
  if (blob_bytes > 0 && !ref_names) return fail(c, ECB_ERR_INVALID, "NULL ref_names");

  // the name table: open addressing on sam_hash, at most half full; the first of two equal names keeps its slot
  const u32 n_slots = std::max<u32>(16u, pow2_ceil((u64)n_references * 2));
  std::vector<SamNameSlot> slots(n_slots, SamNameSlot{0ull, -1, 0});
  for (int32_t t = 0; t < n_references; ++t) {
    const uint8_t* nm = (const uint8_t*)ref_names + ref_name_off[t];
    const u32 len = (u32)(ref_name_off[t + 1] - ref_name_off[t]);
    const unsigned long long h = sam_hash(nm, len);
    for (u32 i = (u32)h & (n_slots - 1);; i = (i + 1) & (n_slots - 1)) {
      SamNameSlot& e = slots[i];
      if (e.tid < 0) {
        e = SamNameSlot{h, t, 0};
        break;
      }
      if (e.hash == h && ref_name_off[e.tid + 1] - ref_name_off[e.tid] == len &&
          memcmp(ref_names + ref_name_off[e.tid], nm, len) == 0)
        break;
    }
  }

  CK(cudaSetDevice(c->device));
  ecb_sam* d = new ecb_sam();
  d->c = c;
  d->n_ref = n_references;
  d->track = track_ranges != 0;
  d->next_line = first_line;
  d->mask = n_slots - 1;
  auto bail = [&](int code) {
    sam_release(d);
    return code;
  };
  const size_t tb = (size_t)n_references * 4 + 4;
  int rc = ECB_OK;
  for (DevBuf* b : {&d->tid_target, &d->tid_hap, &d->range_min, &d->range_max})
    if (rc == ECB_OK) rc = ensure(c, *b, tb);
  if (rc == ECB_OK) rc = ensure(c, d->slots, (size_t)n_slots * sizeof(SamNameSlot));
  if (rc == ECB_OK) rc = ensure(c, d->blob, (size_t)blob_bytes + 16);
  if (rc == ECB_OK) rc = ensure(c, d->name_off, ((size_t)n_references + 1) * 8);
  if (rc != ECB_OK) return bail(rc);
  if (cudaMalloc(&d->d_st, sizeof(SamDevState)) != cudaSuccess || cudaMallocHost(&d->h_st, sizeof(SamDevState)) != cudaSuccess)
    return bail(fail(c, ECB_ERR_CUDA, "decoder state allocation failed"));
  for (auto& e : d->ev)
    if (cudaEventCreate(&e) != cudaSuccess) return bail(fail(c, ECB_ERR_CUDA, "cudaEventCreate failed"));
  memset(d->h_st, 0, sizeof(SamDevState));
  d->h_st->bad = SAM_NO_ERROR;
  std::vector<int32_t> lo((size_t)n_references + 1, INT32_MAX);
  const cudaMemcpyKind h2d = cudaMemcpyHostToDevice;
  bool ok = true;
  if (n_references > 0)
    ok = cudaMemcpyAsync(d->tid_target.p, tid_target, (size_t)n_references * 4, h2d, c->stream) == cudaSuccess &&
         cudaMemcpyAsync(d->tid_hap.p, tid_hap, (size_t)n_references * 4, h2d, c->stream) == cudaSuccess;
  if (ok && blob_bytes > 0) ok = cudaMemcpyAsync(d->blob.p, ref_names, (size_t)blob_bytes, h2d, c->stream) == cudaSuccess;
  ok = ok && cudaMemcpyAsync(d->name_off.p, ref_name_off, ((size_t)n_references + 1) * 8, h2d, c->stream) == cudaSuccess &&
       cudaMemcpyAsync(d->slots.p, slots.data(), (size_t)n_slots * sizeof(SamNameSlot), h2d, c->stream) == cudaSuccess &&
       cudaMemcpyAsync(d->range_min.p, lo.data(), tb, h2d, c->stream) == cudaSuccess &&
       cudaMemsetAsync(d->range_max.p, 0xFF, tb, c->stream) == cudaSuccess &&
       cudaMemcpyAsync(d->d_st, d->h_st, sizeof(SamDevState), h2d, c->stream) == cudaSuccess &&
       cudaStreamSynchronize(c->stream) == cudaSuccess;
  if (!ok) return bail(fail(c, ECB_ERR_CUDA, "decoder initialisation failed"));
  *out = d;
  return ECB_OK;
}

int ecb_sam_parse(ecb_sam* d, const uint8_t* text, int64_t n_bytes, int last, const int32_t** read_group,
                  const int32_t** target_idx, const int32_t** hap_idx, int64_t* rows) {
  if (!d || !read_group || !target_idx || !hap_idx || !rows) return ECB_ERR_INVALID;
  if (d->failed) return fail(d->c, ECB_ERR_STATE, "this decoder failed earlier; create a new one");
  if (d->finished) return fail(d->c, ECB_ERR_STATE, "this decoder has had its last call");
  const int rc = sam_parse(d, text, n_bytes, last, read_group, target_idx, hap_idx, rows);
  if (rc != ECB_OK) d->failed = true;
  return rc;
}

int ecb_sam_counters(const ecb_sam* d, int64_t* all_alignments, int64_t* n_groups) {
  if (!d || !all_alignments || !n_groups) return ECB_ERR_INVALID;
  *all_alignments = d->all_alignments;
  *n_groups = d->group + 1;
  return ECB_OK;
}

int ecb_sam_ranges(ecb_sam* d, int32_t* range_min, int32_t* range_max) {
  if (!d || (d->n_ref > 0 && (!range_min || !range_max))) return ECB_ERR_INVALID;
  ecb_ctx* c = d->c;
  if (!d->track) return fail(c, ECB_ERR_STATE, "ranges were not tracked");
  if (d->n_ref == 0) return ECB_OK;
  CK(cudaSetDevice(c->device));
  CK(cudaMemcpyAsync(range_min, d->range_min.p, (size_t)d->n_ref * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(range_max, d->range_max.p, (size_t)d->n_ref * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return ECB_OK;
}

int ecb_sam_get_stats(const ecb_sam* d, ecb_sam_stats* out) {
  if (!d || !out) return ECB_ERR_INVALID;
  *out = d->stats;
  return ECB_OK;
}

int ecb_sam_destroy(ecb_sam* d) {
  if (!d) return ECB_OK;
  cudaSetDevice(d->c->device);
  sam_release(d);
  return ECB_OK;
}

}  // extern "C"

// ---- collation of alignments by read name (kernels in ecb_collate.cuh) -----------------------------------------
// Rows of one spill in host memory: by fine bucket, file order inside a bucket.
struct CollateSpill {
  u64 m = 0;
  std::vector<u32> offs;                   // [COLLATE_BUCKETS + 1]
  std::unique_ptr<u64[]> lo, hi;           // dropped after the names pass
  std::unique_ptr<int32_t[]> tg, hp;
  std::unique_ptr<u32[]> pos;              // file-order position; after the names pass the first position of its read
};

// Rows placed in collated order, in host memory: by piece.
struct CollateChunk {
  std::vector<u32> offs;                   // [pieces + 1]
  std::unique_ptr<u32[]> id, place;
  std::unique_ptr<int32_t[]> tg, hp;
};

struct ecb_collate {
  ecb_ctx* c = nullptr;
  u64 n = 0;                          // alignments added
  DevBuf key_lo, key_hi, tg_in, hp_in;   // the added columns, in file order (after a spill: the staging area)
  DevBuf table, slot_of, bitmap, word_rank, count, cursor, rg, tg, hp, cuts;
  // after a spill: positions / first positions / places, ids, the partition's outputs and scratch, read lists
  DevBuf pos, idv, o_lo, o_hi, o_tg, o_hp, o_pos, o_id, part_counts, list;
  u32 slots = 0;
  bool pushed = false;
  cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  ecb_collate_stats stats{};
  // the budget and the spill state
  int64_t budget = 0;
  bool spilling = false;
  u64 stage = 0, res = 0, spilled = 0;   // rows the staging area takes, rows in it, rows already spilled
  std::vector<CollateSpill> spills;
  std::vector<CollateChunk> chunks;
  int64_t host_now = 0;
  void* ring[2] = {nullptr, nullptr};    // pinned staging ring of the host copies
  cudaEvent_t ring_ev[2] = {nullptr, nullptr};
  int ring_next = 0;
};

namespace {

#define COLLATE_RING_BYTES ((size_t)8 << 20)
#define COLLATE_MIN_STAGE 32

template <class F>
void for_each_buf(ecb_collate* k, F f) {
  DevBuf* all[] = {&k->key_lo, &k->key_hi, &k->tg_in, &k->hp_in, &k->table, &k->slot_of, &k->bitmap, &k->word_rank,
                   &k->count, &k->cursor, &k->rg, &k->tg, &k->hp, &k->cuts, &k->pos, &k->idv, &k->o_lo, &k->o_hi,
                   &k->o_tg, &k->o_hp, &k->o_pos, &k->o_id, &k->part_counts, &k->list};
  for (DevBuf* b : all) f(*b);
}

int64_t collate_bytes(ecb_collate* k) {
  int64_t total = 0;
  for_each_buf(k, [&](DevBuf& b) { total += (int64_t)b.bytes; });
  return total;
}

void collate_release(ecb_collate* k) {
  ecb_ctx* c = k->c;
  for_each_buf(k, [&](DevBuf& b) { release(c, b); });
  cudaStreamSynchronize(c->stream);
  for (auto& e : k->ev)
    if (e) cudaEventDestroy(e);
  for (int s = 0; s < 2; ++s) {
    if (k->ring[s]) cudaFreeHost(k->ring[s]);
    if (k->ring_ev[s]) cudaEventDestroy(k->ring_ev[s]);
  }
  delete k;
}

void note_peak(ecb_collate* k) { k->stats.device_bytes = std::max(k->stats.device_bytes, collate_bytes(k)); }

void note_host(ecb_collate* k, int64_t delta) {
  k->host_now += delta;
  k->stats.host_bytes = std::max(k->stats.host_bytes, k->host_now);
}

// Exactly `bytes` (rounded up to 256) unless the buffer already holds as many: the budgeted buffers of a spilled
// collation take none of ensure()'s growth slack.
int need(ecb_collate* k, DevBuf& b, size_t bytes) {
  if (b.bytes >= bytes) return ECB_OK;
  release(k->c, b);
  CKR(ensure(k->c, b, bytes));
  note_peak(k);
  return ECB_OK;
}

size_t round256(size_t bytes) { return (bytes + 255) & ~(size_t)255; }

// Device bytes of the one-pass collation of n alignments: rows (24 B, half of the growth slack of the add counted),
// slot, regrouped columns, bitmap and ranks, counts and offsets with R <= n, and the table.
u64 one_pass_bytes(const ecb_ctx* c, u64 n) {
  const u64 want = c->opt_collate_slots > 0 ? (u64)c->opt_collate_slots : n + n / 2;
  const u64 slots = std::max<u64>(1u << 10, pow2_ceil(want));
  return 36 * n + 4 * n + 12 * n + 8 * (n / 32 + 1) + 8 * n + 32 * slots;
}

u32 group_slots(u64 g) { return std::max<u32>(64u, pow2_ceil(g + g / 2)); }

// Device bytes of the names pass of a group of g rows: keys, positions, slots, read list, table.
u64 names_pass_bytes(u64 g) {
  return round256(8 * g) * 2 + round256(4 * g) * 2 + round256(8 * g) + 32 * (u64)group_slots(g);
}

u32 part_tiles(u64 m) { return (u32)std::max<u64>(1, (m + COLLATE_TILE - 1) / COLLATE_TILE); }

int ring_init(ecb_collate* k) {
  ecb_ctx* c = k->c;
  for (int s = 0; s < 2; ++s) {
    if (!k->ring[s]) CK(cudaHostAlloc(&k->ring[s], COLLATE_RING_BYTES, cudaHostAllocDefault));
    if (!k->ring_ev[s]) CK(cudaEventCreateWithFlags(&k->ring_ev[s], cudaEventDisableTiming));
  }
  return ECB_OK;
}

// host -> device through the pinned ring, stream-ordered: work queued after it on the stream sees the bytes.
int ring_h2d(ecb_collate* k, void* dst, const void* src, size_t bytes) {
  ecb_ctx* c = k->c;
  for (size_t off = 0; off < bytes; off += COLLATE_RING_BYTES) {
    const size_t len = std::min(COLLATE_RING_BYTES, bytes - off);
    const int s = k->ring_next;
    k->ring_next ^= 1;
    CK(cudaEventSynchronize(k->ring_ev[s]));
    memcpy(k->ring[s], (const char*)src + off, len);
    CK(cudaMemcpyAsync((char*)dst + off, k->ring[s], len, cudaMemcpyHostToDevice, c->stream));
    CK(cudaEventRecord(k->ring_ev[s], c->stream));
  }
  k->stats.h2d_bytes += (int64_t)bytes;
  return ECB_OK;
}

// device -> host through the pinned ring; returns with the bytes in dst.  The copy of one slot overlaps the host
// copy out of the other.
int ring_d2h(ecb_collate* k, void* dst, const void* src, size_t bytes) {
  ecb_ctx* c = k->c;
  int pend = -1;
  size_t pend_off = 0, pend_len = 0;
  for (size_t off = 0; off < bytes; off += COLLATE_RING_BYTES) {
    const size_t len = std::min(COLLATE_RING_BYTES, bytes - off);
    const int s = k->ring_next;
    k->ring_next ^= 1;
    CK(cudaEventSynchronize(k->ring_ev[s]));
    CK(cudaMemcpyAsync(k->ring[s], (const char*)src + off, len, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaEventRecord(k->ring_ev[s], c->stream));
    if (pend >= 0) {
      CK(cudaEventSynchronize(k->ring_ev[pend]));
      memcpy((char*)dst + pend_off, k->ring[pend], pend_len);
    }
    pend = s, pend_off = off, pend_len = len;
  }
  if (pend >= 0) {
    CK(cudaEventSynchronize(k->ring_ev[pend]));
    memcpy((char*)dst + pend_off, k->ring[pend], pend_len);
  }
  k->stats.d2h_bytes += (int64_t)bytes;
  return ECB_OK;
}

// Stable partition of rows [0, m) by `P` into nb buckets; offs (host) <- the bucket offsets [nb + 1], which are the
// scanned counters of tile 0 (one strided copy).
template <class Part>
int partition(ecb_collate* k, const Part& P, u64 m, u32 nb, std::vector<u32>& offs) {
  ecb_ctx* c = k->c;
  const u32 tiles = part_tiles(m);
  CKR(need(k, k->part_counts, (size_t)nb * tiles * 4));
  ecb_part_count_kernel<Part><<<tiles, 256, 0, c->stream>>>(P, m, nb, tiles, (u32*)k->part_counts.p);
  LAUNCH_CHECK("collate_part_count");
  CKR(device_scan<false>(c, (const u32*)k->part_counts.p, (u32*)k->part_counts.p, (u64)nb * tiles, 0, nullptr));
  ecb_part_scatter_kernel<Part><<<tiles, 256, 0, c->stream>>>(P, m, nb, tiles, (const u32*)k->part_counts.p);
  LAUNCH_CHECK("collate_part_scatter");
  offs.resize((size_t)nb + 1);
  CK(cudaMemcpy2DAsync(offs.data(), 4, k->part_counts.p, (size_t)tiles * 4, 4, nb, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  offs[nb] = (u32)m;
  k->stats.d2h_bytes += (int64_t)nb * 4;
  return ECB_OK;
}

// Move the rows of the staging area to host storage, partitioned by fine bucket.
int collate_spill(ecb_collate* k) {
  const u64 m = k->res;
  if (m == 0) return ECB_OK;
  const auto t0 = std::chrono::steady_clock::now();
  CKR(need(k, k->o_lo, (size_t)m * 8));
  CKR(need(k, k->o_hi, (size_t)m * 8));
  CKR(need(k, k->o_tg, (size_t)m * 4));
  CKR(need(k, k->o_hp, (size_t)m * 4));
  CKR(need(k, k->o_pos, (size_t)m * 4));
  SpillPart P{(const u64*)k->key_lo.p, (const u64*)k->key_hi.p, (const int32_t*)k->tg_in.p, (const int32_t*)k->hp_in.p,
              k->spilled, (u64*)k->o_lo.p, (u64*)k->o_hi.p, (int32_t*)k->o_tg.p, (int32_t*)k->o_hp.p, (u32*)k->o_pos.p};
  CollateSpill sp;
  sp.m = m;
  CKR(partition(k, P, m, COLLATE_BUCKETS, sp.offs));
  sp.lo.reset(new u64[m]);
  sp.hi.reset(new u64[m]);
  sp.tg.reset(new int32_t[m]);
  sp.hp.reset(new int32_t[m]);
  sp.pos.reset(new u32[m]);
  note_host(k, (int64_t)(28 * m + sp.offs.size() * 4));
  CKR(ring_d2h(k, sp.lo.get(), k->o_lo.p, m * 8));
  CKR(ring_d2h(k, sp.hi.get(), k->o_hi.p, m * 8));
  CKR(ring_d2h(k, sp.tg.get(), k->o_tg.p, m * 4));
  CKR(ring_d2h(k, sp.hp.get(), k->o_hp.p, m * 4));
  CKR(ring_d2h(k, sp.pos.get(), k->o_pos.p, m * 4));
  k->spills.push_back(std::move(sp));
  k->spilled += m;
  k->res = 0;
  k->stats.spills++;
  k->stats.spill_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  return ECB_OK;
}

// The add that would pass the budget: the rows held so far are spilled, and from then on device memory is a fixed
// staging area of `stage` rows (the rows, the partition's outputs and its counters).
int collate_start_spilling(ecb_collate* k) {
  ecb_ctx* c = k->c;
  CKR(ring_init(k));
  k->res = k->n;
  CKR(collate_spill(k));
  DevBuf* staged[] = {&k->key_lo, &k->key_hi, &k->tg_in, &k->hp_in, &k->o_lo, &k->o_hi, &k->o_tg, &k->o_hp, &k->o_pos,
                      &k->part_counts};
  for (DevBuf* b : staged) release(c, *b);
  const int64_t fixed = (int64_t)COLLATE_BUCKETS * 4 + 10 * 256;
  const int64_t per_row = 24 + 28 + 4 * COLLATE_BUCKETS / COLLATE_TILE;
  const int64_t stage = (k->budget - fixed) / per_row;
  if (stage < COLLATE_MIN_STAGE)
    return fail(c, ECB_ERR_LIMIT, "the collate budget of %lld bytes cannot hold a staging area of %d alignments",
                (long long)k->budget, COLLATE_MIN_STAGE);
  k->stage = (u64)stage;
  CKR(need(k, k->key_lo, (size_t)stage * 8));
  CKR(need(k, k->key_hi, (size_t)stage * 8));
  CKR(need(k, k->tg_in, (size_t)stage * 4));
  CKR(need(k, k->hp_in, (size_t)stage * 4));
  CKR(need(k, k->o_lo, (size_t)stage * 8));
  CKR(need(k, k->o_hi, (size_t)stage * 8));
  CKR(need(k, k->o_tg, (size_t)stage * 4));
  CKR(need(k, k->o_hp, (size_t)stage * 4));
  CKR(need(k, k->o_pos, (size_t)stage * 4));
  CKR(need(k, k->part_counts, (size_t)COLLATE_BUCKETS * part_tiles(stage) * 4));
  k->spilling = true;
  return ECB_OK;
}

// The name table over rows [0, n) (positions from `pos`, or the row index).  A table that runs out of probes is
// replaced by one four times larger and the insert runs again from the start: positions are file-order indices, so
// a rerun gives the same slots' contents whatever happened before.  exact: budgeted allocation (need).
int collate_table(ecb_collate* k, const u64* lo, const u64* hi, const u32* pos, u64 n, u32 slots, bool exact) {
  ecb_ctx* c = k->c;
  k->slots = slots;
  CKR(exact ? need(k, k->slot_of, (size_t)n * 4) : ensure(c, k->slot_of, (size_t)n * 4));
  for (;;) {
    CKR(exact ? need(k, k->table, (size_t)k->slots * sizeof(EcbEntry)) : ensure(c, k->table, (size_t)k->slots * sizeof(EcbEntry)));
    CK(cudaMemsetAsync(k->table.p, 0xFF, (size_t)k->slots * sizeof(EcbEntry), c->stream));
    CK(cudaMemsetAsync(c->d_ctr->scratch, 0, 2 * sizeof(u32), c->stream));
    CollateParams P{lo, hi, pos, n, (EcbEntry*)k->table.p, k->slots - 1, (u32*)k->slot_of.p, c->d_ctr};
    ecb_collate_insert_kernel<<<grid_for(n, 256, c->sm_count * 8), 256, 0, c->stream>>>(P);
    LAUNCH_CHECK("collate_insert");
    CKR(sync_counters(c));
    if (c->h_ctr->scratch[1] == 0) break;
    if (k->slots >= (1u << 31)) return fail(c, ECB_ERR_LIMIT, "the name table cannot grow beyond 2^31 slots");
    k->slots = k->slots <= (1u << 29) ? k->slots * 4u : (1u << 31);
    k->stats.table_grows++;
  }
  k->stats.table_slots = std::max<int64_t>(k->stats.table_slots, k->slots);
  return ECB_OK;
}

int collate_push(ecb_collate* k, int64_t* n_reads) {
  ecb_ctx* c = k->c;
  const u64 n = k->n;
  *n_reads = 0;
  if (n == 0) return ECB_OK;
  float ms = 0;
  CK(cudaEventRecord(k->ev[0], c->stream));
  const u64 want = c->opt_collate_slots > 0 ? (u64)c->opt_collate_slots : k->n + k->n / 2;
  CKR(collate_table(k, (const u64*)k->key_lo.p, (const u64*)k->key_hi.p, nullptr, k->n,
                    std::max<u32>(1u << 10, pow2_ceil(want)), false));
  k->stats.reads = c->h_ctr->scratch[0];
  const u32 R = (u32)k->stats.reads;
  CK(cudaEventRecord(k->ev[1], c->stream));

  // read order: first positions -> bitmap -> word ranks -> read ids; alignments per read -> read offsets
  const size_t words = (size_t)(n / 32) + 1;
  CKR(ensure(c, k->bitmap, words * 4));
  CKR(ensure(c, k->word_rank, words * 4));
  CKR(ensure(c, k->count, (size_t)R * 4));
  CKR(ensure(c, k->cursor, (size_t)R * 4));
  CK(cudaMemsetAsync(k->bitmap.p, 0, words * 4, c->stream));
  const int g_slots = grid_for(k->slots, 256, c->sm_count * 8);
  ecb_collate_mark_kernel<<<g_slots, 256, 0, c->stream>>>((const EcbEntry*)k->table.p, k->slots, (u32*)k->bitmap.p);
  LAUNCH_CHECK("collate_mark");
  CKR(device_scan<true>(c, (const u32*)k->bitmap.p, (u32*)k->word_rank.p, words, 0, nullptr));
  ecb_collate_ids_kernel<<<g_slots, 256, 0, c->stream>>>((EcbEntry*)k->table.p, k->slots, (const u32*)k->bitmap.p,
                                                         (const u32*)k->word_rank.p, (u32*)k->count.p);
  LAUNCH_CHECK("collate_ids");
  u64 total = 0;
  CKR(device_scan<false>(c, (const u32*)k->count.p, (u32*)k->cursor.p, R, 0, &total));
  if (total != n) return fail(c, ECB_ERR_INVALID, "collation lost alignments (%llu of %llu placed)", (unsigned long long)total,
                              (unsigned long long)n);
  CK(cudaEventRecord(k->ev[2], c->stream));

  // layout: the regrouped columns, then the pieces
  CKR(ensure(c, k->rg, (size_t)n * 4));
  CKR(ensure(c, k->tg, (size_t)n * 4));
  CKR(ensure(c, k->hp, (size_t)n * 4));
  ecb_collate_scatter_kernel<<<grid_for(n, 256, c->sm_count * 8), 256, 0, c->stream>>>(
      (const u32*)k->slot_of.p, (const EcbEntry*)k->table.p, (const int32_t*)k->tg_in.p, (const int32_t*)k->hp_in.p, n,
      (u32*)k->cursor.p, (int32_t*)k->rg.p, (int32_t*)k->tg.p, (int32_t*)k->hp.p);
  LAUNCH_CHECK("collate_scatter");
  const u64 piece = c->opt_collate_piece > 0 ? (u64)c->opt_collate_piece : (u64)ECB_PUSH_LIMIT;
  const size_t max_cuts = (size_t)(2 * (n / piece) + 4);   // two neighbouring pieces hold more than `piece` alignments
  CKR(ensure(c, k->cuts, (max_cuts + 2) * 4));
  ecb_collate_cuts_kernel<<<1, 32, 0, c->stream>>>((const u32*)k->cursor.p, R, n, piece, (u32*)k->cuts.p);
  LAUNCH_CHECK("collate_cuts");
  std::vector<u32> cuts(max_cuts + 2);
  CK(cudaMemcpyAsync(cuts.data(), k->cuts.p, cuts.size() * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaEventRecord(k->ev[3], c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const u32 pieces = cuts[0];
  if (pieces == 0 || pieces > max_cuts || cuts[1 + pieces] != n)
    return fail(c, ECB_ERR_INVALID, "collation cut %u pieces", pieces);
  note_peak(k);

  // push: the columns never leave the device; order_base = the piece's offset in collated order
  CK(cudaEventRecord(k->ev[4], c->stream));
  for (u32 j = 0; j < pieces; ++j) {
    const u64 a = cuts[1 + j], b = cuts[2 + j];
    CKR(ecb_push(c, (const int32_t*)k->rg.p + a, (const int32_t*)k->tg.p + a, (const int32_t*)k->hp.p + a, nullptr,
                 (int64_t)(b - a), (int64_t)a, 0, 1));
    k->stats.pieces++;
  }
  CK(cudaEventRecord(k->ev[5], c->stream));
  CK(cudaEventSynchronize(k->ev[5]));
  CK(cudaEventElapsedTime(&ms, k->ev[0], k->ev[1])); k->stats.table_ms = ms;
  CK(cudaEventElapsedTime(&ms, k->ev[1], k->ev[2])); k->stats.order_ms = ms;
  CK(cudaEventElapsedTime(&ms, k->ev[2], k->ev[3])); k->stats.layout_ms = ms;
  CK(cudaEventElapsedTime(&ms, k->ev[4], k->ev[5])); k->stats.push_ms = ms;
  *n_reads = (int64_t)R;
  return ECB_OK;
}

// ---- collation after a spill (DESIGN.md section 6.2): names per group, order once, layout per chunk, push per piece
// 1. names: the rows of a group of fine buckets go up (keys and positions), the group's name table marks the global
//    bitmap, and the group's reads (first position, alignments) and every row's read's first position come back.
int spilled_names(ecb_collate* k, std::vector<uint2>& reads) {
  ecb_ctx* c = k->c;
  const u64 n = k->n;
  const size_t words = (size_t)(n / 32) + 1;
  const int64_t avail = k->budget - (int64_t)round256(words * 4);
  if (avail <= 0)
    return fail(c, ECB_ERR_LIMIT, "the collate budget of %lld bytes cannot hold the bitmap of %llu alignments (%llu bytes)",
                (long long)k->budget, (unsigned long long)n, (unsigned long long)round256(words * 4));
  // groups of consecutive buckets whose names pass fits next to the bitmap
  std::vector<u64> rows(COLLATE_BUCKETS, 0);
  for (const CollateSpill& sp : k->spills)
    for (u32 b = 0; b < COLLATE_BUCKETS; ++b) rows[b] += sp.offs[b + 1] - sp.offs[b];
  std::vector<u32> bounds{0};
  u64 g = 0;
  for (u32 b = 0; b < COLLATE_BUCKETS; ++b) {
    if (names_pass_bytes(rows[b]) > (u64)avail)
      return fail(c, ECB_ERR_LIMIT, "a name bucket of %llu alignments does not fit the collate budget of %lld bytes",
                  (unsigned long long)rows[b], (long long)k->budget);
    if (g > 0 && names_pass_bytes(g + rows[b]) > (u64)avail) {
      bounds.push_back(b);
      g = 0;
    }
    g += rows[b];
  }
  bounds.push_back(COLLATE_BUCKETS);
  k->stats.groups = (int64_t)bounds.size() - 1;

  CKR(need(k, k->bitmap, words * 4));
  CK(cudaMemsetAsync(k->bitmap.p, 0, words * 4, c->stream));
  for (size_t gi = 0; gi + 1 < bounds.size(); ++gi) {
    const u32 b0 = bounds[gi], b1 = bounds[gi + 1];
    u64 m = 0;
    for (const CollateSpill& sp : k->spills) m += sp.offs[b1] - sp.offs[b0];
    if (m == 0) continue;
    CKR(need(k, k->key_lo, (size_t)m * 8));
    CKR(need(k, k->key_hi, (size_t)m * 8));
    CKR(need(k, k->pos, (size_t)m * 4));
    CKR(need(k, k->list, (size_t)m * 8));
    // spill after spill: the rows of one name stay in file order
    u64 off = 0;
    for (const CollateSpill& sp : k->spills) {
      const u64 a = sp.offs[b0], e = sp.offs[b1];
      if (e == a) continue;
      CKR(ring_h2d(k, (u64*)k->key_lo.p + off, sp.lo.get() + a, (e - a) * 8));
      CKR(ring_h2d(k, (u64*)k->key_hi.p + off, sp.hi.get() + a, (e - a) * 8));
      CKR(ring_h2d(k, (u32*)k->pos.p + off, sp.pos.get() + a, (e - a) * 4));
      off += e - a;
    }
    CKR(collate_table(k, (const u64*)k->key_lo.p, (const u64*)k->key_hi.p, (const u32*)k->pos.p, m, group_slots(m), true));
    const u32 group_reads = c->h_ctr->scratch[0];
    const int g_slots = grid_for(k->slots, 256, c->sm_count * 8);
    ecb_collate_mark_kernel<<<g_slots, 256, 0, c->stream>>>((const EcbEntry*)k->table.p, k->slots, (u32*)k->bitmap.p);
    LAUNCH_CHECK("collate_mark");
    CK(cudaMemsetAsync(&c->d_ctr->scratch[2], 0, sizeof(u32), c->stream));
    ecb_collate_list_kernel<<<g_slots, 256, 0, c->stream>>>((const EcbEntry*)k->table.p, k->slots, (uint2*)k->list.p,
                                                            &c->d_ctr->scratch[2]);
    LAUNCH_CHECK("collate_list");
    ecb_collate_first_kernel<<<grid_for(m, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        (const u32*)k->slot_of.p, (const EcbEntry*)k->table.p, m, (u32*)k->pos.p);
    LAUNCH_CHECK("collate_first");
    const size_t r0 = reads.size();
    reads.resize(r0 + group_reads);
    note_host(k, (int64_t)group_reads * 8);
    CKR(ring_d2h(k, reads.data() + r0, k->list.p, (size_t)group_reads * 8));
    off = 0;
    for (CollateSpill& sp : k->spills) {
      const u64 a = sp.offs[b0], e = sp.offs[b1];
      if (e == a) continue;
      CKR(ring_d2h(k, sp.pos.get() + a, (const u32*)k->pos.p + off, (e - a) * 4));
      off += e - a;
    }
  }
  for (CollateSpill& sp : k->spills) {   // the keys are done with
    sp.lo.reset();
    sp.hi.reset();
    note_host(k, -(int64_t)(16 * sp.m));
  }
  DevBuf* done[] = {&k->key_lo, &k->key_hi, &k->pos, &k->list, &k->slot_of, &k->table};
  for (DevBuf* b : done) release(c, *b);
  return ECB_OK;
}

int collate_push_spilled(ecb_collate* k, int64_t* n_reads) {
  ecb_ctx* c = k->c;
  const u64 n = k->n;
  *n_reads = 0;
  CKR(collate_spill(k));   // the rows still in the staging area
  DevBuf* staged[] = {&k->key_lo, &k->key_hi, &k->tg_in, &k->hp_in, &k->o_lo, &k->o_hi, &k->o_tg, &k->o_hp, &k->o_pos,
                      &k->part_counts};
  for (DevBuf* b : staged) release(c, *b);
  float ms = 0;
  CK(cudaEventRecord(k->ev[0], c->stream));

  // 1. names
  std::vector<uint2> reads;
  CKR(spilled_names(k, reads));
  const u64 R = reads.size();
  k->stats.reads = (int64_t)R;
  CK(cudaEventRecord(k->ev[1], c->stream));

  // 2. order: word ranks of the bitmap, alignments per read id from the read lists, read offsets, piece cuts
  const size_t words = (size_t)(n / 32) + 1;
  const int64_t global = (int64_t)(round256(words * 4) * 2 + round256(R * 4) + round256((R + 1) * 4));
  if (global + 2 * 256 >= k->budget)
    return fail(c, ECB_ERR_LIMIT, "the collate budget of %lld bytes cannot hold the read order of %llu alignments in %llu "
                "reads (%lld bytes)", (long long)k->budget, (unsigned long long)n, (unsigned long long)R, (long long)global);
  CKR(need(k, k->word_rank, words * 4));
  CKR(device_scan<true>(c, (const u32*)k->bitmap.p, (u32*)k->word_rank.p, words, 0, nullptr));
  CKR(need(k, k->count, (size_t)R * 4));
  CKR(need(k, k->cursor, (size_t)(R + 1) * 4));
  const u64 per_upload = std::max<u64>(1, std::min<u64>(R, (u64)(k->budget - global - 256) / 8));
  CKR(need(k, k->list, (size_t)per_upload * 8));
  for (u64 a = 0; a < R; a += per_upload) {
    const u64 len = std::min(per_upload, R - a);
    CKR(ring_h2d(k, k->list.p, reads.data() + a, len * 8));
    ecb_collate_list_ids_kernel<<<grid_for(len, 256, c->sm_count * 8), 256, 0, c->stream>>>(
        (const uint2*)k->list.p, len, (const u32*)k->bitmap.p, (const u32*)k->word_rank.p, (u32*)k->count.p);
    LAUNCH_CHECK("collate_list_ids");
  }
  release(c, k->list);
  std::vector<uint2>().swap(reads);
  note_host(k, -(int64_t)R * 8);
  u64 total = 0;
  CKR(device_scan<false>(c, (const u32*)k->count.p, (u32*)k->cursor.p, R, 0, &total));
  if (total != n) return fail(c, ECB_ERR_INVALID, "collation lost alignments (%llu of %llu placed)", (unsigned long long)total,
                              (unsigned long long)n);
  const u32 n32 = (u32)n;   // cursor[R] = n: cursor + 1 are the read ends
  CK(cudaMemcpyAsync((u32*)k->cursor.p + R, &n32, 4, cudaMemcpyHostToDevice, c->stream));
  // a piece's columns and its upload area (28 B per alignment) fit the budget; at most COLLATE_MAX_PARTS pieces
  const u64 fit = (u64)std::max<int64_t>(1, (k->budget - 8 * 256) / 28);
  const u64 piece = std::min<u64>(c->opt_collate_piece > 0 ? (u64)c->opt_collate_piece : (u64)ECB_PUSH_LIMIT, fit);
  const size_t max_cuts = (size_t)(2 * (n / piece) + 4);
  if (max_cuts > COLLATE_MAX_PARTS)
    return fail(c, ECB_ERR_LIMIT, "pieces of %llu alignments cut %llu alignments into more than %d pieces (collate budget "
                "%lld bytes)", (unsigned long long)piece, (unsigned long long)n, COLLATE_MAX_PARTS, (long long)k->budget);
  CKR(need(k, k->cuts, (max_cuts + 2) * 4));
  ecb_collate_cuts_kernel<<<1, 32, 0, c->stream>>>((const u32*)k->cursor.p + 1, (u32)R, n, piece, (u32*)k->cuts.p);
  LAUNCH_CHECK("collate_cuts");
  std::vector<u32> cuts(max_cuts + 2);
  CK(cudaMemcpyAsync(cuts.data(), k->cuts.p, cuts.size() * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  k->stats.d2h_bytes += (int64_t)cuts.size() * 4;
  const u32 pieces = cuts[0];
  if (pieces == 0 || pieces > max_cuts || cuts[1 + pieces] != n)
    return fail(c, ECB_ERR_INVALID, "collation cut %u pieces", pieces);
  CK(cudaEventRecord(k->ev[2], c->stream));

  // 3. layout: every row takes its read id and its place in collated order, and the rows are partitioned by piece
  const int64_t fixed = global + (int64_t)round256((max_cuts + 2) * 4) + 4 * (int64_t)pieces + 10 * 256;
  const int64_t per_row = 32 + (4 * (int64_t)pieces + COLLATE_TILE - 1) / COLLATE_TILE;
  const u64 chunk = (u64)std::max<int64_t>(0, (k->budget - fixed) / per_row);
  if (chunk == 0)
    return fail(c, ECB_ERR_LIMIT, "the collate budget of %lld bytes cannot hold the read order and a layout chunk",
                (long long)k->budget);
  for (CollateSpill& sp : k->spills) {
    for (u64 a = 0; a < sp.m; a += chunk) {
      const u64 m = std::min(chunk, sp.m - a);
      DevBuf* cols[] = {&k->tg_in, &k->hp_in, &k->pos, &k->idv, &k->o_tg, &k->o_hp, &k->o_pos, &k->o_id};
      for (DevBuf* b : cols) CKR(need(k, *b, (size_t)m * 4));
      CKR(ring_h2d(k, k->tg_in.p, sp.tg.get() + a, m * 4));
      CKR(ring_h2d(k, k->hp_in.p, sp.hp.get() + a, m * 4));
      CKR(ring_h2d(k, k->pos.p, sp.pos.get() + a, m * 4));
      ecb_collate_place_kernel<<<grid_for(m, 256, c->sm_count * 8), 256, 0, c->stream>>>(
          (u32*)k->pos.p, m, (const u32*)k->bitmap.p, (const u32*)k->word_rank.p, (u32*)k->cursor.p, (u32*)k->idv.p);
      LAUNCH_CHECK("collate_place");
      PiecePart P{(const u32*)k->idv.p, (const u32*)k->pos.p, (const int32_t*)k->tg_in.p, (const int32_t*)k->hp_in.p,
                  (const u32*)k->cuts.p + 1, pieces, (u32*)k->o_id.p, (u32*)k->o_pos.p, (int32_t*)k->o_tg.p,
                  (int32_t*)k->o_hp.p};
      CollateChunk ch;
      CKR(partition(k, P, m, pieces, ch.offs));
      ch.id.reset(new u32[m]);
      ch.place.reset(new u32[m]);
      ch.tg.reset(new int32_t[m]);
      ch.hp.reset(new int32_t[m]);
      note_host(k, (int64_t)(16 * m + ch.offs.size() * 4));
      CKR(ring_d2h(k, ch.id.get(), k->o_id.p, m * 4));
      CKR(ring_d2h(k, ch.place.get(), k->o_pos.p, m * 4));
      CKR(ring_d2h(k, ch.tg.get(), k->o_tg.p, m * 4));
      CKR(ring_d2h(k, ch.hp.get(), k->o_hp.p, m * 4));
      k->chunks.push_back(std::move(ch));
    }
    sp.tg.reset();
    sp.hp.reset();
    sp.pos.reset();
    note_host(k, -(int64_t)(12 * sp.m + sp.offs.size() * 4));
  }
  k->spills.clear();
  {
    DevBuf* done[] = {&k->bitmap, &k->word_rank, &k->count, &k->cursor, &k->cuts, &k->tg_in, &k->hp_in, &k->pos,
                      &k->idv, &k->o_tg, &k->o_hp, &k->o_pos, &k->o_id, &k->part_counts};
    for (DevBuf* b : done) release(c, *b);
  }
  CK(cudaEventRecord(k->ev[3], c->stream));

  // 4. push: per piece, every chunk's rows of the piece go up and land at place - piece start
  u64 longest = 0;
  for (u32 j = 0; j < pieces; ++j) longest = std::max<u64>(longest, cuts[2 + j] - cuts[1 + j]);
  const u64 upload = std::max<u64>(1, std::min(longest, piece));
  CKR(need(k, k->rg, (size_t)longest * 4));
  CKR(need(k, k->tg, (size_t)longest * 4));
  CKR(need(k, k->hp, (size_t)longest * 4));
  DevBuf* up[] = {&k->idv, &k->tg_in, &k->hp_in, &k->pos};
  for (DevBuf* b : up) CKR(need(k, *b, (size_t)upload * 4));
  for (u32 j = 0; j < pieces; ++j) {
    const u64 a = cuts[1 + j], b = cuts[2 + j];
    for (const CollateChunk& ch : k->chunks) {
      for (u64 s = ch.offs[j]; s < ch.offs[j + 1]; s += upload) {
        const u64 m = std::min<u64>(upload, ch.offs[j + 1] - s);
        CKR(ring_h2d(k, k->idv.p, ch.id.get() + s, m * 4));
        CKR(ring_h2d(k, k->tg_in.p, ch.tg.get() + s, m * 4));
        CKR(ring_h2d(k, k->hp_in.p, ch.hp.get() + s, m * 4));
        CKR(ring_h2d(k, k->pos.p, ch.place.get() + s, m * 4));
        ecb_collate_piece_kernel<<<grid_for(m, 256, c->sm_count * 8), 256, 0, c->stream>>>(
            (const u32*)k->idv.p, (const int32_t*)k->tg_in.p, (const int32_t*)k->hp_in.p, (const u32*)k->pos.p, m, (u32)a,
            (int32_t*)k->rg.p, (int32_t*)k->tg.p, (int32_t*)k->hp.p);
        LAUNCH_CHECK("collate_piece");
      }
    }
    CKR(ecb_push(c, (const int32_t*)k->rg.p, (const int32_t*)k->tg.p, (const int32_t*)k->hp.p, nullptr, (int64_t)(b - a),
                 (int64_t)a, 0, 1));
    k->stats.pieces++;
  }
  CK(cudaEventRecord(k->ev[4], c->stream));
  CK(cudaEventSynchronize(k->ev[4]));
  for (const CollateChunk& ch : k->chunks) note_host(k, -(int64_t)(16 * (u64)ch.offs.back() + ch.offs.size() * 4));
  k->chunks.clear();
  CK(cudaEventElapsedTime(&ms, k->ev[0], k->ev[1])); k->stats.table_ms = ms;
  CK(cudaEventElapsedTime(&ms, k->ev[1], k->ev[2])); k->stats.order_ms = ms;
  CK(cudaEventElapsedTime(&ms, k->ev[2], k->ev[3])); k->stats.layout_ms = ms;
  CK(cudaEventElapsedTime(&ms, k->ev[3], k->ev[4])); k->stats.push_ms = ms;
  *n_reads = (int64_t)R;
  return ECB_OK;
}

}  // namespace

extern "C" {

int ecb_collate_create(ecb_ctx* c, ecb_collate** out) {
  if (!c || !out) return ECB_ERR_INVALID;
  *out = nullptr;
  if (c->with_cells) return fail(c, ECB_ERR_INVALID, "collation covers the single-sample path only");
  CK(cudaSetDevice(c->device));
  size_t free_bytes = 0, total_bytes = 0;
  CK(cudaMemGetInfo(&free_bytes, &total_bytes));
  ecb_collate* k = new ecb_collate();
  k->c = c;
  // automatic: half the free memory, the other half is left to the context's EC table and results
  k->budget = c->opt_collate_budget > 0 ? c->opt_collate_budget : (int64_t)(free_bytes / 2);
  for (auto& e : k->ev)
    if (cudaEventCreate(&e) != cudaSuccess) {
      collate_release(k);
      return fail(c, ECB_ERR_CUDA, "cudaEventCreate failed");
    }
  *out = k;
  return ECB_OK;
}

int ecb_collate_add(ecb_collate* k, const uint64_t* key_lo, const uint64_t* key_hi, const int32_t* target_idx,
                    const int32_t* hap_idx, int64_t n, int on_device) {
  if (!k) return ECB_ERR_INVALID;
  ecb_ctx* c = k->c;
  if (k->pushed) return fail(c, ECB_ERR_STATE, "this collator has pushed; create a new one");
  if (n < 0) return fail(c, ECB_ERR_INVALID, "negative n");
  if (n == 0) return ECB_OK;
  if (!key_lo || !key_hi || !target_idx || !hap_idx) return fail(c, ECB_ERR_INVALID, "NULL column");
  if (k->n + (u64)n >= 0xFFFFFFFFull) return fail(c, ECB_ERR_LIMIT, "a collator takes fewer than 2^32 - 1 alignments");
  CK(cudaSetDevice(c->device));
  const u64 total = k->n + (u64)n;
  const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  if (!k->spilling && one_pass_bytes(c, total) > (u64)k->budget) CKR(collate_start_spilling(k));
  if (!k->spilling) {
    CKR(ensure(c, k->key_lo, (size_t)total * 8, true));
    CKR(ensure(c, k->key_hi, (size_t)total * 8, true));
    CKR(ensure(c, k->tg_in, (size_t)total * 4, true));
    CKR(ensure(c, k->hp_in, (size_t)total * 4, true));
  }
  CK(cudaEventRecord(k->ev[0], c->stream));
  if (!k->spilling) {
    CK(cudaMemcpyAsync((u64*)k->key_lo.p + k->n, key_lo, (size_t)n * 8, kind, c->stream));
    CK(cudaMemcpyAsync((u64*)k->key_hi.p + k->n, key_hi, (size_t)n * 8, kind, c->stream));
    CK(cudaMemcpyAsync((int32_t*)k->tg_in.p + k->n, target_idx, (size_t)n * 4, kind, c->stream));
    CK(cudaMemcpyAsync((int32_t*)k->hp_in.p + k->n, hap_idx, (size_t)n * 4, kind, c->stream));
  } else {
    // the staging area takes what it can; a full one spills
    for (u64 done = 0; done < (u64)n;) {
      if (k->res == k->stage) CKR(collate_spill(k));
      const u64 r = std::min<u64>((u64)n - done, k->stage - k->res);
      CK(cudaMemcpyAsync((u64*)k->key_lo.p + k->res, key_lo + done, (size_t)r * 8, kind, c->stream));
      CK(cudaMemcpyAsync((u64*)k->key_hi.p + k->res, key_hi + done, (size_t)r * 8, kind, c->stream));
      CK(cudaMemcpyAsync((int32_t*)k->tg_in.p + k->res, target_idx + done, (size_t)r * 4, kind, c->stream));
      CK(cudaMemcpyAsync((int32_t*)k->hp_in.p + k->res, hap_idx + done, (size_t)r * 4, kind, c->stream));
      k->res += r;
      done += r;
    }
  }
  CK(cudaEventRecord(k->ev[1], c->stream));
  CK(cudaEventSynchronize(k->ev[1]));   // the caller's buffers are free again
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, k->ev[0], k->ev[1]));
  k->stats.add_ms += ms;
  if (!on_device) k->stats.h2d_bytes += n * 24;
  k->n = total;
  k->stats.alignments = (int64_t)total;
  note_peak(k);
  return ECB_OK;
}

int ecb_collate_push(ecb_collate* k, int64_t* n_reads) {
  if (!k || !n_reads) return ECB_ERR_INVALID;
  if (k->pushed) return fail(k->c, ECB_ERR_STATE, "this collator has pushed already");
  ecb_ctx* c = k->c;
  k->pushed = true;
  CK(cudaSetDevice(c->device));
  return k->spilling ? collate_push_spilled(k, n_reads) : collate_push(k, n_reads);
}

int ecb_collate_get_stats(const ecb_collate* k, ecb_collate_stats* out) {
  if (!k || !out) return ECB_ERR_INVALID;
  *out = k->stats;
  return ECB_OK;
}

int ecb_collate_destroy(ecb_collate* k) {
  if (!k) return ECB_OK;
  cudaSetDevice(k->c->device);
  collate_release(k);
  return ECB_OK;
}

}  // extern "C"
