/*
 * ecb200.h — C ABI of libecb200.so: B200 (sm_100a) equivalence-class builder for alntools bam2ec.
 *
 * The reference (churchill-lab/alntools) is pure Python and has no FFI; the seam this library
 * replaces is the body of its per-alignment grouping loop, the chunk merge, the EC -> COO loop and
 * the scipy canonicalisation, fed with int32 columns instead of pysam objects:
 *
 *   ecb_push      replaces  alntools/bam_utils.py:258-344  (process_convert_bam hot loop: group by
 *                           read, set of tids per read, ec[key] += 1) and the chunk-ordered merge
 *                           alntools/bam_utils.py:680-698 (EC id = rank of first occurrence);
 *                           with cells: alntools/bam_utils_multisample.py:209-300 and :503-560.
 *   ecb_finalize  replaces  alntools/bam_utils.py:788-847 (EC -> per-haplotype COO -> APM) plus the
 *                           matrix part of alntools/bin_utils.py:208-232,246-275 (sum 2^h*data[h],
 *                           tocsr, N as CSC); with cells: bam_utils_multisample.py:595-636,702-791.
 *
 * Host code (alntools_b200/*.py) keeps the reference's convert()/methods/CLI signatures, decodes
 * the BAM, applies the filters (bam_utils.py:264-270) and the read-name comparison (:301-306), and
 * hands over columns.  No torch types cross this boundary: plain pointers and sizes only.
 *
 * All functions return 0 on success and a negative ecb_status on failure; the message is available
 * through ecb_last_error().  Nothing here ever falls back to a CPU implementation.
 *
 * Threading: a context is bound to one CUDA device and one stream and is not thread-safe; use one
 * context per GPU.  Calls block the calling thread until the work they describe is finished unless
 * stated otherwise (ctypes releases the GIL around them).
 */
#ifndef ECB200_H
#define ECB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ecb_ctx ecb_ctx;

enum ecb_status {
  ECB_OK = 0,
  ECB_ERR_INVALID = -1,     /* bad argument / contract violation */
  ECB_ERR_CUDA = -2,        /* CUDA runtime error (message has the CUDA string) */
  ECB_ERR_NO_DEVICE = -3,   /* no usable sm_100 device */
  ECB_ERR_LIMIT = -4,       /* a format limit was exceeded (int32 file fields, read too long, ...) */
  ECB_ERR_EMPTY = -5,       /* finalize with zero equivalence classes (the reference raises too:
                               alntools/matrix/Sparse3DMatrix.py:45-46) */
  ECB_ERR_STATE = -6,       /* call sequence error */
  ECB_ERR_FORMAT = -7       /* malformed BAM input of the device decoder (ecb_bam_decode; since version 2002),
                               malformed EC-file arrays (ecb_push_ecs / ecb_sample_append; since version 2007), or
                               a bad SAM line (ecb_sam_parse; since version 2008) */
};

/* Longest read (alignments sharing one name) a push accepts by default, and the longest one the grouping kernel
 * keys inline.  ECB_OPT_MAX_READ raises the limit: longer reads then take a sort-based pass of their own. */
#define ECB_MAX_READ_ALIGNMENTS 16384
/* target_idx < 2^26 and hap_idx < 31 (the EC file stores the haplotype mask in an int32,
 * alntools/bin_utils.py:232). */
#define ECB_MAX_TARGETS (1 << 26)
#define ECB_MAX_HAPS 31

enum ecb_option {
  ECB_OPT_RESULT_ON_DEVICE = 1, /* 1: ecb_result pointers are DEVICE pointers (no D2H copy) */
  ECB_OPT_TABLE_SLOTS = 2,      /* initial EC hash-table capacity (rounded up to a power of two) */
  ECB_OPT_PAIR_SLOTS = 3,       /* initial (file, EC, cell) table capacity */
  ECB_OPT_GRID_CTAS = 4,        /* CTAs of the grouping kernel (0 = one persistent CTA per SM) */
  ECB_OPT_HOT_CACHE = 5,        /* 1 (default): per-CTA shared-memory cache of hot ECs in front of the HBM table */
  ECB_OPT_VERIFY_KEYS = 6,      /* 1: every push re-derives each read's set of (target, haplotype) pairs and
                                   compares it with the row of the EC the read was counted in, turning
                                   a 128-bit key collision into ECB_ERR_LIMIT (slow; a debugging aid) */
  ECB_OPT_CHUNK_LEN = 7,        /* alignments per work chunk of the grouping kernel (0 = automatic) */
  ECB_OPT_PAGEABLE_RESULTS = 8, /* 1: host results go to ordinary (malloc) memory instead of pinned memory:
                                   cheaper for a context that finalizes once, slower when reused */
  ECB_OPT_BAM_WINDOW = 9,       /* inflated bytes per window of the device BAM decoder (0 = automatic, 1 GiB);
                                   a window always takes at least one block */
  ECB_OPT_COLLATE_SLOTS = 10,   /* initial slots of a collator's name table (0 = automatic: 1.5 x the alignments
                                   added, rounded up to a power of two); the table grows when it runs out of probes */
  ECB_OPT_COLLATE_PIECE = 11,   /* most alignments one push of a collator carries (0 = the push limit, 2^31 - 8192) */
  ECB_OPT_COLLATE_BUDGET = 12,  /* device bytes a collator may hold, read at ecb_collate_create (0 = automatic: half
                                   of the device's free memory at that moment, the rest is left to the context's EC
                                   table and results; since version 2004) */
  ECB_OPT_MAX_READ = 13,        /* longest read a push accepts (default ECB_MAX_READ_ALIGNMENTS; 0 = the push limit,
                                   2^31 - 8192; other values below ECB_MAX_READ_ALIGNMENTS are ECB_ERR_INVALID).  A
                                   longer read fails the push with ECB_ERR_LIMIT.  Reads above ECB_MAX_READ_ALIGNMENTS
                                   are deferred by the grouping kernel and keyed, counted and given their rows by a
                                   sort of their alignments on the device (24 bytes per such alignment while it
                                   runs); shorter reads take the inline path either way.  The default stays as it
                                   is because in a file grouped by name so long a read is more often a broken input
                                   than a real one.  Since version 2005 */
};

typedef struct ecb_result {
  int64_t n_ec;              /* E: number of equivalence classes (after the cell filter)          */
  int64_t nnz_a;             /* Z                                                                 */
  const int32_t* a_indptr;   /* [E+1]  CSR row offsets of the A matrix (E x T)                    */
  const int32_t* a_indices;  /* [Z]    main-target index, ascending inside a row                  */
  const int32_t* a_data;     /* [Z]    haplotype bitmask, bit h = sorted-haplotype index h        */
  int64_t n_samples;         /* S: 1 without cells; number of kept cells with cells; samples closed
                                by ecb_finalize_samples                                            */
  int64_t nnz_n;
  const int32_t* n_indptr;   /* [S+1]  CSC column offsets of the N matrix (E x S)                 */
  const int32_t* n_indices;  /* [nnz_n] EC ids, ascending inside a column                         */
  const int32_t* n_data;     /* [nnz_n] read counts                                               */
  const int32_t* cell_order; /* [S] original cell_idx of every output column; NULL without cells  */
  int64_t n_reads;           /* reads counted over all pushes (after drop_last_group)             */
  int64_t n_alignments;      /* alignments pushed                                                 */
} ecb_result;

typedef struct ecb_stats {
  double group_ms;        /* device time of the grouping/insert kernel(s) of the last push        */
  double harvest_ms;      /* device time of the row-harvest kernels of the last push              */
  double push_ms;         /* device time of the whole last push (incl. H2D when host pointers)    */
  double finalize_ms;     /* device time of the last finalize (incl. D2H unless result on device) */
  int64_t kernel_launches;/* kernels launched by this library since create/reset                  */
  int64_t table_slots;    /* current EC table capacity                                            */
  int64_t table_used;     /* ECs in the table                                                     */
  int64_t table_grows;    /* rehash events                                                        */
  int64_t overflow_reads; /* reads that had to be replayed after a table growth                   */
  int64_t h2d_bytes;      /* bytes copied host->device since create/reset                         */
  int64_t d2h_bytes;      /* bytes copied device->host since create/reset                         */
  int64_t row_entries;    /* (target, mask) pairs reserved in the row arena (upper bound of nnz)   */
  /* since version 2005 */
  int64_t long_reads;     /* reads longer than ECB_MAX_READ_ALIGNMENTS in the last push (deferred) */
  double long_ms;         /* device time of the deferred pass of the last push                    */
  /* since version 2006 */
  int64_t samples;        /* samples closed since create/reset (ecb_sample_close)                  */
  int64_t sample_pairs;   /* (EC, sample) entries they recorded                                    */
  double sample_ms;       /* device time of the closes, summed                                     */
  /* since version 2007 */
  int64_t ec_pushes;      /* ecb_push_ecs calls since create/reset                                 */
  int64_t ec_rows;        /* EC rows they pushed                                                   */
  int64_t ec_claimed;     /* ECs those rows claimed (rows whose set was new to the context)        */
  double ec_ms;           /* device time of those pushes, summed (incl. H2D when host arrays)      */
  double ec_check_ms;     /* ... of it spent in the exact check of the rows that found an EC       */
} ecb_stats;

/* Library/ABI version (major*1000 + minor). */
int ecb_version(void);

/* Create a context on CUDA device `device`.  n_targets/n_haps bound the column values;
 * with_cells selects the per-cell (multisample) path; alignments_hint sizes tables and staging. */
int ecb_create(ecb_ctx** out, int device, int n_targets, int n_haps, int with_cells,
               int64_t alignments_hint);

int ecb_set_option(ecb_ctx* ctx, int option, int64_t value);

/* Run all work of this context on an existing CUDA stream (a cudaStream_t passed as void*),
 * e.g. torch.cuda.current_stream().cuda_stream.  NULL restores the context's own stream; the legacy
 * default stream must be named explicitly (cudaStreamLegacy), because its plain handle is NULL too. */
int ecb_set_stream(ecb_ctx* ctx, void* cuda_stream);

/*
 * Push one contiguous run of VALID alignments (already filtered, name-grouped).
 *   read_group[n]  consecutive equal values form one read; values only need to change between reads
 *   target_idx[n]  main-target index of the alignment's reference   (0 <= v < n_targets)
 *   hap_idx[n]     index into the SORTED haplotype list             (0 <= v < n_haps)
 *   cell_idx[n]    cell id of the alignment's read (value on the read's first alignment is used);
 *                  NULL unless the context was created with_cells
 *   order_base     global index of this push's first alignment in reference read order: EC ids are
 *                  ranked by order_base + offset of the EC's first read, so pushes/shards may arrive
 *                  in any order as long as their [order_base, order_base+n) ranges do not overlap
 *   drop_last_group 1 reproduces alntools/bam_utils_multisample.py:306-308 (the last read of a file
 *                  is never flushed); one push = one file in that case
 *   on_device      0: host pointers (pinned preferred, copied with cudaMemcpyAsync);
 *                  1: device pointers on this context's device
 * Reads must not span pushes.  Buffers are caller-owned and may be reused after return.
 */
int ecb_push(ecb_ctx* ctx, const int32_t* read_group, const int32_t* target_idx,
             const int32_t* hap_idx, const int32_t* cell_idx, int64_t n, int64_t order_base,
             int drop_last_group, int on_device);

/* Build the A (CSR) and N (CSC) matrices.  min_cell_count follows
 * alntools/bam_utils_multisample.py:596-608 (<=0 means 1; ignored without cells).
 * Result buffers are library-owned (pinned host memory, or device memory with
 * ECB_OPT_RESULT_ON_DEVICE) and stay valid until the next finalize/reset/destroy. */
int ecb_finalize(ecb_ctx* ctx, int64_t min_cell_count, ecb_result* out);

/* ---- several samples in one single-sample context (since version 2006) ----------------------------------------
 * An EC file holds an E x S count matrix N.  Files pushed one after the other into one single-sample context share
 * its EC table, so EC identity, EC ids and the A matrix are those of one build over the concatenated columns: an EC id
 * is the rank of the EC's first occurrence over sample 1, then sample 2, and so on.  Every way of pushing works
 * unchanged inside a sample: host or device columns, several pushes, ecb_bam_decode, a collator, long reads, table
 * growth and replay.
 *
 * ecb_sample_close: the alignments pushed since the previous close (or since create/reset) are one sample; an empty
 *   sample is allowed.  One kernel compares every EC's count (read through the table after the pushes have completed)
 *   with its count at the previous close and appends (provisional id, delta) for every delta > 0 to a device list
 *   with one atomic per warp.  *nonzeros = the sample's pairs, brought back by the call's one host round trip.  From
 *   then on, order_base of ecb_push counts from the end of the closed samples' order range (the largest
 *   order_base + n pushed so far), so that every sample can be pushed from order_base 0, as one file on its own is.
 * ecb_finalize_samples: A, the EC ids and the other fields as ecb_finalize; N (CSC) has one column per closed sample:
 *   entry (e, s) is the reads of sample s in EC e, zeros are not stored, EC ids ascend inside a column and an empty
 *   sample is an empty column.  The pairs get their EC ids, the LSD radix sort orders them by (sample, EC id) and the
 *   scan of the pairs per sample gives n_indptr.  Results are delivered as by ecb_finalize (pinned, pageable or on
 *   the device, valid until the next finalize/reset/destroy).  Fails with ECB_ERR_INVALID when alignments were
 *   pushed after the last close, with ECB_ERR_LIMIT for more than 2^31 - 1 entries of N, and with ECB_ERR_EMPTY when
 *   no sample holds a read.  ecb_finalize still gives the one-sample result of everything pushed.
 * Both refuse contexts created with cells (ECB_ERR_INVALID).  ecb_reset forgets the samples.  Device memory: 4 bytes
 * per EC for the counts at the last close and 8 bytes per pair; during ecb_finalize_samples the sort adds 24 bytes
 * per pair and its histograms. */
int ecb_sample_close(ecb_ctx* ctx, int64_t* nonzeros);
int ecb_finalize_samples(ecb_ctx* ctx, ecb_result* out);

/* ---- ECs given as the rows of EC files (since version 2007) ---------------------------------------------------
 * A merge of EC files feeds each file's A rows and N columns into one single-sample context instead of reads, and
 * takes the result from ecb_finalize_samples: for every file, ecb_push_ecs, then ecb_sample_append.  EC ids are ranks
 * of first occurrence, so the merged ids follow (file, row id in that file), and the merge of the convert() outputs of
 * several BAM files is what the samples of those files give.
 *
 * ecb_push_ecs: the n_ec rows of one EC file's A matrix (CSR: a_indptr[n_ec + 1], a_indices = main targets ascending
 *   inside a row, a_data = haplotype masks) as ECs of this context.  Row e's key is the set hash of its (target,
 *   haplotype) elements: the key ecb_push gives a read with that set.  Its first occurrence is order_base + e, counted,
 *   as ecb_push counts after a close, from the end of the closed samples' range.  A new key claims an EC that holds the
 *   row; a known key is compared element for element with the row its EC holds.  No read is counted.
 *   The host checks a_indptr (0 to nnz, rising, no empty row; copied back first when it is device memory) before any
 *   kernel reads it; one pass over the entries then checks the values (target in [0, n_targets), targets strictly
 *   ascending in a row, mask not 0 and below 1 << n_haps) and sums the keys, and its flags come back before anything
 *   is inserted: a malformed file leaves the context as it was (ECB_ERR_FORMAT, naming the kind and the first bad
 *   entry and its row).  After the insert, two rows of one push with one set fail with ECB_ERR_FORMAT, and a row whose
 *   key an EC with a different row holds (a 128-bit key collision, never merged) with ECB_ERR_LIMIT; after either,
 *   every call but ecb_reset / ecb_destroy fails with ECB_ERR_STATE.  The table grows before the insert, so that it is
 *   at most half full after it.  Refused (ECB_ERR_STATE) when alignments were pushed after the last ecb_sample_close.
 * ecb_sample_append: n_samples samples given as columns (CSC: n_indptr[n_samples + 1], n_indices = row ids of the
 *   LAST ecb_push_ecs, n_data = counts), closed at once: entry i adds (EC of row n_indices[i], n_data[i]) to the samples'
 *   pair list, which ecb_finalize_samples sorts into N.  Zeros are dropped; a row index outside the last push or a
 *   negative count fails with ECB_ERR_FORMAT, before anything is added.  *nonzeros = pairs added.  One pass over the
 *   entries, one scan and one host round trip, whatever the number of columns.  Later ecb_push / ecb_push_ecs order
 *   keys count from the end of the pushed rows.
 * Between the two calls the rows are open input: ecb_push, ecb_sample_close (ECB_ERR_STATE) and ecb_finalize_samples
 * (ECB_ERR_INVALID) refuse.  A later ecb_push_ecs replaces rows that were not appended (their ECs stay, without
 * counts, and the later rows follow them in the order).  ecb_finalize refuses a context that received EC rows, and so does the multi-GPU exchange (ECB_ERR_STATE):
 * they carry no reads.  Both refuse contexts created with cells (ECB_ERR_INVALID).  ecb_reset forgets everything.
 * Host arrays are copied with one cudaMemcpyAsync each.  Device memory: 28 bytes per row of the largest push and 12 per
 * A entry (staging of host arrays; 8 of them stay in the row arena for a new row); per N entry 4 bytes of flags and 8
 * bytes in the pair list, plus 8 of staging for host arrays. */
int ecb_push_ecs(ecb_ctx* ctx, const int32_t* a_indptr, const int32_t* a_indices, const int32_t* a_data,
                 int64_t n_ec, int64_t nnz, int64_t order_base, int on_device);
int ecb_sample_append(ecb_ctx* ctx, const int32_t* n_indptr, const int32_t* n_indices, const int32_t* n_data,
                      int64_t n_samples, int64_t nnz, int on_device, int64_t* nonzeros);

/* Forget all pushed data but keep allocations (tables, staging) for the next job. */
int ecb_reset(ecb_ctx* ctx);

int ecb_get_stats(const ecb_ctx* ctx, ecb_stats* out);

int ecb_destroy(ecb_ctx* ctx);

/* Message of the last failing call on this context (or of ecb_create when ctx is NULL). */
const char* ecb_last_error(const ecb_ctx* ctx);

/* ---- multi-GPU exchange -------------------------------------------------------------------------
 * Reads shard across GPUs by contiguous chunk (alntools/utils.py:67-87 + bam_utils.py:647-680: each
 * worker gets a contiguous run of chunks and results are merged in chunk order).  Each rank pushes its
 * shard into a LOCAL context with order_base = global offset of the shard, or counted from its own first
 * alignment and moved there with ecb_rebase.  The merge of alntools/bam_utils.py:680-698 (counts of equal
 * keys summed, EC id = rank of the first occurrence over all shards) is the exchange over peer memory
 * further down; it leaves the final matrices partitioned, one contiguous EC-id range per rank.
 */
/* Add `delta` (>= 0) to the order key of everything pushed so far: a rank that decodes one shard of a file
 * pushes with order_base counted from its own first alignment and is moved to its global position once every
 * rank knows how many alignments the shards in front of it hold.  Single-sample contexts, before the exchange. */
int ecb_rebase(ecb_ctx* ctx, int64_t delta);

/* ---- the exchange over peer memory (one process per GPU on an NVLink / NVSwitch box) --------------------
 * Each rank creates an ARENA on its OWNER context (device memory from cudaMalloc, exportable through CUDA IPC),
 * hands the 64-byte IPC handle to its peers and maps theirs.  Two dispatches of fixed-size records go through
 * it, each one kernel that stores straight into the destination ranks' arenas over NVLink (one remote
 * atomicAdd per CTA tile and destination reserves the space):
 *   ecb_export_to_arenas (LOCAL context)   every local EC as {key, first, count} to its owner rank (hash of the
 *                                          key);
 *   ecb_import_arena     (OWNER context)   the owner merges what arrived: counts summed, smallest first
 *                                          occurrence kept (alntools/bam_utils.py:693-698);
 *   ecb_order_dispatch   (OWNER context)   every merged EC as {key, position inside the shard, count} to the rank
 *                                          whose shard [shard_lo[r], shard_hi[r]) of the global read order holds
 *                                          its first occurrence;
 *   ecb_order_build      (OWNER + LOCAL)   EC ids are ranks of first-occurrence positions and the shards
 *                                          partition the positions, so what arrived is one contiguous id range:
 *                                          it is ordered with a bitmap over this rank's OWN positions and the
 *                                          rows are taken from the LOCAL context - the rank that holds an EC's
 *                                          first occurrence has met the EC in its own reads.  Rows never travel;
 *                                          nothing global is built (no bitmap over all positions, no
 *                                          all-reduce).  id_base of the result is left 0: the slice starts after
 *                                          the ECs of the shards in front, which the caller learns from one
 *                                          all-gather of the slice sizes.
 * The caller brackets the stores with barriers:
 *     ecb_arena_reset (every rank) - barrier - ecb_export_to_arenas - barrier - ecb_import_arena -
 *     ecb_arena_reset - barrier - ecb_order_dispatch - barrier - ecb_order_build.
 * On a caller-provided stream (ecb_set_stream) reset, export and dispatch are stream-ordered and the barriers
 * are collectives on that stream (the host does not wait); a context on its own stream synchronises in each.
 * arena_bases[r] = base address of rank r's arena as seen from THIS process (own base for r == rank);
 * cap_records = records (of 32 bytes) every arena can take. */
int ecb_arena_create(ecb_ctx* owner_ctx, int64_t cap_records, void* ipc_handle_out /* 64 bytes */, void** base_out);
int ecb_arena_open_peer(ecb_ctx* owner_ctx, const void* ipc_handle /* 64 bytes */, void** base_out);
int ecb_arena_reset(ecb_ctx* owner_ctx);
int ecb_export_to_arenas(ecb_ctx* local_ctx, int world, void* const* arena_bases, int64_t cap_records,
                         int64_t* min_base, int64_t* max_end);
int ecb_import_arena(ecb_ctx* owner_ctx);

/* This rank's slice of the final matrices: a_indptr[n_ec + 1] (offsets local to the slice), a_indices, a_data
 * and n_data (read counts), all device memory of the owner context, valid until the next call on it.
 * Besides bad arguments and CUDA errors, ecb_order_build fails, before any row is copied, with
 *   ECB_ERR_LIMIT    "exchange arena too small for the second dispatch", a shard of more than 2^32 positions, or a
 *                    slice beyond the int32 fields of the EC file;
 *   ECB_ERR_INVALID  more ECs arrived than the shard has positions or the local context holds ECs, or "second
 *                    dispatch: ..." - an EC the local context has never seen, two ECs with one first position
 *                    (order_base ranges of one rank's pushes overlapped), or a record outside the shard.
 * The owner and the local context stay usable. */
typedef struct ecb_slice {
  int64_t id_base, n_ec, nnz;
  const int32_t *a_indptr, *a_indices, *a_data, *n_data;
} ecb_slice;
int ecb_order_dispatch(ecb_ctx* owner_ctx, int world, void* const* arena_bases, int64_t cap_records,
                       const int64_t* shard_lo, const int64_t* shard_hi);
int ecb_order_build(ecb_ctx* owner_ctx, const ecb_ctx* local_ctx, int64_t shard_lo, int64_t shard_hi, ecb_slice* out);

/* ---- the per-cell exchange (contexts created with cells; since version 2001) ----------------------------
 * The same two dispatches, with (EC, cell) pairs travelling beside the ECs.  Every rank pushes its own files,
 * one push per file with drop_last_group = 1, at RANK-MAJOR order keys: order_base = rank * 2^40 + (alignments
 * of this rank's earlier files).  So every position of a rank lies behind those of all ranks in front of it, no
 * count is exchanged before the pushes, no rebase is needed, and a rank's positions still span less than 2^32.
 * Cells carry GLOBAL ids: the first appearance over the ranks' cell-name lists taken in rank order (the id the
 * one-GPU build gives); cell_map[local id] = global id (device int32, NULL = identity).  Sequence, per rank:
 *   ecb_cells_summary        (LOCAL)  cell_key[g] = this rank's sort key of global cell g (~0 if absent),
 *                                     cell_total[g] = its reads here (device uint64 arrays of n_cells);
 *   caller: all-gather the keys as [world x n_cells], all-reduce the totals with SUM;
 *   ecb_cells_order          (LOCAL)  every rank takes the same decision: a cell's key is (first rank that
 *                                     holds it, that rank's key); cells below min_cell_count (<= 0: 1) are
 *                                     dropped.  -> n_samples (kept cells, ECB_ERR_EMPTY when none, the same on
 *                                     every rank) and cell_order (device, global cell id of every column, valid
 *                                     until the next call on the context);
 *   ecb_cells_dispatch_counts         exact records per destination rank of the next dispatch: counts[r] ECs,
 *                                     counts[world + r] pairs (device int64 [2 * world], written on the
 *                                     context's stream).  shard_lo / shard_hi NULL: dispatch 1 (LOCAL context,
 *                                     after ecb_cells_order); given: dispatch 2 (OWNER, after the import).  The
 *                                     caller all-reduces them and sizes the arenas from the largest;
 *   ecb_cells_arena_create   (OWNER)  one IPC allocation with two record areas (cap_ec EC records, cap_pairs
 *                                     pair records), each with its own header; replaces a smaller arena of an
 *                                     earlier call, closing the peer arenas opened through ecb_arena_open_peer
 *                                     (the caller exchanges the new handles).  ecb_arena_reset clears both
 *                                     headers;
 *   ecb_cells_export_to_arenas (LOCAL) every local EC as {key, first, reads in kept cells} - ECs without such
 *                                     reads too: this rank may hold the EC's first occurrence - and every local
 *                                     (EC, cell) pair with a kept column as {EC key, column, count} to the owner;
 *   ecb_cells_import_arena   (OWNER)  ECs merged as by ecb_import_arena, pairs merged by (EC, column);
 *   ecb_cells_order_dispatch (OWNER)  merged ECs with reads in kept cells, and every merged pair, to the rank
 *                                     whose shard holds the EC's first occurrence;
 *   ecb_cells_order_build    (OWNER + LOCAL) the A slice as ecb_order_build, and the slice's N entries.
 * Barriers as in the single-sample exchange.  cap_ec / cap_pairs are the same on every rank.  An arena that
 * turns out too small sets its overflow flag; import and build then fail with ECB_ERR_LIMIT. */
int ecb_cells_summary(ecb_ctx* local_ctx, const int32_t* cell_map, int64_t map_len, int64_t n_cells, uint64_t* cell_key,
                      uint64_t* cell_total);
int ecb_cells_order(ecb_ctx* local_ctx, int world, const uint64_t* cell_keys, const uint64_t* cell_totals, int64_t n_cells,
                    int64_t min_cell_count, const int32_t* cell_map, int64_t* n_samples, const int32_t** cell_order);
int ecb_cells_dispatch_counts(ecb_ctx* ctx, int world, const int64_t* shard_lo, const int64_t* shard_hi, int64_t* counts);
int ecb_cells_arena_create(ecb_ctx* owner_ctx, int64_t cap_ec, int64_t cap_pairs, void* ipc_handle_out /* 64 bytes */,
                           void** base_out);
int ecb_cells_export_to_arenas(ecb_ctx* local_ctx, int world, void* const* arena_bases, int64_t cap_ec, int64_t cap_pairs,
                               int64_t* min_base, int64_t* max_end);
int ecb_cells_import_arena(ecb_ctx* owner_ctx);
int ecb_cells_order_dispatch(ecb_ctx* owner_ctx, int world, void* const* arena_bases, int64_t cap_ec, int64_t cap_pairs,
                             const int64_t* shard_lo, const int64_t* shard_hi);

/* This rank's slice of the per-cell matrices: the A part as ecb_slice; N as the slice's entries in column-major
 * order - n_col_counts[n_samples] entries per column, n_indices (EC ids local to the slice, ascending inside a
 * column), n_data (counts).  Device memory of the owner context, valid until the next call on it. */
typedef struct ecb_cells_slice {
  int64_t n_ec, nnz;
  const int32_t *a_indptr, *a_indices, *a_data;
  int64_t n_samples, nnz_n;
  const int32_t *n_col_counts, *n_indices, *n_data;
} ecb_cells_slice;
int ecb_cells_order_build(ecb_ctx* owner_ctx, const ecb_ctx* local_ctx, int64_t shard_lo, int64_t shard_hi, int64_t n_samples,
                          ecb_cells_slice* out);

/* ---- device decode of single-sample BAM files (since version 2002) ------------------------------------------
 * The GPU form of libbamcols' single-sample path (include/bamcols.h): BGZF inflate, the record hop, the filters of
 * alntools/bam_utils.py:264-270, name trimming (:301-304) and the name-change test (:306), producing in device
 * memory the columns bamcols_emit produces, ready for ecb_push(..., on_device = 1).  A decoder is bound to one
 * context and uses its device, stream and memory pool; destroy it before the context.  A decoder that has
 * failed refuses further calls: create a fresh one (after ecb_reset when the context's pushes are abandoned).
 *
 * ecb_bam_create: tid_target / tid_hap[n_references] as for bamcols_set_tables (copied); track_ranges = 1
 * records the smallest and largest pos of the valid alignments of every reference (--rangefile).
 *
 * ecb_bam_decode: one call per run of whole BGZF blocks, in file order.
 *   bytes[n_bytes]      compressed bytes on the host (pinned preferred), copied to the device
 *   block_off[i]        offset in bytes of block i's raw DEFLATE payload, block_len[i] its length,
 *   block_isize[i]      its inflated size (ISIZE; at most 65 536, larger blocks are refused with ECB_ERR_FORMAT)
 *                       - the table bamcols_blocks lists
 *   skip                inflated bytes of the first block before the first record (the low 16 bits of the first
 *                       record's virtual offset); 0 after the first call
 *   last                1 on the final call: the last read is closed, and bytes left after the last whole record
 *                       are a truncated record
 * Returns DEVICE pointers to the rows of every read closed by this call (valid until the next call on the decoder);
 * read_group continues from call to call as bamcols_emit's does.  The blocks are inflated in windows of
 * ECB_OPT_BAM_WINDOW bytes; records and reads may span blocks, windows and calls.  Corrupt blocks, truncated
 * records, block_size < 32 and bad read-name lengths fail with ECB_ERR_FORMAT, and so does a valid alignment whose
 * refID lies outside the header (with its own message). */
typedef struct ecb_bam ecb_bam;
typedef struct ecb_bam_stats {
  int64_t h2d_bytes;       /* compressed bytes copied host->device                                            */
  int64_t inflated_bytes;
  int64_t blocks;
  int64_t windows;
  int64_t hop_rounds;      /* join rounds of the record hop (1 per window when every segment guessed right)     */
  int64_t records;         /* = all_alignments                                                                 */
  double h2d_ms;           /* stream time between CUDA events around each phase, summed over the calls: the  */
  double inflate_ms;       /* hop and rules phases include the host round trips of their count read-backs    */
  double hop_ms;
  double rules_ms;
} ecb_bam_stats;
int ecb_bam_create(ecb_ctx* ctx, const int32_t* tid_target, const int32_t* tid_hap, int32_t n_references,
                   int track_ranges, ecb_bam** out);
int ecb_bam_decode(ecb_bam* d, const uint8_t* bytes, int64_t n_bytes, const int64_t* block_off, const int32_t* block_len,
                   const int32_t* block_isize, int64_t n_blocks, int64_t skip, int last, const int32_t** read_group,
                   const int32_t** target_idx, const int32_t** hap_idx, int64_t* rows);
/* records seen so far (valid or not) and reads started */
int ecb_bam_counters(const ecb_bam* d, int64_t* all_alignments, int64_t* n_groups);
/* host int32[n_references] each; min > max where no valid alignment was seen (as bamcols_ranges) */
int ecb_bam_ranges(ecb_bam* d, int32_t* range_min, int32_t* range_max);
int ecb_bam_get_stats(const ecb_bam* d, ecb_bam_stats* out);
int ecb_bam_destroy(ecb_bam* d);

/* ---- device parse of single-sample SAM text (since version 2008) -------------------------------------------------
 * SAM text in, the columns ecb_bam_decode gives for the BAM file that holds the same alignments out, in device memory,
 * ready for ecb_push(..., on_device = 1): lines found and QNAME, FLAG, RNAME, POS, RNEXT and PNEXT parsed on the GPU,
 * then the filters, name trimming and the name-change test of the BAM decoder.  A decoder is bound to one context and
 * uses its device, stream and memory pool; destroy it before the context.  A decoder that has failed refuses further
 * calls.
 *
 * ecb_sam_create: the @SQ names of the header, in order: name t is ref_names[ref_name_off[t], ref_name_off[t + 1])
 *   (not NUL-terminated; ref_name_off[0] = 0); tid_target / tid_hap[n_references] as for ecb_bam_create (copied).  The
 *   names go into a device hash table (the first of two equal names wins).  first_line: the line number of the first
 *   byte the first call gives (the header's line count + 1), for error messages.  track_ranges as for ecb_bam_create.
 * ecb_sam_parse: one call per run of whole alignment lines (every line ends in '\n', except possibly the last line of
 *   the `last` call), at most 2 GiB, in input order; the text is copied with one host-to-device copy (pinned host
 *   memory preferred).  Returns DEVICE pointers to the rows of every read closed by this call (valid until the next
 *   call); read_group continues from call to call as ecb_bam_decode's does, and reads may span calls.  A bad line fails
 *   with ECB_ERR_FORMAT and a message "line N: <what>" for the first bad line of the call: a line starting with '@',
 *   fewer than 11 tab-separated fields, QNAME empty or longer than 254 bytes, FLAG not a decimal in [0, 65535], POS or
 *   PNEXT not a decimal in [0, 2^31 - 1], RNAME not '*' or an @SQ name, RNEXT not '*', '=' or an @SQ name, or a valid
 *   alignment whose RNAME is '*'.  MAPQ, CIGAR, TLEN, SEQ, QUAL and tags are not looked at. */
typedef struct ecb_sam ecb_sam;
typedef struct ecb_sam_stats {
  int64_t bytes;           /* text bytes copied host->device                                                  */
  int64_t lines;           /* alignment lines parsed (= all_alignments)                                       */
  int64_t calls;
  double h2d_ms;           /* stream time between CUDA events around each phase, summed over the calls: the   */
  double lines_ms;         /* lines and fields phases include the host round trips of their count read-backs  */
  double fields_ms;
  double rules_ms;
} ecb_sam_stats;
int ecb_sam_create(ecb_ctx* ctx, const char* ref_names, const int64_t* ref_name_off, int32_t n_references,
                   const int32_t* tid_target, const int32_t* tid_hap, int64_t first_line, int track_ranges, ecb_sam** out);
int ecb_sam_parse(ecb_sam* d, const uint8_t* text, int64_t n_bytes, int last, const int32_t** read_group,
                  const int32_t** target_idx, const int32_t** hap_idx, int64_t* rows);
/* alignment lines seen so far (valid or not) and reads started */
int ecb_sam_counters(const ecb_sam* d, int64_t* all_alignments, int64_t* n_groups);
/* host int32[n_references] each; min > max where no valid alignment was seen */
int ecb_sam_ranges(ecb_sam* d, int32_t* range_min, int32_t* range_max);
int ecb_sam_get_stats(const ecb_sam* d, ecb_sam_stats* out);
int ecb_sam_destroy(ecb_sam* d);

/* ---- collation of alignments by read name (since version 2003) ----------------------------------------------
 * For files that are not grouped by read name.  A read is the set of valid alignments that share a trimmed name,
 * wherever they lie in the file; reads are ordered by their first alignment.  The result equals ecb_push of the same
 * alignments regrouped that way (each read contiguous, reads in that order).  A collator is bound to one
 * single-sample context and uses its device, stream and memory pool; destroy it before the context.
 *
 * ecb_collate_add: append n alignments in file order - the rows of bamcols_emit_keys (include/bamcols.h): 128-bit
 *   name key (never all ones), target_idx, hap_idx.  on_device 0: host pointers (pinned preferred), 1: device
 *   pointers of the context's device.  Copied; the buffers may be reused after return.  Fewer than 2^32 - 1
 *   alignments in all.  Two names with equal keys are one read (DESIGN.md section 6.2).
 * ecb_collate_push: regroup everything added in device memory and push it into the context (ecb_push with
 *   on_device = 1, order_base = offset in collated order, in pieces of at most ECB_OPT_COLLATE_PIECE alignments that
 *   end at read ends; a longer read is a piece of its own).  Once per collator; *n_reads = reads formed.  The
 *   context's limits apply: a read of more than ECB_OPT_MAX_READ alignments fails with ECB_ERR_LIMIT.
 * Device memory: while the one-pass collation of the alignments added so far fits the budget (ECB_OPT_COLLATE_BUDGET;
 * 88 to 144 bytes per alignment with the automatic table, DESIGN.md section 6.2), the rows stay on the device as above.
 * An add that would pass it spills: the rows go to host memory (28 bytes per alignment), partitioned into 4096 buckets
 * by name key, and from then on the collator holds a fixed staging area.  The push then works in passes over groups of
 * buckets (names), once over all reads (order), over chunks of rows (layout) and over pieces (push), each within the
 * budget.  The outputs do not depend on the budget.  A budget that cannot hold the staging area, the bitmap over all
 * alignments with the per-read counts and offsets (n/4 + 8 bytes per read), or one bucket's names pass fails with
 * ECB_ERR_LIMIT and a message naming the budget; so does a ECB_OPT_COLLATE_PIECE that cuts a spilled collation into
 * more than 4096 pieces.  A piece holds at least one read, and a name table that runs out of probes grows, so those
 * two may pass the budget by what they need; with ECB_OPT_MAX_READ raised, one long read can pass it by its own
 * rows and the long-read pass of its push.  Running out of device memory otherwise fails with ECB_ERR_CUDA and the
 * allocator's message. */
typedef struct ecb_collate ecb_collate;
typedef struct ecb_collate_stats {
  int64_t alignments;      /* added                                                                            */
  int64_t reads;           /* reads formed (after the push)                                                    */
  int64_t table_slots;     /* name table slots at the end                                                      */
  int64_t table_grows;     /* times the name table was replaced by a larger one                                */
  int64_t pieces;          /* pushes into the context                                                          */
  int64_t device_bytes;    /* peak device memory held by the collator                                          */
  int64_t h2d_bytes;       /* bytes copied host->device: the add calls, and after a spill the passes           */
  double add_ms;           /* stream time of the add copies (and the spills inside them), summed               */
  double table_ms;         /* name table, growth included                                                      */
  double order_ms;         /* bitmap, ranks, read ids and offsets (with one host round trip)                   */
  double layout_ms;        /* scatter to collated order and the piece cuts (with one host round trip)          */
  double push_ms;          /* the pushes into the context                                                      */
  /* since version 2004; after a spill table_ms, order_ms, layout_ms and push_ms time the four passes */
  int64_t spills;          /* times the staging area went to host memory (0: the one-pass collation ran)       */
  int64_t groups;          /* groups of name buckets of the names pass                                         */
  int64_t host_bytes;      /* peak host memory holding spilled rows                                            */
  int64_t d2h_bytes;       /* bytes copied device->host                                                        */
  double spill_ms;         /* wall time of the spills, summed                                                  */
} ecb_collate_stats;
int ecb_collate_create(ecb_ctx* ctx, ecb_collate** out);
int ecb_collate_add(ecb_collate* c, const uint64_t* key_lo, const uint64_t* key_hi, const int32_t* target_idx,
                    const int32_t* hap_idx, int64_t n, int on_device);
int ecb_collate_push(ecb_collate* c, int64_t* n_reads);
int ecb_collate_get_stats(const ecb_collate* c, ecb_collate_stats* out);
int ecb_collate_destroy(ecb_collate* c);

#ifdef __cplusplus
}
#endif
#endif /* ECB200_H */
