/*
 * bamcols.h — C ABI of libbamcols.so: the host column emitter in front of libecb200.
 *
 * What it replaces: the per-alignment front half of alntools/bam_utils.py:253-306
 * (process_convert_bam: iterate pysam records, skip unmapped / unusable paired-end alignments
 * :264-270, trim the read name at the first blank :301-304, start a new read when the name changes
 * :306) and of alntools/bam_utils_multisample.py:209-300 (same loop; the cell id is field 14 of the
 * '|||'-split name of the read :270-280, the remembered name is left untrimmed after the first
 * switch :292).  pysam/htslib do the BGZF/BAM decode for the reference; here the decode is part of
 * this library (zlib inflate of BGZF blocks on a thread pool, then one pass over the fixed-offset
 * record fields refID, flag, next_refID, next_pos, l_read_name, read_name).
 *
 * Output: int32 columns, one row per VALID alignment, written into caller-owned (ideally pinned)
 * buffers — exactly what ecb_push (include/ecb200.h) takes:
 *     read_group  non-decreasing, +1 whenever the reference would start a new read
 *     target_idx  tid_target[refID]      hap_idx  tid_hap[refID]
 *     cell_idx    (per-cell mode) dense id of the cell name, shared by all files of a job
 *
 * All functions return 0 / a count on success and a negative bamcols_status on failure; the message
 * is available through bamcols_last_error().  A reader is not thread-safe; it runs its own worker
 * threads for the inflate step.
 */
#ifndef BAMCOLS_H
#define BAMCOLS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bamcols bamcols;
typedef struct bamcols_cells bamcols_cells;

enum bamcols_status {
  BAMCOLS_OK = 0,
  BAMCOLS_ERR_IO = -1,       /* open/read/mmap failure */
  BAMCOLS_ERR_FORMAT = -2,   /* not BGZF / not BAM / truncated / corrupt block */
  BAMCOLS_ERR_INVALID = -3,  /* bad argument or call sequence */
  BAMCOLS_ERR_CELL_FIELD = -4, /* per-cell mode: a read name has fewer than 15 '|||' fields (the
                                  reference raises IndexError at bam_utils_multisample.py:273) */
  BAMCOLS_ERR_TID = -5       /* a valid alignment's refID is outside the header's reference list */
};

/* Open a BAM file and parse its header.  n_threads <= 0: one inflate worker per hardware thread. */
int bamcols_open(bamcols** out, const char* path, int n_threads);
void bamcols_close(bamcols* r);
const char* bamcols_last_error(const bamcols* r); /* r == NULL: error of the last failed open */

/* Header: references in @SQ order (= tid order), as pysam's .references / .lengths. */
int bamcols_n_references(const bamcols* r);
const char* bamcols_reference_name(const bamcols* r, int tid);
int bamcols_reference_length(const bamcols* r, int tid);
/* All names at once: *names = every name followed by a NUL, in tid order; *lengths = int32[n_references];
 * returns the byte length of *names.  The pointers stay valid until bamcols_close. */
int64_t bamcols_reference_blob(const bamcols* r, const char** names, const int32_t** lengths);

/* tid -> (main-target index, haplotype index) lookups built by the host from the header
 * (alntools/bam_utils.py:561-633).  Copied. */
int bamcols_set_tables(bamcols* r, const int32_t* tid_target, const int32_t* tid_hap, int n_references);

/* The same tables built natively (alntools/bam_utils.py:561-633): main targets = target-file ids first
 * (first_targets: each id followed by a NUL; may be empty), then unseen targets in header order; a name is
 * split at its LAST '_' unless that is its first character; haplotypes sorted; lengths[target][hap].
 * Installs the tid lookups (no bamcols_set_tables needed).  Two @SQ names that collapse to the same
 * (target, haplotype) are refused.  bamcols_tables hands the results out (names as NUL-separated blobs). */
int bamcols_build_tables(bamcols* r, const char* first_targets, int64_t first_len);
int bamcols_tables(const bamcols* r, int32_t* n_targets, int32_t* n_haps, const char** targets, int64_t* targets_len,
                   const char** haps, int64_t* haps_len, const int32_t** tid_target, const int32_t** tid_hap,
                   const int32_t** lengths);
/* The targets section of the EC file, T x [len(name), name bytes, H x length] as little-endian int32s
 * (alntools/bin_utils.py:153-159), from the tables of bamcols_build_tables.  Returns the number of bytes (the
 * buffer belongs to the reader), or 0 when a target name is not ASCII: the reference writes the length in
 * characters there and the caller has to reproduce that from the decoded names. */
int64_t bamcols_target_section(bamcols* r, const char** bytes);

/* Cell-name dictionary of one per-cell job: names get dense ids in order of first appearance. */
int bamcols_cells_create(bamcols_cells** out);
void bamcols_cells_destroy(bamcols_cells* c);
int64_t bamcols_cells_count(const bamcols_cells* c);
const char* bamcols_cells_name(const bamcols_cells* c, int64_t idx);

/* Decode on and write up to `capacity` rows.  Returns the number of rows written (>= 0).
 * Only whole reads are returned (a read is never split between two calls) except that a read longer
 * than `capacity` is an error; *done is set to 1 once the file is exhausted (the last call may
 * return 0 rows).  read_group continues from call to call.  cells == NULL selects the single-sample
 * rules, otherwise the per-cell rules apply and cell_idx must be non-NULL. */
int64_t bamcols_emit(bamcols* r, bamcols_cells* cells, int32_t* read_group, int32_t* target_idx, int32_t* hap_idx,
                     int32_t* cell_idx, int64_t capacity, int* done);

/* The rows of collation (ecb_collate_add in include/ecb200.h): one row per VALID alignment in file order, with the
 * filters, errors, all_alignments counter and --rangefile tracking of the single-sample rules, but no read_group:
 *     key_lo, key_hi  128-bit key of the read name trimmed at its first blank unless that blank is its first
 *                     character (alntools/bam_utils.py:301-304); equal names give equal keys, and no key is all
 *                     ones (the device table's empty slot)
 *     target_idx, hap_idx  as for bamcols_emit
 * Up to `capacity` rows per call; a call may end anywhere, since reads are formed later over the whole file.  *done
 * is set once the file is exhausted.  A reader that has used bamcols_emit refuses this call, and the other way round. */
int64_t bamcols_emit_keys(bamcols* r, uint64_t* key_lo, uint64_t* key_hi, int32_t* target_idx, int32_t* hap_idx,
                          int64_t capacity, int* done);

/* Shards of ONE file for several readers (one per GPU / process), without temporary files.  The reference plans
 * chunks as BGZF virtual offsets at read boundaries (alntools/bam_utils.py:1174-1304) and then copies every
 * chunk into its own temporary BAM (:157-195); here every reader opens the same file and confines itself to
 * its range.  bamcols_plan_shards: voffsets[n_shards + 1], voffsets[k] = virtual offset (compressed offset of
 * a block << 16 | offset inside the inflated block) of the first record of shard k - a record whose trimmed
 * name differs from its predecessor's, at or behind k/n of the compressed bytes; voffsets[0] = first record of
 * the file, voffsets[n_shards] = -1 (end of file); -1 also marks an empty shard at the end.  The plan depends
 * on the file only, so every process computes the same one.  bamcols_set_range (before the first
 * bamcols_emit): the reader emits the records of [vbegin, vend) only (vend = -1: to the end of the file). */
int bamcols_plan_shards(bamcols* r, int n_shards, int64_t* voffsets);
int bamcols_set_range(bamcols* r, int64_t vbegin, int64_t vend);

/* The BGZF blocks from compressed offset c_begin on, without inflating them (the block table of the device decoder,
 * ecb_bam_decode in include/ecb200.h): at most max_blocks blocks whose compressed bytes fit in max_bytes - at least
 * one block whenever one is left.  payload_off[i] = offset of block i's raw DEFLATE payload counted from c_begin,
 * payload_len[i] its length, isize[i] its inflated size; *c_end = offset behind the last listed block.  Returns the
 * number of blocks (0 at the end of the file) or BAMCOLS_ERR_FORMAT with the messages of the reader. */
int64_t bamcols_blocks(bamcols* r, int64_t c_begin, int64_t max_bytes, int64_t max_blocks, int64_t* payload_off,
                       int32_t* payload_len, int32_t* isize, int64_t* c_end);

/* Counters so far: records seen (valid or not) and reads started. */
int64_t bamcols_all_alignments(const bamcols* r);
int64_t bamcols_n_groups(const bamcols* r);

/* --rangefile support (alntools/bam_utils.py:282-286): record the smallest and largest reference_start
 * of the valid alignments of every reference.  Enable before the first bamcols_emit; bamcols_ranges
 * returns n_references and two int32[n_references] arrays (min > max: no valid alignment). */
int bamcols_track_ranges(bamcols* r, int enable);
int bamcols_ranges(const bamcols* r, const int32_t** min_pos, const int32_t** max_pos);

/* Wall-clock seconds spent so far per phase: inflate, record hop, validity, read starts, row write,
 * copy-out (single-sample path; diagnostics for the host-side timing report). */
int bamcols_phase_seconds(const bamcols* r, double* out6);

/* The block decoder on its own (tests, timing): inflate a raw DEFLATE stream whose inflated size is known,
 * as every BGZF block is.  mode 0 = as the reader does it (whole-buffer decoder, zlib for anything it
 * declines), 1 = zlib only, 2 = whole-buffer decoder only.  Returns 1 if exactly dst_len bytes were
 * produced from a well-formed stream, 0 if not, < 0 on bad arguments. */
int bamcols_inflate_raw(const uint8_t* src, int64_t src_len, uint8_t* dst, int64_t dst_len, int mode);

#ifdef __cplusplus
}
#endif
#endif /* BAMCOLS_H */
