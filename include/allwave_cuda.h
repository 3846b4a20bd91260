/*
 * allwave_cuda.h -- C ABI of liballwave_cuda.so: the B200 (sm_100a) drop-in for allwave's
 * alignment hot path.  Plain pointers and sizes only; no C++/torch types cross this boundary.
 *
 * What it replaces in the reference (/root/reference):
 *   - the per-pair call chain  AllPairParallelIterator -> align_pair -> lib_wfa2
 *     (src/iterator.rs:182-252, src/alignment.rs:25-66, :201-261)       => aw_align_pairs / aw_batch_*
 *   - lib_wfa2::affine_wavefront::AffineWavefronts {with_penalties_and_memory_mode,
 *     with_penalties_affine2p_and_memory_mode, set_alignment_scope, set_alignment_span,
 *     set_heuristic, align, score, cigar}  (call sites src/alignment.rs:226-236,263-289,
 *     src/wfa.rs:188-231)                                              => aw_aligner_*
 *   - determine_orientation_mash / sketch_sequence_stranded / jaccard_similarity
 *     (src/alignment.rs:69-139)                                         => done inside aw_align_pairs,
 *                                                                          exposed by aw_orient_pairs
 *   - mash::compute_distance_matrix_with_params' sketches + Jaccard counts
 *     (src/mash.rs:78-107,40-56,141-165)                                => aw_mash_jaccard_counts
 *   - count_cigar_operations, parse_cigar_lengths, cigar_bytes_to_string, alignment_to_paf
 *     (src/alignment.rs:292-376, src/lib.rs:71-112)                     => fields of aw_result
 *
 * Every function returns 0 (AW_OK) or a negative aw_status; no exception or panic crosses the ABI.
 * There is NO CPU fallback: without a CUDA device every compute entry point returns AW_ENODEVICE.
 */
#ifndef ALLWAVE_CUDA_H
#define ALLWAVE_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AW_ABI_VERSION 1

typedef enum aw_status {
    AW_OK = 0,
    AW_EINVAL = -1,        /* bad argument */
    AW_ENODEVICE = -2,     /* no usable CUDA device / CUDA runtime error at init */
    AW_ECUDA = -3,         /* CUDA runtime error (see aw_last_error) */
    AW_ENOMEM = -4,        /* host or device allocation failed */
    AW_EUNSUPPORTED = -5,  /* e.g. match_score > 0, max_score_scope > 512 */
    AW_EWORKSPACE = -6,    /* internal per-pair status: device workspace too small, the pair is re-run by the retry ladder
                              (a pair that still fails after the ladder is delivered as AW_EALIGN + failure sentinel) */
    AW_ECALLBACK = -7,     /* the user callback returned non-zero; run cancelled */
    AW_EALIGN = -8         /* per-pair: alignment failed (mirrors AlignmentStatus != Completed) */
} aw_status;

/* mirrors AlignmentParams, src/types.rs:37-45 (max_divergence is unused by the path) */
typedef struct aw_params {
    int32_t match_score;
    int32_t mismatch_penalty;
    int32_t gap_open;
    int32_t gap_extend;
    int32_t gap2_open;       /* Some(..) iff has_gap2_open   */
    int32_t gap2_extend;     /* Some(..) iff has_gap2_extend */
    uint8_t has_gap2_open;
    uint8_t has_gap2_extend;
} aw_params;

/* one directed pair (query_idx, target_idx) of the list AllPairIterator builds, src/iterator.rs:40-46 */
typedef struct aw_pair {
    uint32_t query_idx;
    uint32_t target_idx;
} aw_pair;

/* how align_pair picks the strand, src/alignment.rs:35-39 */
typedef enum aw_orientation_mode {
    AW_ORIENT_MASH = 0,    /* determine_orientation_mash (CLI default)            */
    AW_ORIENT_WFA = 1,     /* determine_orientation_wfa (--wfa-orientation)       */
    AW_ORIENT_FORWARD = 2  /* no orientation step: query is used as given         */
} aw_orientation_mode;

/* mirrors AlignmentResult, src/types.rs:14-33, plus the strings the CLI derives from it */
typedef struct aw_result {
    uint64_t query_idx, target_idx;
    uint64_t query_start, query_end, target_start, target_end;
    uint8_t is_reverse;
    int32_t status;             /* AW_OK, or AW_EALIGN with the reference's failure sentinel filled in */
    int32_t score;              /* WFA2 convention: -(penalty); i32::MAX on failure                   */
    uint64_t num_matches, alignment_length;
    const uint8_t* cigar_bytes; /* WFA2 letters M X I D, one per column; NULL unless requested        */
    uint64_t cigar_len;
    const char* cg;             /* cigar_bytes_to_string: "12=1X3I..." (not NUL-terminated)           */
    uint64_t cg_len;
    const char* paf;            /* alignment_to_paf line without '\n' (not NUL-terminated)            */
    uint64_t paf_len;
} aw_result;

/* return non-zero to cancel the run (mirrors a callback Err, src/iterator.rs:235-251) */
typedef int (*aw_result_cb)(const aw_result* result, void* user);

typedef struct aw_ctx aw_ctx;
typedef struct aw_batch aw_batch;
typedef struct aw_aligner aw_aligner;

/* flags for aw_align_pairs / aw_batch_create */
#define AW_FLAG_CIGAR_BYTES 1u  /* also materialise expanded cigar_bytes                    */
#define AW_FLAG_ORDERED 2u      /* accepted, no effect: per-result callbacks are always delivered in pair order within a call */
#define AW_FLAG_NO_PAF 4u       /* skip PAF text (stats + cg only)                           */
#define AW_FLAG_PAF_BLOCKS 8u   /* aw_align_stream: every PAF line is followed by '\n' in the device text arena and whole
                                   batches are handed to the block callback (the CLI's writer, src/main.rs:347-367)   */
#define AW_FLAG_SCORE_ONLY 16u  /* the optimal score of each pair only (WFA2's score scope), without CIGAR or PAF; implies
                                   AW_FLAG_NO_PAF, and AW_EINVAL with AW_FLAG_CIGAR_BYTES or AW_FLAG_PAF_BLOCKS.  Per result:
                                   status, score, is_reverse and the indices as usual; query_start = target_start = 0 and
                                   query_end / target_end = the sequence lengths (End2End covers both); num_matches =
                                   alignment_length = 0; cigar_bytes, cg and paf are NULL with length 0.  A failed pair is
                                   AW_EALIGN with score INT32_MAX (no sentinel line).  aw_batch_stats [2..4] are 0.
                                   The biWFA recursion stops at its top level, whose breakpoint score is the optimal score. */

/* ---- library / device ---- */
int aw_abi_version(void);
const char* aw_strerror(int status);
const char* aw_last_error(void);            /* thread-local detail of the last failure */
int aw_device_count(void);                  /* 0 when no CUDA device is visible        */

/* ---- context: one per GPU (the path shards by pairs; no collective) ---- */
int aw_create(int device, aw_ctx** out);
void aw_destroy(aw_ctx* ctx);
/* tuning knobs; key is one of "ctas_per_sm", "threads_per_cta", "max_wavefront_width", "hist_mb", "chunk_pairs",
 * "ws16", "max_retry_attempts" (0 disables the retry ladder: pairs whose first-try workspace was too small fail) */
int aw_set_option(aw_ctx* ctx, const char* key, int64_t value);
/* returns every parked device / pinned buffer of the library's caching allocator to the driver */
void aw_trim_cache(void);

/* Copies the sequences (ASCII, any bytes) to the device, builds the reverse complements
 * (reverse_complement, src/alignment.rs:178-190), the 2-bit packing and validity flags.
 * ids are FASTA record ids (Sequence.id, src/types.rs:7-10); the caller may free everything
 * after return. */
int aw_load_sequences(aw_ctx* ctx, uint32_t n, const uint8_t* const* seqs, const uint64_t* lens,
                      const char* const* ids);
uint32_t aw_num_sequences(const aw_ctx* ctx);
/* penalties of the two orientation alignments of AW_ORIENT_WFA (AllPairIterator::with_orientation_params,
 * src/iterator.rs:95-98); default AlignmentParams::edit_distance() = 0,1,1,1 */
int aw_set_orientation_params(aw_ctx* ctx, const aw_params* params);

/* ---- the hot path, host-facing: align a pair list, stream results to a callback ---- */
int aw_align_pairs(aw_ctx* ctx, const aw_params* params, int orientation_mode, const aw_pair* pairs,
                   uint64_t npairs, uint32_t flags, aw_result_cb cb, void* user);

/* Streaming form of the same call (the parallel driver of src/iterator.rs:208-252 + the CLI's writer thread,
 * src/main.rs:347-374): the library PULLS chunks of the pair list from `next` (returns the number of pairs and sets
 * *pairs, valid until the following call; 0 ends the run) and keeps two batches in flight per context: while batch k+1
 * runs on the GPU, batch k is copied back on a second stream and delivered.  Several contexts (GPUs) can pull from one
 * shared source, which is how the host shards a pair list dynamically.  Delivery: `cb` per result (may be NULL), and/or
 * -- with AW_FLAG_PAF_BLOCKS -- `block_cb` with newline-terminated PAF text (`n_lines` lines, completion order).
 * A non-zero return of either callback cancels the run with AW_ECALLBACK. */
typedef uint64_t (*aw_chunk_source)(void* user, const aw_pair** pairs);
typedef int (*aw_paf_block_cb)(const char* text, uint64_t len, uint64_t n_lines, void* user);
int aw_align_stream(aw_ctx* ctx, const aw_params* params, int orientation_mode, uint32_t flags, aw_chunk_source next,
                    void* next_user, aw_result_cb cb, aw_paf_block_cb block_cb, void* user);

/* ---- the hot path, device-resident (what bench.py times as `value`) ----
 * create: uploads the pair list and sizes the workspace; launch: enqueues every kernel of the
 * path (orientation, biWFA, CIGAR/PAF emission) on `stream` (a cudaStream_t, NULL = the
 * context's own stream) without synchronising; fetch: synchronises, copies results D2H and
 * invokes cb.  A batch can be launched repeatedly. */
int aw_batch_create(aw_ctx* ctx, const aw_params* params, int orientation_mode, const aw_pair* pairs,
                    uint64_t npairs, uint32_t flags, aw_batch** out);
int aw_batch_launch(aw_ctx* ctx, aw_batch* batch, void* stream);
int aw_batch_fetch(aw_ctx* ctx, aw_batch* batch, aw_result_cb cb, void* user);
/* counters of the last launch: [0] kernels launched, [1] pairs retried with a larger workspace,
 * [2] PAF bytes, [3] CIGAR runs, [4] sum of block_len (PAF column 11), [5] failed pairs,
 * [6] wavefront cells computed, [7] wavefront steps ([2..7] are filled by aw_batch_fetch) */
int aw_batch_stats(aw_ctx* ctx, aw_batch* batch, uint64_t out[8]);
/* device time of the dominant (alignment) kernel of the last launch, from CUDA events recorded
 * on the launch stream around that kernel alone; valid after aw_batch_fetch or a stream sync */
int aw_batch_kernel_ms(aw_ctx* ctx, aw_batch* batch, float* out_ms);
/* summed device clocks (thread 0 of each CTA) of the last fetched launch: [0] breakpoint phase 1,
 * [1] phase 2 (overlap), [2] base-case wavefronts, [3] backtrace, [4] CIGAR/PAF emission, [5] other */
int aw_batch_debug_cycles(aw_ctx* ctx, aw_batch* batch, uint64_t out[6]);
void aw_batch_destroy(aw_ctx* ctx, aw_batch* batch);

/* ---- orientation only: out_is_reverse[i] in {0,1} for each pair (AW_ORIENT_MASH) ---- */
int aw_orient_pairs(aw_ctx* ctx, const aw_pair* pairs, uint64_t npairs, uint8_t* out_is_reverse);
/* scheduling aid (north_star: "partitioner balanced by predicted cost (length times divergence)"): out[i] = mash distance
 * of pair i estimated from the stranded sketches of the strand determine_orientation_mash would pick, in [0,1] */
int aw_estimate_divergence(aw_ctx* ctx, const aw_pair* pairs, uint64_t npairs, float* out);
/* stranded (canonical=0; slot 2*i forward, 2*i+1 reverse-complement) or canonical (canonical=1;
 * one per sequence) bottom-`sketch_size` sketch of sequence `idx`; returns the entry count in
 * *out_n (<= sketch_size), entries ascending with duplicates kept */
int aw_get_sketch(aw_ctx* ctx, uint32_t idx, int reverse_complement, int canonical, int k,
                  uint32_t sketch_size, uint64_t* out, uint32_t* out_n);
/* all-pairs canonical Jaccard counts for tree sparsification (src/mash.rs:141-165): for i<j,
 * inter[i*n+j], uni[i*n+j] (row-major n x n, upper triangle filled, mirrored) */
int aw_mash_jaccard_counts(aw_ctx* ctx, int k, uint32_t sketch_size, uint32_t* inter, uint32_t* uni);

/* ---- lib_wfa2::AffineWavefronts-shaped single-pair API (binds where src/alignment.rs:263-289
 *      and src/wfa.rs:188-231 construct and drive the WFA2 aligner) ---- */
typedef enum aw_memory_mode { AW_MEMORY_HIGH = 0, AW_MEMORY_MEDIUM = 1, AW_MEMORY_LOW = 2, AW_MEMORY_ULTRALOW = 3 } aw_memory_mode;
typedef enum aw_alignment_scope { AW_SCOPE_SCORE = 0, AW_SCOPE_ALIGNMENT = 1 } aw_alignment_scope;
typedef enum aw_alignment_span { AW_SPAN_END2END = 0, AW_SPAN_ENDSFREE = 1 } aw_alignment_span;
typedef enum aw_heuristic { AW_HEURISTIC_NONE = 0 } aw_heuristic;
/* AlignmentStatus of lib_wfa2 */
typedef enum aw_alignment_status { AW_ALIGN_COMPLETED = 0, AW_ALIGN_PARTIAL = 1, AW_ALIGN_MAX_STEPS = -100, AW_ALIGN_OOM = -200, AW_ALIGN_UNATTAINABLE = -300, AW_ALIGN_UNDEFINED = -1 } aw_alignment_status;

int aw_aligner_new_affine(aw_ctx* ctx, int32_t match_, int32_t mismatch, int32_t gap_opening, int32_t gap_extension,
                          int memory_mode, aw_aligner** out);
int aw_aligner_new_affine2p(aw_ctx* ctx, int32_t match_, int32_t mismatch, int32_t gap_opening1, int32_t gap_extension1,
                            int32_t gap_opening2, int32_t gap_extension2, int memory_mode, aw_aligner** out);
/* AW_SCOPE_SCORE: align() computes the score only (AW_FLAG_SCORE_ONLY), cigar() is empty; AW_SCOPE_ALIGNMENT (default): both */
int aw_aligner_set_alignment_scope(aw_aligner* a, int scope);
int aw_aligner_set_alignment_span(aw_aligner* a, int span);     /* only AW_SPAN_END2END    */
int aw_aligner_set_heuristic(aw_aligner* a, int heuristic);     /* only AW_HEURISTIC_NONE  */
int aw_aligner_get_memory_mode(const aw_aligner* a);
/* align(pattern = query, text = target); returns an aw_alignment_status */
int aw_aligner_align(aw_aligner* a, const uint8_t* pattern, int32_t pattern_len, const uint8_t* text, int32_t text_len);
int32_t aw_aligner_score(const aw_aligner* a);
/* valid until the next align on this aligner (like wf.cigar()) */
const uint8_t* aw_aligner_cigar(const aw_aligner* a, uint64_t* len);
void aw_aligner_delete(aw_aligner* a);

#ifdef __cplusplus
}
#endif
#endif
