/*
 * floxer_gpu.h -- C ABI of the B200 (sm_100a) implementation of floxer's PEX hierarchical
 * verification hot path.  Plain pointers and sizes only; no exception crosses this boundary;
 * every function returns FXG_OK (0) or a negative FXG_ERR_* code and fxg_last_error() has
 * the text.  All citations are file:line into the reference tree (floxer 0.2.0).
 *
 * What each entry point replaces:
 *   fxg_set_references   the host-resident `input::references` (include/input.hpp:30-33,
 *                        src/main/floxer.cpp:49-51) as seen by verification: packed once, kept in HBM.
 *   fxg_align_batch      N independent calls of `alignment::align(reference_span, query_span, config)`
 *                        (include/alignment.hpp:73-77, src/lib/alignment.cpp:83-181).
 *   fxg_verify_reads     the anchor loop of a verification task for whole reads:
 *                        `for anchor in package.anchors: query_verifier{...}.verify()`
 *                        (src/lib/parallelization.cpp:230-249, include/verification.hpp:22-48,
 *                        src/lib/verification.cpp:8-245), forward package(s) first, then reverse
 *                        complement (src/lib/parallelization.cpp:14-43), including the shared
 *                        verified-interval sets (src/lib/intervals.cpp:84-127).
 *   *_stage/_run/_fetch  the same work split so that a caller can keep inputs resident in HBM.
 *   fxg_seed_reads       search::searcher::search_seeds (src/lib/search.cpp:143-324) for both orientations of every read
 *                        of a batch (src/lib/parallelization.cpp:94-101), on the device: the q-gram seeder of
 *                        fxg_seeder_search with its index (fxg_gpu_seeder_create) built from the resident references.
 *   fxg_seed_verify_reads a search task's seeding and verification of a batch in one call (src/lib/parallelization.cpp:94-101
 *                        then :230-249): fxg_seed_reads + fxg_verify_reads with the anchors kept in device memory.
 *   fxg_parse_fastq      the queries' reader (input::read_queries, src/lib/input.cpp) for a FASTQ text, on the device.
 *   fxg_map_fastq        a whole run over one FASTQ text: parsing, seeding, verification and BAM / SAM output.
 *
 * Struct layouts fxg_pex_node and fxg_anchor are byte-identical to pex::pex_tree::node
 * (include/pex.hpp:59-70) and search::anchor_t (include/search.hpp:27-31) on LP64, so the
 * reference's vectors can be passed without conversion.
 */
#ifndef FLOXER_GPU_H
#define FLOXER_GPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FXG_OK 0
#define FXG_ERR_INVALID_ARGUMENT (-1)  /* bad enum / rank > 5 / out-of-range span; maps onto the reference's std::runtime_error */
#define FXG_ERR_CUDA (-2)              /* CUDA runtime failure (no device, OOM, launch error) */
#define FXG_ERR_OUT_OF_MEMORY (-3)     /* host allocation failure */
#define FXG_ERR_OVERFLOW (-4)          /* caller-provided output buffer too small; required size reported */
#define FXG_ERR_STATE (-5)             /* call order violated (e.g. verify before set_references) */

#define FXG_NULL_ID UINT64_MAX         /* pex::pex_tree::node::null_id, include/pex.hpp:60 */
#define FXG_REF_INLINE UINT32_MAX      /* task reads its reference span from the inline pool */
#define FXG_MAX_RANK 5                 /* alphabet ranks 0..5, include/input.hpp:63-66 */
#define FXG_MAX_QUERY_LENGTH 100000    /* input::queries::MAX_ALLOWED_QUERY_LENGTH, include/input.hpp:42 */

/* alignment::alignment_mode, include/alignment.hpp:53-55 */
enum { FXG_MODE_EXISTS = 0, FXG_MODE_NO_CIGAR = 1, FXG_MODE_CIGAR = 2 };
/* alignment::query_orientation, include/alignment.hpp:14-16 */
enum { FXG_FORWARD = 0, FXG_REVERSE_COMPLEMENT = 1 };
/* pex::verification_kind_t, include/pex.hpp:43-45 */
enum { FXG_KIND_DIRECT_FULL = 0, FXG_KIND_HIERARCHICAL = 1 };
/* BAM CIGAR op codes; an op is stored as (length << 4) | code.  seqan3 extended cigar, alignment.cpp:178 */
enum { FXG_CIGAR_I = 1, FXG_CIGAR_D = 2, FXG_CIGAR_EQ = 7, FXG_CIGAR_X = 8 };

typedef struct fxg_ctx fxg_ctx;
typedef struct fxg_batch fxg_batch;     /* staged fxg_align_batch */
typedef struct fxg_job fxg_job;         /* staged fxg_verify_reads */

typedef struct { uint64_t parent_id, query_index_from, query_index_to, num_errors; } fxg_pex_node;
typedef struct { uint64_t pex_leaf_index, reference_id, reference_position, num_errors; } fxg_anchor;

/* one alignment::align call: the two spans + alignment_config (include/alignment.hpp:57-62) */
typedef struct {
    uint64_t ref_offset;             /* start of the reference span inside reference `ref_id` (or the inline pool) */
    uint64_t reference_span_offset;  /* alignment_config::reference_span_offset (added to the begin position) */
    uint64_t query_offset;           /* start of the query span inside the query pool */
    uint32_t ref_len;                /* reference span length  (reference.size()) */
    uint32_t query_len;              /* query span length      (query.size())     */
    uint32_t ref_id;                 /* resident reference index, or FXG_REF_INLINE */
    uint32_t max_errors;             /* alignment_config::num_allowed_errors */
    uint8_t mode;                    /* FXG_MODE_*  */
    uint8_t orientation;             /* passed through to the result */
    uint8_t reserved[6];
} fxg_align_task;

/* alignment::alignment_result, include/alignment.hpp:64-71 */
typedef struct {
    uint64_t start_in_reference;     /* query_alignment::start_in_reference */
    uint64_t cigar_offset;           /* first op in the cigar pool (uint32 elements) */
    uint32_t cigar_len;              /* number of ops (0 unless FXG_MODE_CIGAR) */
    uint32_t num_errors;             /* query_alignment::num_errors */
    uint8_t exists;                  /* 1 = alignment_exists, 0 = no_adequate_alignment_exists */
    uint8_t orientation;
    uint8_t reserved[6];
} fxg_align_result;

/* one read with its PEX tree and anchors; mirrors parallelization::shared_verification_data
 * (include/parallelization.hpp:41-66) + the anchor packages of one query */
typedef struct {
    uint64_t query_offset;           /* into BOTH the forward and the reverse-complement pool */
    uint64_t node_offset;            /* into the node pool: num_inner inner nodes (root first), then num_leaves leaves */
    uint64_t anchor_offset;          /* into the anchor pool: forward anchors, then reverse-complement anchors */
    uint32_t query_len;
    uint32_t num_inner;
    uint32_t num_leaves;
    uint32_t num_anchors_forward;
    uint32_t num_anchors_reverse;
    uint32_t reserved;
} fxg_read;

/* pex::pex_verification_config (include/pex.hpp:47-53) + cli without_cigar (include/floxer_cli.hpp:67) */
typedef struct {
    double extra_verification_ratio;
    uint8_t verification_kind;       /* FXG_KIND_* */
    uint8_t interval_optimization;   /* 0 / 1 */
    uint8_t without_cigar;           /* 0 / 1 */
    uint8_t reserved[5];
} fxg_verify_config;

/* alignment::query_alignment + the reference it was inserted for (alignments.insert(aln, reference.internal_id)) */
typedef struct {
    uint64_t start_in_reference;
    uint64_t cigar_offset;
    uint32_t cigar_len;
    uint32_t num_errors;
    uint32_t read_index;
    uint32_t reference_id;
    uint8_t orientation;
    uint8_t reserved[7];
} fxg_alignment;

/* the three hot-path histograms (src/lib/verification.cpp:130,239,241) as count/sum, plus DP work */
typedef struct {
    uint64_t n_aligned_inner, sum_aligned_inner;
    uint64_t n_aligned_root, sum_aligned_root;
    uint64_t n_avoided_root, sum_avoided_root;
    uint64_t cells_inner, cells_root;        /* sum of m' * n' over every align call of the reference walk */
} fxg_stats;

/* device-side accounting since the last fxg_reset_counters */
typedef struct {
    uint64_t kernel_launches;        /* launches of this library's kernels */
    uint64_t dp_tasks;               /* bit-vector DP tasks executed (score passes + trace passes) */
    uint64_t dp_word_steps;          /* 32-cell Myers word-steps issued by the score passes (band-limited) */
    uint64_t dp_cells_full;          /* sum of m' * n' of those tasks (full-matrix convention) */
    uint64_t trace_bytes;            /* bytes of checkpoint records the root score passes may write for the traceback */
    uint64_t h2d_bytes, d2h_bytes;
    double dp_kernel_ms;             /* CUDA-event time of the DP kernels on the context's stream */
    double trace_kernel_ms;          /* CUDA-event time of the traceback kernels */
    uint64_t waves;                  /* host scheduling rounds of fxg_verify_* */
    double run_ms;                   /* CUDA-event time from the first to the last device operation of *_run calls */
    uint64_t trace_word_steps;       /* unused (the traceback recomputes tiles from checkpoints; no trace passes) */
    double root_launch_ms;           /* CUDA-event time of the largest launch of every root wave (the dominant launch) ... */
    uint64_t root_launch_word_steps; /* ... and the word-steps those launches issued */
    uint64_t shared_tracebacks;      /* accepted root alignments that took begin position and CIGAR from an identical one */
    uint64_t inferred_inner;         /* inner-node alignments whose existence followed from another walk of the same node */
    uint64_t shared_score_passes;    /* root windows whose result was read off a score pass over the union of several windows */
    uint64_t rescored_roots;         /* root windows scored again on their own because the shared pass could not vouch for them */
    uint64_t batches;                /* batches the queue ran for fxg_verify_run / fxg_verify_reads calls ... */
    uint64_t batch_jobs;             /* ... and the jobs in them (several callers' jobs are merged into one batch) */
    double alloc_ms;                 /* host time spent allocating device / page-locked memory (process-wide) ... */
    uint64_t alloc_calls;            /* ... and the allocations: both stay flat in the steady state */
    uint64_t root_launches;          /* launches that root_launch_ms / root_launch_word_steps cover */
} fxg_counters;

/* ---- life cycle ----
 * Environment read by fxg_create (all optional; defaults in brackets):
 *   FXG_GROUPS        [6]   worker groups = batches in flight at the same time (1..32); callers beyond that wait in the queue
 *   FXG_MERGE_JOBS    [16]  / FXG_MERGE_WALKS [1048576] / FXG_MERGE_WAIT_US [300]: how many waiting jobs (and anchors) one batch
 *                           takes, and how long a job waits for company while other batches run
 *   FXG_WORKERS       [2 per host core over all groups and local ranks, 1..4; 8 for a call that runs alone]  workers per group
 *   FXG_SPIN_US       [20]  microseconds a worker polls for its launches before it sleeps on the event
 *   FXG_DEVICE_LEVELS [1]   0: the inner tree levels are scheduled from the host, one launch and wait per level
 *   FXG_INFER_INNER   [1]   0: every inner-node window is computed (no per-node election)
 *   FXG_SHARE_ROOTS   [1]   0: every root window is scored on its own
 *   FXG_ROOT_CHUNKS / FXG_ROOT_CHUNK_MIN, FXG_MERGED_PARTS, FXG_DEVICE_ROOTS, FXG_FORCE_WIDE, FXG_LATENCY_WEIGHT, FXG_PROFILE,
 *   FXG_TRACE_WAVES, FXG_TRACE_BATCHES: development aids (DESIGN.md)
 *   FXG_SEED_CANDIDATES [2^26]  (read by fxg_gpu_seeder_create) q-gram occurrences one chunk of an fxg_seed_reads call
 *                           sorts at a time (a seed with more gets a chunk of its own): bounds its device memory
 * None of them changes a result.  When the library is loaded it sets CUDA_DEVICE_MAX_CONNECTIONS=32 unless the variable is
 * already set (INTEGRATION.md, section 4). */
int fxg_create(int device, fxg_ctx** out);
void fxg_destroy(fxg_ctx* ctx);
const char* fxg_last_error(const fxg_ctx* ctx);           /* valid until the next call on ctx */
const char* fxg_version(void);

/* packs (4 bit / base, ranks 0..5 exact) and uploads every reference once; replaces earlier ones */
int fxg_set_references(fxg_ctx* ctx, size_t n_references, const uint8_t* const* rank_sequences,
                       const uint64_t* lengths);

/* ---- alignment::align, batched ---- */
int fxg_align_batch(fxg_ctx* ctx, const fxg_align_task* tasks, size_t n_tasks,
                    const uint8_t* query_pool, size_t query_pool_len,
                    const uint8_t* inline_ref_pool, size_t inline_ref_pool_len,
                    fxg_align_result* results, uint32_t* cigar_pool, size_t cigar_capacity,
                    size_t* cigar_used);
int fxg_align_batch_stage(fxg_ctx* ctx, const fxg_align_task* tasks, size_t n_tasks,
                          const uint8_t* query_pool, size_t query_pool_len,
                          const uint8_t* inline_ref_pool, size_t inline_ref_pool_len, fxg_batch** out);
int fxg_align_batch_run(fxg_ctx* ctx, fxg_batch* batch);  /* device work only; returns after it completed.  (The tasks' DP passes are
                                                            * derived when the batch is staged; they are derived again here if the
                                                            * references were replaced in between.) */
int fxg_align_batch_fetch(fxg_ctx* ctx, fxg_batch* batch, fxg_align_result* results,
                          uint32_t* cigar_pool, size_t cigar_capacity, size_t* cigar_used);
void fxg_batch_free(fxg_ctx* ctx, fxg_batch* batch);

/* ---- query_verifier::verify for every anchor of every read ---- */
int fxg_verify_stage(fxg_ctx* ctx, const fxg_verify_config* config,
                     const fxg_read* reads, size_t n_reads,
                     const uint8_t* forward_pool, const uint8_t* reverse_complement_pool, size_t pool_len,
                     const fxg_pex_node* nodes, size_t n_nodes,
                     const fxg_anchor* anchors, size_t n_anchors, fxg_job** out);
int fxg_verify_run(fxg_ctx* ctx, fxg_job* job);
size_t fxg_job_num_alignments(const fxg_job* job);
const fxg_alignment* fxg_job_alignments(const fxg_job* job);   /* per read, in the reference's single-thread order */
size_t fxg_job_cigar_len(const fxg_job* job);
const uint32_t* fxg_job_cigar_pool(const fxg_job* job);
const fxg_stats* fxg_job_stats(const fxg_job* job);
void fxg_job_free(fxg_ctx* ctx, fxg_job* job);
/* stage + run in one call */
int fxg_verify_reads(fxg_ctx* ctx, const fxg_verify_config* config,
                     const fxg_read* reads, size_t n_reads,
                     const uint8_t* forward_pool, const uint8_t* reverse_complement_pool, size_t pool_len,
                     const fxg_pex_node* nodes, size_t n_nodes,
                     const fxg_anchor* anchors, size_t n_anchors, fxg_job** out);

/* ---- PEX tree construction (host only; pex::pex_tree::pex_tree, src/lib/pex.cpp:84-256) ----
 * build_strategy: 0 = recursive (default of the reference), 1 = bottom_up (include/pex.hpp:24-27).
 * Writes malloc'ed arrays (release with fxg_pex_free): inner[0] is the root when n_inner > 0, otherwise the
 * single leaf is the root; leaves are in left-to-right order; parent_id indexes inner. */
int fxg_pex_build(uint64_t total_query_length, uint64_t query_num_errors, uint64_t leaf_max_num_errors,
                  int build_strategy, fxg_pex_node** inner, size_t* n_inner, fxg_pex_node** leaves, size_t* n_leaves);
void fxg_pex_free(fxg_pex_node* nodes);

/* ---- SAM records (host only; row N3 of the scope table) ----
 * Replaces output::alignment_output::write_alignments_for_query (src/lib/output.cpp:49-108) for every read, plus the
 * @HD / @SQ header (src/lib/output.cpp:197-212).  fxg_write_sam takes the alignments as arrays -- grouped by read_index in
 * read order, as fxg_job_alignments returns them, with their CIGAR pool -- and needs neither a context nor a GPU;
 * fxg_job_write_sam feeds it a job's results.  `reads` / `forward_pool` are the arrays the alignments were made from,
 * `queries[i]` holds the id and the quality string of read i (input::query_record, include/input.hpp:22-28).
 * with_header = 0 leaves out the @HD / @SQ lines so that the records of several jobs can follow one header.  Refusals:
 * FXG_ERR_INVALID_ARGUMENT for a missing argument, an alignment whose reference id is out of range or that has CIGAR
 * operations but no pool; FXG_ERR_STATE for alignments not grouped by read in read order (the first problem met in
 * read order decides).  Names and CIGARs of any length are written.
 * Writes a malloc'ed, NUL-terminated buffer; release it with fxg_free. */
typedef struct { const char* id; const char* quality; } fxg_sam_query;
int fxg_write_sam(const fxg_alignment* alignments, size_t n_alignments, const uint32_t* cigar_pool,
                  size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                  const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool, const fxg_sam_query* queries,
                  int with_header, char** text, size_t* text_len);
int fxg_job_write_sam(const fxg_job* job, size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                      const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool, const fxg_sam_query* queries,
                      int with_header, char** text, size_t* text_len);
void fxg_free(void* p);

/* The same records as a BAM file image (BGZF blocks incl. the end-of-file block; the container the reference writes,
 * src/lib/output.cpp:197-212 with a .bam path).  fxg_write_bam takes the alignments as arrays -- grouped by read_index in
 * read order, as fxg_job_alignments returns them -- and needs neither a context nor a GPU; fxg_job_write_bam feeds it a
 * job's results.  with_header = 0 leaves out the BAM header (magic, text, reference list) so that the record blocks of
 * several jobs can follow one header.  Writes a malloc'ed buffer; release it with fxg_free. */
int fxg_write_bam(const fxg_alignment* alignments, size_t n_alignments, const uint32_t* cigar_pool,
                  size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                  const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool, const fxg_sam_query* queries,
                  int with_header, uint8_t** bytes, size_t* bytes_len);
int fxg_job_write_bam(const fxg_job* job, size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                      const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool, const fxg_sam_query* queries,
                      int with_header, uint8_t** bytes, size_t* bytes_len);

/* fxg_write_bam with the work on the device of ctx: record assembly and BGZF deflate run there and only the finished
 * image comes back.  Contract:
 *  - the same records: the uncompressed stream is byte-identical to fxg_write_bam's for the same arguments (header,
 *    record order, primary choice, flags, MAPQ 255, bin, SEQ with '$' as N, QUAL or 0xff, NM, the CG:B,I tag);
 *  - the same blocks: the stream is cut at the same 0xff00-byte boundaries, so block i has the ISIZE and CRC32 of
 *    fxg_write_bam's block i, and the 28-byte end-of-file block is identical.  Only the deflate payloads differ: LZ77
 *    with dynamic Huffman codes, or a stored block where that is not larger;
 *  - the same refusals: an input fxg_write_bam refuses is refused with the same code before any device work
 *    (FXG_ERR_STATE: alignments not grouped by read; FXG_ERR_INVALID_ARGUMENT: a reference id out of range, a name of
 *    more than 254 characters; FXG_ERR_OVERFLOW: a CIGAR of more than 65535 operations spanning 2^28 bases or more);
 *  - deterministic: the same input gives the same bytes;
 *  - concurrent: the call works on a stream of its own and does not hold the context's lock, so several writers and
 *    verification batches can run at once.  Its copies go through page-locked staging and are counted in fxg_counters
 *    h2d_bytes / d2h_bytes.  Needs no references.
 * Writes a malloc'ed buffer; release it with fxg_free. */
int fxg_write_bam_device(fxg_ctx* ctx, const fxg_alignment* alignments, size_t n_alignments, const uint32_t* cigar_pool,
                         size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                         const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool, const fxg_sam_query* queries,
                         int with_header, uint8_t** bytes, size_t* bytes_len);
int fxg_job_write_bam_device(fxg_ctx* ctx, const fxg_job* job, size_t n_references, const char* const* reference_ids,
                             const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool,
                             const fxg_sam_query* queries, int with_header, uint8_t** bytes, size_t* bytes_len);

/* fxg_write_sam with the work on the device of ctx: the records are formatted there (and, with bgzf = 1, compressed)
 * and only the finished bytes come back.  Contract:
 *  - bgzf = 0, the same text: byte-identical to fxg_write_sam's for the same arguments, NUL-terminated (bytes_len does
 *    not count the NUL).  That covers the @HD line and one @SQ line per reference with the full 64-bit LN; the name, '*'
 *    for a null id; the record order (a read's alignments in their stable order by reference id) and the primary (the
 *    first in that order with the read's fewest errors); flag 0 / 16, + 256 when secondary; the reference name;
 *    POS = min(start, INT32_MAX) + 1; MAPQ 255; the CIGAR as <len><op> with I D = X, '?' for other op codes, '*' without
 *    operations, written out whatever its length; "*\t0\t0"; SEQ and QUAL on the primary only -- SEQ the forward read
 *    with rank 0 as '$', 1..5 as ACGTN, >= 6 as N, '*' when empty; QUAL verbatim whatever its length, '*' when null or
 *    empty --; NM:i:; and one flag-4 record without NM for a read without alignments;
 *  - bgzf = 1, BGZF-compressed SAM (what htslib reads as .sam.gz): the text above cut at 0xff00-byte boundaries, one
 *    BGZF block per chunk with that chunk's ISIZE and CRC32, then the 28-byte end-of-file block;
 *  - the same refusals as fxg_write_sam, with the same codes, before any device work;
 *  - deterministic, concurrent and counted as fxg_write_bam_device: a stream of its own without the context's lock,
 *    one upload through page-locked staging, copies counted in fxg_counters h2d_bytes / d2h_bytes.  Needs no references.
 * Writes a malloc'ed buffer; release it with fxg_free. */
int fxg_write_sam_device(fxg_ctx* ctx, const fxg_alignment* alignments, size_t n_alignments, const uint32_t* cigar_pool,
                         size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                         const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool, const fxg_sam_query* queries,
                         int with_header, int bgzf, uint8_t** bytes, size_t* bytes_len);
int fxg_job_write_sam_device(fxg_ctx* ctx, const fxg_job* job, size_t n_references, const char* const* reference_ids,
                             const uint64_t* reference_lengths, const fxg_read* reads, size_t n_reads, const uint8_t* forward_pool,
                             const fxg_sam_query* queries, int with_header, int bgzf, uint8_t** bytes, size_t* bytes_len);

/* ---- a q-gram seeder behind the anchor interface (host only; row N2 of the scope table) ----
 * Stands in for search::searcher::search_seeds (src/lib/search.cpp:143-324), whose FM-index library cannot be built
 * offline: per PEX leaf every reference position where the leaf matches a prefix of the reference with at most
 * leaf.num_errors edits, as search::anchor_t, after the reference's caps (max_num_anchors_hard / _soft,
 * include/floxer_cli.hpp:52-53) and erase_useless_anchors (search.cpp:352-389), in seed -> reference -> position order.
 * q = length of the indexed q-grams (4..14); a leaf must be at least q * (num_errors + 1) long.  The index copies the
 * references.  fxg_seeder_search writes a malloc'ed array (release with fxg_free) and may be called from several threads. */
typedef struct fxg_seeder fxg_seeder;
int fxg_seeder_create(size_t n_references, const uint8_t* const* rank_sequences, const uint64_t* lengths, uint32_t q, fxg_seeder** out);
void fxg_seeder_free(fxg_seeder* seeder);
int fxg_seeder_search(const fxg_seeder* seeder, const uint8_t* query, size_t query_len, const fxg_pex_node* leaves, size_t n_leaves,
                      uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors, fxg_anchor** anchors, size_t* n_anchors);

/* ---- the same seeder on the device, for whole read batches ---- */
typedef struct fxg_gpu_seeder fxg_gpu_seeder;
typedef struct {
    uint64_t seeds;              /* (read, strand, leaf) triples searched */
    uint64_t candidates;         /* candidate starts before de-duplication */
    uint64_t checked;            /* distinct candidate starts checked with the banded DP */
    uint64_t hits;               /* raw anchors (distance <= leaf errors) */
    uint64_t dropped_hard;       /* raw anchors of seeds removed by the hard cap */
    uint64_t cut_soft;           /* raw anchors removed by the soft cap */
    uint64_t erased;             /* anchors removed by erase_useless_anchors */
    uint64_t reserved;
} fxg_seed_stats;

/* q-gram index (q = 4..14) of the references resident in ctx (fxg_set_references), built on the device from the packed
 * store (no second copy of the references): 4^(q+1) bytes of buckets + 4 bytes per indexed position of device memory.
 * FXG_ERR_INVALID_ARGUMENT for references of 2^32 bases or more (as fxg_seeder_create), FXG_ERR_STATE without references. */
int  fxg_gpu_seeder_create(fxg_ctx* ctx, uint32_t q, fxg_gpu_seeder** out);
void fxg_gpu_seeder_free(fxg_ctx* ctx, fxg_gpu_seeder* seeder);
/* fxg_seeder_search for both orientations of every read of a batch.  `reads` is in/out: query_offset, query_len,
 * node_offset, num_inner, num_leaves are read; anchor_offset, num_anchors_forward, num_anchors_reverse are written, so
 * (reads, pools, nodes, *anchors) can be passed to fxg_verify_stage / fxg_verify_reads as they are.  Anchors: malloc'ed,
 * release with fxg_free; per read the forward orientation's anchors, then the reverse complement's, each in
 * seed -> reference -> position order, equal to what fxg_seeder_search returns for that orientation.  stats may be NULL.
 * A leaf fxg_seeder_search refuses fails the whole call with FXG_ERR_INVALID_ARGUMENT before any device work;
 * FXG_ERR_STATE once fxg_set_references has replaced the references the seeder was made from (and fxg_set_references
 * fails with FXG_ERR_STATE while a seeding call runs).  Several threads may seed on one context at a time, beside
 * verification runs: each call works on a stream of its own. */
int  fxg_seed_reads(fxg_ctx* ctx, const fxg_gpu_seeder* seeder, fxg_read* reads, size_t n_reads,
                    const uint8_t* forward_pool, const uint8_t* reverse_complement_pool, size_t pool_len,
                    const fxg_pex_node* nodes, size_t n_nodes,
                    uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors,
                    fxg_anchor** anchors, size_t* n_anchors, fxg_seed_stats* stats);

/* fxg_seed_reads followed by fxg_verify_reads on the same batch, without the anchors leaving the device.  `reads` is
 * in/out exactly as for fxg_seed_reads (anchor_offset, num_anchors_forward, num_anchors_reverse are written).  The job
 * is the one fxg_verify_reads would return for the seeded batch: the same alignments in the same order, the same CIGARs
 * and statistics; it is read with fxg_job_* / fxg_job_write_sam / fxg_job_write_bam and, like fxg_verify_reads's job,
 * cannot be run again.  stats may be NULL.
 * The query pools go up once; the seeder writes the surviving anchors straight into the job's device records and only
 * their counts per read (8 bytes) come back.  An input either call refuses is refused with its code and text before any
 * device work (a seeding refusal first); a rank above 5 in a pool is reported after the run, as fxg_verify_reads does.
 * The job joins the batch queue like an fxg_verify_reads job and merges with jobs of the same fxg_verify_config;
 * fxg_set_references fails with FXG_ERR_STATE while the call runs.  The copies it makes, seeding included, are counted
 * in fxg_counters h2d_bytes / d2h_bytes. */
int  fxg_seed_verify_reads(fxg_ctx* ctx, const fxg_gpu_seeder* seeder, const fxg_verify_config* config,
                           fxg_read* reads, size_t n_reads,
                           const uint8_t* forward_pool, const uint8_t* reverse_complement_pool, size_t pool_len,
                           const fxg_pex_node* nodes, size_t n_nodes,
                           uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors,
                           fxg_seed_stats* stats, fxg_job** out);

/* ---- FASTQ input on the device ----
 * The text of fxg_parse_fastq / fxg_map_fastq holds whole FASTQ records of four lines: '@' and a header, the sequence,
 * '+' and anything, the quality.  Lines end at '\n'; one '\r' before the end of a line is dropped; the last line may lack
 * its '\n' (multi-line records are not read).  A read's id is its header after '@' up to the first space or tab.  Its
 * ranks follow input.cpp:165-176 ('$' -> 0, A C G T in either case -> 1..4, any other byte -> 5), its reverse complement
 * swaps A<->T and C<->G.  Its error budget k is query_errors, or floating_point_error_aware_ceil(m * error_probability)
 * when query_errors is FXG_NULL_ID (math.hpp:22-27, input.cpp:26-34), and its PEX tree is fxg_pex_build(m, k,
 * seed_errors, build_strategy).  The text is uploaded once, through page-locked staging, on a stream of the call's own;
 * the device finds the lines and records, checks them, cuts the ids, converts the ranks and lays out the kept reads'
 * pools; the trees are built on the host.  A text of 2^31 bytes or more is refused (split it at a record boundary). */
typedef struct {
    double error_probability;   /* used when query_errors == FXG_NULL_ID */
    uint64_t query_errors;      /* k of every read, or FXG_NULL_ID */
    uint64_t seed_errors;       /* the leaves' error budget (leaf_max_num_errors) */
    uint32_t build_strategy;    /* 0 recursive, 1 bottom_up */
    uint32_t reserved;
} fxg_read_config;
/* a record's status: kept, or skipped and not written -- k < seed_errors (input.cpp:114-129), m = 0 or
 * m > FXG_MAX_QUERY_LENGTH (input.cpp:106-110), or (fxg_map_fastq) a leaf the q-gram seeder refuses */
enum { FXG_READ_KEPT = 0, FXG_READ_TOO_FEW_ERRORS = 1, FXG_READ_BAD_LENGTH = 2, FXG_READ_UNSEEDABLE = 3 };
enum { FXG_FORMAT_BAM = 0, FXG_FORMAT_SAM = 1, FXG_FORMAT_SAM_BGZF = 2 };

/* where a kept read came from: its record's index and the spans of its id and its quality in the text */
typedef struct { uint64_t record, id_offset, quality_offset; uint32_t id_len, quality_len; } fxg_read_span;

typedef struct fxg_parsed fxg_parsed;
/* the arrays of a parsed text; they live as long as the fxg_parsed.  reads / pools / nodes go into fxg_seed_reads,
 * fxg_seed_verify_reads and fxg_verify_reads as they are (the reads' anchor fields are zero). */
typedef struct {
    size_t n_records; const uint8_t* statuses;           /* per record: FXG_READ_* */
    size_t n_reads; const fxg_read* reads; const fxg_read_span* spans;    /* the kept reads, in record order */
    size_t pool_len; const uint8_t* forward_pool; const uint8_t* reverse_complement_pool;
    size_t n_nodes; const fxg_pex_node* nodes;
} fxg_parsed_view;

/* Parses text[0, text_len).  A malformed record (a header without '@', a third line without '+', a record cut short)
 * fails the call with FXG_ERR_INVALID_ARGUMENT and fxg_last_error names the first one's index.  Copies the pools back. */
int fxg_parse_fastq(fxg_ctx* ctx, const fxg_read_config* config, const char* text, size_t text_len, fxg_parsed** out);
int fxg_parsed_get(const fxg_parsed* parsed, fxg_parsed_view* view);
void fxg_parsed_free(fxg_parsed* parsed);

typedef struct {
    uint64_t records;            /* FASTQ records in the text */
    uint64_t reads[4];           /* records per FXG_READ_* status; reads[FXG_READ_KEPT] were mapped and written */
    uint64_t alignments;
    fxg_seed_stats seed;
} fxg_map_summary;

/* Maps a FASTQ text in one call: fxg_parse_fastq on the device, the trees on the host, then the kept reads -- less those
 * with a leaf the q-gram seeder refuses (fewer than q * (errors + 1) bases or more than 8 errors: FXG_READ_UNSEEDABLE, a
 * limit of the stand-in seeder, counted and not written) -- through fxg_seed_verify_reads and the device record writer
 * (format FXG_FORMAT_*: fxg_write_bam_device, fxg_write_sam_device with bgzf 0 or 1).  The output is that of those calls
 * composed on the kept reads in record order, with each read's id and quality: SAM the same bytes, BAM and BGZF SAM the
 * same uncompressed stream and blocks.  The query pools do not go up a second time: the job's pool is filled from the
 * parsed pool on the device, SEQ is read from it and the names and qualities from the device copy of the text.  Refusals
 * keep the codes of the calls composed (for example a name of more than 254 characters in BAM).  Several threads may map
 * on one context.  Copies are counted in fxg_counters h2d_bytes / d2h_bytes.  summary may be NULL.
 * Writes a malloc'ed buffer; release it with fxg_free. */
int fxg_map_fastq(fxg_ctx* ctx, const fxg_gpu_seeder* seeder, const fxg_read_config* read_config, const fxg_verify_config* verify_config,
                  uint64_t max_anchors_hard, uint64_t max_anchors_soft, int erase_useless_anchors,
                  const char* text, size_t text_len, size_t n_references, const char* const* reference_ids, const uint64_t* reference_lengths,
                  int format, int with_header, uint8_t** bytes, size_t* bytes_len, fxg_map_summary* summary);

/* ---- accounting / measurement helpers ---- */
int fxg_get_counters(const fxg_ctx* ctx, fxg_counters* out);
int fxg_reset_counters(fxg_ctx* ctx);
/* issue-rate microbenchmark: dependent-free LOP3/IADD3/SHF stream in the 8:1:2 mix of one Myers word-step;
 * returns thread-instructions per second (the int32 roofline denominator, SURVEY 8d) */
int fxg_measure_int32_peak(fxg_ctx* ctx, double* thread_instructions_per_second);

/* the engine's shape for one alignment::align call of a query of length m against a window of length n with at most k
 * errors: 32-bit words per lane (block height / 32), lanes per ring (64: the multi-warp kernel), blocks of the query and
 * the band-limited word-steps of the pass.  Needs no device (tests check the ring rule of DESIGN.md 4.1 on it).
 * with_traceback != 0: a pass whose CIGAR is wanted -- the block width is chosen with the traceback's cost in the sum.
 * FXG_ERR_INVALID_ARGUMENT if no alignment is possible (m = 0 or m - n > k). */
int fxg_engine_shape(uint32_t n, uint32_t m, uint32_t k, int with_traceback, uint32_t* words_per_lane, uint32_t* ring_lanes, uint32_t* blocks,
                     uint64_t* word_steps);

#ifdef __cplusplus
}
#endif
#endif
