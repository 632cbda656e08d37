/*
 * fadegpu.h -- C ABI of libfadegpu: the B200 (sm_100a) implementation of the soft-clip
 * realignment hot path of `fade annotate` (blachlylab/fade).
 *
 * The reference has no FFI seam of its own: align_clip() calls dparasail and dhtslib directly
 * (source/analysis.d:63,67).  This header therefore defines the seam at the narrowest cut that
 * contains all heavy work, and each entry point names the reference code it replaces:
 *
 *   fadegpu_create            <- Parasail("ACTGN",10,2,2,-3) profile construction, source/anno.d:36,
 *                                and the two numeric flags that reach the path, source/app.d:17-18
 *   fadegpu_load_reference    <- IndexedFastaFile(args[2]) + every fai.fetchSequence(...).toUpper
 *                                under the global mutex, source/anno.d:23, source/analysis.d:61-64
 *   fadegpu_submit/_wait      <- the body of `foreach(rec; parallel(bam.allRecords))`,
 *                                source/anno.d:44-50, i.e. per record steps a-d of align_clip:
 *                                length floor (analysis.d:34), reverse complement (analysis.d:40,
 *                                util.d:18-34), window arithmetic (analysis.d:45-59), window fetch
 *                                (analysis.d:63), p.sw_striped (analysis.d:67), res.cigar
 *                                (analysis.d:69) and the accept predicates (analysis.d:69-80,98-104)
 *
 * Everything above the seam (BAM/SAM decode, parse_clips on the read's CIGAR, the SA lookup, rs
 * byte assembly, am/as/ar/ab string formatting, BAM encode, the CLI) stays on the host; see
 * include/fadehost.h and INTEGRATION.md for the D binding.
 *
 * Conventions: plain C; every function returns 0 (FADEGPU_OK) or a negative fadegpu_status and
 * never throws or aborts.  There is NO CPU fallback: without a CUDA device (or with the kernels
 * failing to launch) calls fail with FADEGPU_E_CUDA / FADEGPU_E_NODEV.
 * Threading: a ctx (and its batches) is driven by one host thread at a time; distinct ctxs may be
 * driven concurrently.  A ctx owns one helper thread (started by the first queued submit of a batch
 * or a job) that plans and launches queued batches and jobs.  All buffers handed out are owned by
 * the library.
 */
#ifndef FADEGPU_H
#define FADEGPU_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define FADEGPU_ABI_VERSION 2
#define FADEGPU_MAX_OPS 10 /* CIGAR ops materialised per read: fade rejects anything above 10 (analysis.d:69);
                              n_ops always holds the full count */

typedef enum {
    FADEGPU_OK = 0,
    FADEGPU_E_ARG = -1,   /* bad argument */
    FADEGPU_E_CUDA = -2,  /* CUDA runtime / kernel failure */
    FADEGPU_E_OOM = -3,   /* host or device allocation failed */
    FADEGPU_E_STATE = -4, /* call sequence error (no reference, batch in flight, ...) */
    FADEGPU_E_NODEV = -5  /* no usable CUDA device */
} fadegpu_status;

typedef struct fadegpu_ctx fadegpu_ctx;     /* opaque; one per (host thread, GPU) */
typedef struct fadegpu_batch fadegpu_batch; /* opaque; pinned host + device buffers */

typedef struct fadegpu_params {
    int32_t window_size;   /* --window-size, source/app.d:18, default 300 */
    int32_t min_length;    /* --min-length,  source/app.d:17, default 5   */
    int32_t gap_open;      /* 10  source/anno.d:36 */
    int32_t gap_extend;    /* 2   */
    int32_t match;         /* 2   */
    int32_t mismatch;      /* -3  */
    uint32_t flags;        /* FADEGPU_F_* */
    int64_t scratch_bytes; /* cap on the device checkpoint scratch per launch; 0 = default */
    int32_t host_threads;  /* host threads of the library's per-read loops (gather of fadegpu_submit_inputs,
                              scatter of fadegpu_wait, FADEGPU_F_HOST_BINNING); 0 = all cores */
    int32_t reserved;
} fadegpu_params;

/* params.flags */
#define FADEGPU_F_FORCE_GENERIC 1u /* route every alignment through the generic (slow) kernel */
#define FADEGPU_F_NO_SHORTCUT 8u   /* traceback: always replay blocks, never use the ungapped-diagonal proof
                                      (A/B switch; results are identical) */
#define FADEGPU_F_HOST_BINNING 16u  /* both submit calls: classify, sort and gather the reads on the host (the first
                                      implementation, kept as an A/B switch) instead of binning them on the device */
#define FADEGPU_F_SYNC_SUBMIT 32u   /* fadegpu_submit: plan and launch on the calling thread (errors of the batch
                                      are then returned by fadegpu_submit itself instead of fadegpu_wait) */
#define FADEGPU_F_TAGS_ONLY 4u     /* the caller only needs what fade writes into the tags: an alignment whose score already
                                      fails `score > clip_len*0.9*2` (analysis.d:43,76,100) for both clips gets no end cell and
                                      no traceback -- its record carries the score, n_ops = 0 and FADEGPU_R_SCORE_ONLY; flags[]
                                      (art_left / art_right) and the records of every other read are unchanged */
#define FADEGPU_F_NO_SCATTER 2u    /* fadegpu_wait fills only flags[] and the compact results
                                      (fadegpu_get_results), not the other per-read output arrays */

/* per-read result flags */
#define FADEGPU_R_ALIGNED 1u    /* SW ran for this read (some clip passed the length floor) */
#define FADEGPU_R_ART_LEFT 2u   /* status.art_left  (analysis.d:82)  */
#define FADEGPU_R_ART_RIGHT 4u  /* status.art_right (analysis.d:106) */
#define FADEGPU_R_OPS_TRUNC 8u  /* n_ops > FADEGPU_MAX_OPS, only the first ones are materialised */
#define FADEGPU_R_GENERIC 16u   /* served by the generic kernel (wildcard letters / odd sizes) */
#define FADEGPU_R_SCORE_ONLY 64u /* FADEGPU_F_TAGS_ONLY: only `score` is valid in this read's record (no artifact possible) */
#define FADEGPU_R_OVERSIZE 32u  /* NOT aligned: the read's window exceeds 2^31 DP cells (a spliced record spanning
                                   megabases); counted in fadegpu_stats.n_oversize, the batch goes on */

/* Struct-of-arrays view of a batch.  Inputs are filled by the caller before fadegpu_submit;
 * outputs are valid after fadegpu_wait until the next submit of the same batch. */
typedef struct fadegpu_batch_view {
    int64_t max_reads, max_seq_bytes;
    /* ---- inputs ---- */
    uint8_t *seq4;        /* BAM 4-bit packed bases exactly as in bam1_t (util.d:25,31), reads concatenated */
    int64_t *seq_off;     /* [n+1] byte offset of read k's bases inside seq4 */
    int32_t *l_qseq;      /* [n] rec.length */
    int32_t *tid;         /* [n] rec.tid (contig index of fadegpu_load_reference) */
    int64_t *pos;         /* [n] rec.pos, 0-based */
    int32_t *aligned_len; /* [n] rec.cigar.alignedLength (reference span), analysis.d:53 */
    int32_t *clip_left;   /* [n] parse_clips(rec.cigar)[0].length, 0 = none or early-out record */
    int32_t *clip_right;  /* [n] parse_clips(rec.cigar)[1].length */
    /* ---- outputs: flags is written for every read; all the others are defined only for reads
     *      whose flags have FADEGPU_R_ALIGNED set, and are NULL (not allocated) when the ctx was
     *      created with FADEGPU_F_NO_SCATTER: use fadegpu_get_results then ---- */
    uint8_t *flags;       /* [n] FADEGPU_R_* */
    int32_t *score;       /* [n] res.score */
    int32_t *beg_query;   /* [n] */
    int32_t *end_query;   /* [n] */
    int32_t *beg_ref;     /* [n] res.position, window relative */
    int32_t *end_ref;     /* [n] */
    int64_t *win_start;   /* [n] `start` of analysis.d:45-51; am POS = win_start + beg_ref */
    int32_t *n_ops;       /* [n] res.cigar.length including the S padding */
    uint32_t *ops;        /* [n * FADEGPU_MAX_OPS] BAM-encoded (len<<4|op), forward order */
    /* ---- compact inputs (fadegpu_submit_compact): an alternative to the seven input arrays above ---- */
    uint8_t *gate;                 /* [n] min(255, max(clip_left, clip_right)): the one byte per read that is copied
                                      to the device for EVERY read; it decides the length floor (analysis.d:34) there */
    struct fadegpu_read_meta *meta; /* [n] everything else about a read; the GPU fetches only the records it aligns */
} fadegpu_batch_view;

/* One read of the compact layout: 32 bytes, fetched by the GPU over PCIe as one sector, and only for
 * the reads whose gate byte passes the length floor (about one in six in fade's workload). */
typedef struct fadegpu_read_meta {
    int64_t pos;          /* rec.pos, 0-based */
    uint32_t seq_off;     /* byte offset of the read's bases inside seq4 (compact batches hold < 4 GiB of bases) */
    int32_t l_qseq;       /* rec.length */
    int32_t tid;          /* rec.tid */
    int32_t aligned_len;  /* rec.cigar.alignedLength, analysis.d:53 */
    uint32_t clip_left;   /* parse_clips(rec.cigar)[0].length, 0 = none */
    uint32_t clip_right;  /* parse_clips(rec.cigar)[1].length */
} fadegpu_read_meta;

typedef struct fadegpu_stats {
    int64_t n_reads;          /* reads in the last submit */
    int64_t n_aligned;        /* reads for which SW ran (once per read) */
    int64_t n_generic;        /* of those, served by the generic kernel */
    int64_t cells;            /* sum qlen*tlen over aligned reads (counted once per read) */
    int64_t h2d_bytes, d2h_bytes;
    int32_t kernel_launches;  /* kernels launched by the last submit */
    float kernel_ms;          /* device time of all kernels of the last submit (CUDA events) */
    float fill_ms, trace_ms, generic_ms; /* per-stage device time (events on the ctx stream) */
    float total_ms;           /* H2D + kernels + D2H device time */
    int64_t scratch_bytes;    /* checkpoint scratch used */
    float host_submit_ms;     /* wall clock of the host part of fadegpu_submit (binning, gather, queueing) */
    float host_wait_ms;       /* wall clock of the host part of fadegpu_wait after the stream finished (scatter) */
    float host_classify_ms, host_sort_ms, host_gather_ms;   /* parts of host_submit_ms */
    int32_t host_threads;     /* threads actually used */
    int32_t reserved;
    int64_t n_oversize;       /* reads left unaligned because their window exceeds 2^31 DP cells (FADEGPU_R_OVERSIZE) */
} fadegpu_stats;

int fadegpu_abi_version(void);
int fadegpu_device_count(int *n);
int fadegpu_default_params(fadegpu_params *p);
int fadegpu_create(int device, const fadegpu_params *p, fadegpu_ctx **out);
void fadegpu_destroy(fadegpu_ctx *ctx);
/* ctx may be NULL: returns the calling thread's last error outside any ctx */
const char *fadegpu_last_error(const fadegpu_ctx *ctx);

/* Host ASCII contigs (any case, any letters) are packed (2-bit + N plane + wildcard plane) and
 * uploaded once; the reference then stays resident in HBM.  Replaces anno.d:23 + analysis.d:61-64. */
int fadegpu_load_reference(fadegpu_ctx *ctx, int32_t n_contigs, const char *const *names,
                           const int64_t *lengths, const char *const *seqs);
/* Optional: device-to-device copy (NVLink peer copy when available) of src's packed reference. */
int fadegpu_share_reference(fadegpu_ctx *dst, const fadegpu_ctx *src);
int fadegpu_reference_info(const fadegpu_ctx *ctx, int32_t *n_contigs, int64_t *total_bases,
                           int64_t *device_bytes);

int fadegpu_alloc_batch(fadegpu_ctx *ctx, int64_t max_reads, int64_t max_seq_bytes,
                        fadegpu_batch **out);
int fadegpu_get_batch_view(fadegpu_batch *b, fadegpu_batch_view *view);
void fadegpu_free_batch(fadegpu_batch *b);

/* Asynchronous: returns at once.  The per-read arrays of the pinned view are DMA'd to the device as
 * they are and the binning (length floor, windows, sort by window length) runs on the GPU; a thread
 * owned by the ctx turns the small histogram into the launch plan and queues the kernels.  Uploads
 * and binning of one batch overlap with the kernels of the previous one and with the result copies
 * of the one before.  The view's input arrays must stay untouched until fadegpu_wait, which also
 * reports any error of the batch (inconsistent seq_off, window too large, CUDA failure). */
int fadegpu_submit(fadegpu_ctx *ctx, fadegpu_batch *b, int64_t n_reads);

/* Same, for a batch whose view holds the COMPACT layout (gate[], meta[], seq4; seq_bytes = bytes of seq4 in use):
 * one byte per read is copied to the device; the 32-byte records and the bases of the reads that pass the
 * length floor are fetched by the GPU from the pinned view.  About 22 bytes per read cross PCIe on fade's workload
 * instead of 51 (and 18 instead of 22 come back: 72-byte result records of the aligned reads, flags[] and the index). */
int fadegpu_submit_compact(fadegpu_ctx *ctx, fadegpu_batch *b, int64_t n_reads, int64_t seq_bytes);

/* Same, reading the inputs from caller-owned host arrays (pageable is fine: the library gathers
 * the reads that need SW into its own pinned staging before the H2D copy).  The arrays are only
 * read during the call.  n_reads <= max_reads of the batch; the results land in the batch's view. */
typedef struct fadegpu_inputs {
    const uint8_t *seq4;
    const int64_t *seq_off;
    const int32_t *l_qseq, *tid;
    const int64_t *pos;
    const int32_t *aligned_len, *clip_left, *clip_right;
} fadegpu_inputs;
int fadegpu_submit_inputs(fadegpu_ctx *ctx, fadegpu_batch *b, int64_t n_reads, const fadegpu_inputs *in);
/* Blocks until the batch is done and scatters the results into the view's output arrays. */
int fadegpu_wait(fadegpu_ctx *ctx, fadegpu_batch *b);

/* Compact results of the last fadegpu_wait: one record per read for which SW ran, in the
 * library's processing order (by window length; unspecified among equal lengths, so it may differ
 * between two runs on the same input -- address records through result_index), plus a per-read
 * index into them.  Always filled (cheaper for the
 * host than the per-read arrays of the view: nothing is scattered but flags[] and the index). */
typedef struct fadegpu_result {
    int32_t score;                 /* res.score */
    int32_t end_query, end_ref;    /* end cell, window relative */
    int32_t beg_query, beg_ref;    /* beg_ref == res.position */
    int32_t n_ops;                 /* res.cigar.length including the S padding */
    uint32_t flags;                /* FADEGPU_R_* */
    int32_t read;                  /* index of the read inside the batch */
    uint32_t ops[FADEGPU_MAX_OPS]; /* BAM-encoded, forward order */
} fadegpu_result;
typedef struct fadegpu_results_view {
    int64_t n_results;
    const fadegpu_result *results;   /* [n_results] */
    const int64_t *win_start;        /* [n_results] `start` of analysis.d:45-51 */
    const int32_t *result_index;     /* [n_reads]  index into results, -1 = no SW for this read */
} fadegpu_results_view;
int fadegpu_get_results(const fadegpu_batch *b, fadegpu_results_view *r);

/* Measurement helpers (bench.py): stats of the last submit, and a re-run of ONLY the kernels on
 * the inputs already resident in HBM (no host work, no copies), timed with CUDA events on the ctx
 * stream.  ms_out receives the device milliseconds of `iters` passes. */
int fadegpu_get_stats(const fadegpu_batch *b, fadegpu_stats *s);
/* Device timeline of the batch's last submit relative to the start of `origin`'s last submit (both of the same ctx,
 * both waited for): ms[0] start of the uploads, ms[1] the compute stream reaches the batch (first fill starts), ms[2] end
 * of its kernels, ms[3] results on the host, ms[4] inputs ready on the upload stream, ms[5] end of its last fill; -1 where
 * the last submit did not record the event.  For pipeline diagnostics (tools/e2e_timeline.py). */
int fadegpu_get_timeline(const fadegpu_batch *b, const fadegpu_batch *origin, float ms[6]);
int fadegpu_replay_kernels(fadegpu_ctx *ctx, fadegpu_batch *b, int32_t iters, float *ms_out);
/* The same over several resident batches of the ctx, queued back to back the way consecutive submits
 * queue them (the traceback rounds of one batch run under the fill of the next): device
 * milliseconds of `iters` passes over all of them, first fill to last traceback. */
int fadegpu_replay_batches(fadegpu_ctx *ctx, fadegpu_batch *const *batches, int32_t n_batches, int32_t iters,
                           float *ms_out);

/* ---- Pairwise Smith-Waterman with traceback on caller-supplied sequences ----
 * Pair k is query[query_off[k] .. query_off[k+1]) against target[target_off[k] .. target_off[k+1]).
 *
 * Alignment semantics: exactly P1-P5 (SURVEY 8a) with the ctx's scoring, the query taken as given (no reverse
 *   complement) and the whole target as the window.  Query and target are upper-cased, as the reference path does
 *   (toUpper, source/analysis.d:63).
 * Target letters: any byte -- ACGT, N as a real symbol, everything else a wildcard, as in fadegpu_load_reference.
 * Query letters: they must lie in the BAM nt16 alphabet =ACMGRSVTWYHKDBN, in either case (the kernels read queries as
 *   nt16 codes).  Any other letter fails the call with FADEGPU_E_ARG, and fadegpu_last_error names the first pair
 *   holding one.
 * Scoring: from the ctx (fadegpu_params); a ctx used only for pairs needs no fadegpu_load_reference.  The ctx's
 *   FADEGPU_F_FORCE_GENERIC applies; FADEGPU_F_TAGS_ONLY does not: every pair is traced back.
 * CIGAR ops: n_ops is always exact.  ops_out[k * max_ops ..] holds the first min(n_ops, max_ops) ops of pair k's forward
 *   CIGAR (BAM-encoded, S padding included, zero-filled), and FADEGPU_R_OPS_TRUNC is set when n_ops > max_ops -- the
 *   convention of the 10-op records.  max_ops = 3 * max(query length) never truncates: a local alignment starts and
 *   ends with a diagonal step, every =/X run holds one, between two of them lie at most one I and one D run, plus at
 *   most two S ops.  ops_out may be NULL iff max_ops == 0.
 * Empty pairs: a pair with an empty query or target gets flags = 0 and a zero record.
 * Oversize pairs: a pair with query length * target length > 2^31 is not aligned; it gets FADEGPU_R_OVERSIZE and is
 *   counted in stats_out->n_oversize.  FADEGPU_R_ART_* and FADEGPU_R_SCORE_ONLY are never set.
 * In-flight batches: while a batch of the ctx is submitted and not yet waited for, the call fails with
 *   FADEGPU_E_STATE.
 * No side effects on batches: the results of waited batches (fadegpu_get_results) stay valid, and
 *   fadegpu_replay_kernels / fadegpu_replay_batches of existing batches keep working.
 *
 * Synchronous.  The arrays are host memory (pageable is fine) and only read during the call.  out[n_pairs] receives
 * the records in PAIR ORDER.  stats_out (may be NULL) receives, for this call: n_reads = n_pairs, n_aligned, n_generic,
 * cells, n_oversize, kernel_launches, h2d / d2h bytes, kernel_ms (the SW kernels: fills, traceback, generic) and
 * total_ms (upload to results home); the per-stage fill / trace / generic times are not taken (0). */
typedef struct fadegpu_pairs {
    const char *query;  const int64_t *query_off;    /* [n+1] ASCII queries, concatenated */
    const char *target; const int64_t *target_off;   /* [n+1] ASCII targets, concatenated */
} fadegpu_pairs;                                     /* 32 bytes */

typedef struct fadegpu_pair_result {
    int32_t score, end_query, end_ref, beg_query, beg_ref;  /* as fadegpu_result; beg_ref == res.position */
    int32_t n_ops;                                          /* full length of the forward CIGAR, S padding included (P5) */
    uint32_t flags;         /* FADEGPU_R_ALIGNED | FADEGPU_R_GENERIC | FADEGPU_R_OPS_TRUNC | FADEGPU_R_OVERSIZE only */
    int32_t reserved;
} fadegpu_pair_result;                                      /* 32 bytes */

int fadegpu_align_pairs(fadegpu_ctx *ctx, int64_t n_pairs, const fadegpu_pairs *in, int32_t max_ops,
                        fadegpu_pair_result *out, uint32_t *ops_out, fadegpu_stats *stats_out);

/* ---- Smith-Waterman with traceback of caller-supplied queries against intervals of the resident reference ----
 * Region k is query[query_off[k] .. query_off[k+1]) against [start[k], end[k]) of contig tid[k] (the index into the
 * contigs of fadegpu_load_reference), on strand[k]: 0 aligns the query as given, 1 its reverse complement.
 *
 * Alignment semantics: exactly P1-P5 (SURVEY 8a) with the ctx's scoring and the interval as the window, upper-cased as
 *   every window is.  The reverse complement of strand 1 is the nt16 complement (source/util.d:18-34), so IUPAC
 *   letters stay valid.  beg_query / end_query index the query as it was aligned (for strand 1: its reverse
 *   complement, as the annotate records do); beg_ref / end_ref are relative to start, so the reference position of
 *   the alignment is start + beg_ref.
 * Query letters: as fadegpu_align_pairs; a letter outside nt16 fails the call with FADEGPU_E_ARG naming the first
 *   region holding one (checked on the device).
 * Scoring: from the ctx; FADEGPU_F_FORCE_GENERIC applies, FADEGPU_F_TAGS_ONLY does not: every region is traced back.
 *   No length floor and no accept predicate applies.
 * Records and CIGAR ops: as fadegpu_align_pairs, in REGION ORDER: n_ops is always exact, max_ops / ops_out /
 *   FADEGPU_R_OPS_TRUNC follow the same rules, flags hold only ALIGNED | GENERIC | OPS_TRUNC | OVERSIZE.
 * Empty regions: an empty query or an empty interval gives flags = 0 and a zero record.
 * Oversize regions: query length * (end - start) > 2^31, or end - start > 0x7fffffff: not aligned, FADEGPU_R_OVERSIZE,
 *   counted in stats_out->n_oversize.
 * Argument errors (FADEGPU_E_ARG, checked on the host before anything is uploaded; fadegpu_last_error names the first
 *   offending region): tid outside [0, n_contigs), start < 0, start > end, end > the contig's length, strand other
 *   than 0 or 1, decreasing query offsets, null arrays.
 * State errors (FADEGPU_E_STATE): no reference is loaded, or a batch of the ctx is in flight.  Waited batches keep
 *   their results, and fadegpu_replay_kernels / fadegpu_replay_batches of existing batches keep working.
 *
 * Synchronous.  The arrays are host memory (pageable is fine) and only read during the call.  stats_out (may be NULL)
 * receives the fields of fadegpu_align_pairs; h2d_bytes counts what was staged: the query offsets, the per-region
 * arrays and the query letters (no reference letters), plus the launch plan. */
typedef struct fadegpu_regions {
    const char *query; const int64_t *query_off;    /* [n+1] ASCII queries, concatenated */
    const int32_t *tid;                             /* [n] contig index of fadegpu_load_reference */
    const int64_t *start, *end;                     /* [n] 0-based half-open interval [start, end) on contig tid */
    const uint8_t *strand;                          /* [n] 0: the query as given, 1: its reverse complement */
} fadegpu_regions;                                  /* 48 bytes */

int fadegpu_align_regions(fadegpu_ctx *ctx, int64_t n_regions, const fadegpu_regions *in, int32_t max_ops,
                          fadegpu_pair_result *out, uint32_t *ops_out, fadegpu_stats *stats_out);

/* ---- Score-only Smith-Waterman of pairs and regions: score and end cell, no traceback ----
 * fadegpu_score_pairs / fadegpu_score_regions take exactly the inputs of fadegpu_align_pairs / fadegpu_align_regions
 * (without max_ops and ops_out) and validate them the same way: the same letter rules, the same FADEGPU_E_ARG cases and
 * messages naming the first offending pair or region (with the calling function's name), FADEGPU_E_STATE while a batch
 * of the ctx is in flight and, for regions, when no reference is loaded.  The ctx's scoring and FADEGPU_F_FORCE_GENERIC
 * apply, FADEGPU_F_TAGS_ONLY does not, and FADEGPU_F_NO_SHORTCUT changes no record.
 *
 * Records, in PAIR / REGION ORDER: score, end_query and end_ref equal, field for field, those of the traced call on the
 *   same input (P1-P3: the end cell is the first column, then the first row, holding the score); beg_query, beg_ref and
 *   n_ops are 0; flags hold only ALIGNED | GENERIC | OVERSIZE (FADEGPU_R_SCORE_ONLY keeps its annotate meaning and is
 *   not set).  Empty items give flags = 0 and a zero record; oversize items are not aligned, get FADEGPU_R_OVERSIZE and
 *   are counted in stats_out->n_oversize, as in the traced calls.
 * What it saves: the traceback rounds after the end cell is found (no traced block replay, no walk), the CIGAR spill
 *   and the ops copy home.
 * No side effects on batches: waited batches keep their results, and fadegpu_replay_kernels / fadegpu_replay_batches
 *   keep working.
 *
 * Synchronous; host arrays, only read during the call.  stats_out (may be NULL) receives the fields the traced calls
 * fill; d2h_bytes counts the 32-byte records and the binning histogram, no ops. */
int fadegpu_score_pairs(fadegpu_ctx *ctx, int64_t n_pairs, const fadegpu_pairs *in,
                        fadegpu_pair_result *out, fadegpu_stats *stats_out);
int fadegpu_score_regions(fadegpu_ctx *ctx, int64_t n_regions, const fadegpu_regions *in,
                          fadegpu_pair_result *out, fadegpu_stats *stats_out);

/* ---- Jobs: pair and region calls submitted now and collected later, several in flight on one ctx ----
 * A job is one fadegpu_align_* / fadegpu_score_* call split in two: fadegpu_submit_pairs / fadegpu_submit_regions stage
 *   the inputs, upload them and start the binning, then return; the ctx's helper thread plans and launches the kernels
 *   and queues the records home; fadegpu_job_wait blocks until they are there.  While the host stages job k+1, the GPU
 *   runs job k: the upload and binning of k+1 and the result copies of k-1 overlap the kernels of k.  The device work
 *   of a job is exactly the synchronous call's.
 * Results: after fadegpu_job_wait, fadegpu_job_results_view gives the records (in PAIR / REGION ORDER) and the ops,
 *   byte-identical to those of the synchronous call on the same input, ctx and flags: fadegpu_align_pairs /
 *   fadegpu_align_regions, or with FADEGPU_JOB_SCORE_ONLY fadegpu_score_pairs / fadegpu_score_regions (max_ops must then
 *   be 0).  Letters, empty and oversize items, max_ops / FADEGPU_R_OPS_TRUNC and the ctx's flags all follow that call.
 *   The view points into pinned memory owned by the job, where the result copies land; it stays valid until the job's
 *   next submit or its destroy.  While the job is in flight the view call fails with FADEGPU_E_STATE; before the
 *   first successful wait it gives n = 0.
 * Inputs: host arrays (pageable is fine), read only during the submit, which copies them into the job's pinned staging:
 *   the caller may overwrite them as soon as it returns.
 * Errors: the host-side checks run at submit, with the FADEGPU_E_ARG cases and messages of the synchronous call under
 *   the submit function's name; a refused submit leaves the job idle.  Errors found on the device (a query letter
 *   outside nt16, the internal "no result record" check) are returned by fadegpu_job_wait of that job only, with the
 *   synchronous messages; other jobs in flight are not affected.  FADEGPU_E_STATE: a submit of a job in flight, a wait
 *   on a job not submitted since its last wait, a region submit with no reference loaded, a job used with a ctx other
 *   than its own, a job submit while an annotate batch of the ctx is in flight, and fadegpu_submit /
 *   fadegpu_submit_compact / fadegpu_submit_inputs while a job of the ctx is in flight.  Batches and jobs are not in
 *   flight together; waited batches keep their results and fadegpu_replay_* keep working.
 * Synchronous calls made while jobs are in flight run after them, in submit order; their records do not change.
 * FADEGPU_F_SYNC_SUBMIT: a submit plans and launches on the calling thread, and device-found errors are returned by the
 *   submit itself (the job is then idle).
 * Stats (fadegpu_job_wait's stats_out, may be NULL): the fields the synchronous call fills.  n_*, cells, h2d_bytes,
 *   d2h_bytes and kernel_launches equal the synchronous call's; kernel_ms and total_ms come from the job's own events
 *   and can include overlapped work of neighbouring jobs; host_submit_ms is the wall time of the submit call.
 * Lifetime: fadegpu_job_destroy waits for the job first if it is in flight.  fadegpu_destroy waits for the jobs in
 *   flight and frees every job of the ctx (their handles are then invalid).  The helper thread is the ctx's one, started
 *   by its first queued submit of either kind and joined by fadegpu_destroy.  A ctx and its jobs are driven by one host
 *   thread at a time. */
typedef struct fadegpu_job fadegpu_job;             /* opaque: staging, device buffers and pinned records of one call */
int fadegpu_job_create(fadegpu_ctx *ctx, fadegpu_job **out);
void fadegpu_job_destroy(fadegpu_job *job);

#define FADEGPU_JOB_SCORE_ONLY 1u                  /* the fadegpu_score_* semantics: score and end cell, no traceback */
int fadegpu_submit_pairs(fadegpu_ctx *ctx, fadegpu_job *job, int64_t n_pairs, const fadegpu_pairs *in,
                         int32_t max_ops, uint32_t job_flags);
int fadegpu_submit_regions(fadegpu_ctx *ctx, fadegpu_job *job, int64_t n_regions, const fadegpu_regions *in,
                           int32_t max_ops, uint32_t job_flags);
int fadegpu_job_wait(fadegpu_ctx *ctx, fadegpu_job *job, fadegpu_stats *stats_out);

typedef struct fadegpu_job_results {
    int64_t n;                                      /* items of the last submit */
    const fadegpu_pair_result *records;             /* [n], item order; NULL when n == 0 */
    const uint32_t *ops;                            /* [n * max_ops], as ops_out of the synchronous call; NULL when
                                                       max_ops == 0 or n == 0 */
    int32_t max_ops, reserved;
} fadegpu_job_results;                              /* 32 bytes */
int fadegpu_job_results_view(const fadegpu_job *job, fadegpu_job_results *r);

/* INT16x2 ALU roofline denominator (SURVEY 8d): measures packed VIMNMX/VIADDMNMX issue rate.
 * ops_per_sec_out = packed (2-lane) instructions * 32 threads per second over the whole GPU. */
int fadegpu_measure_alu_peak(fadegpu_ctx *ctx, double *ops_per_sec_out, double *sm_clock_mhz_out);

#ifdef __cplusplus
}
#endif
#endif
