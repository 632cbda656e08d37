// fadegpu.cu -- C ABI (include/fadegpu.h) and host runtime of libfadegpu: contexts, packed
// reference upload, pinned batch buffers, queued submits, launch planning, streams, results.
//
// fadegpu_submit (the pinned view), fadegpu_submit_compact (gate bytes + compact records) and fadegpu_submit_inputs (the
// caller's arrays) check their arguments and the ctx's state (refuse_submit) and run one sequence (submit_batch).
// A device-binned submit is: (caller's arrays only: gather of the reads past the length floor, on the
// caller's thread) -> submit_device_binning on the ctx thread (the caller's with FADEGPU_F_SYNC_SUBMIT): upload,
// bin_classify_kernel (length floor of source/analysis.d:34, window arithmetic of source/analysis.d:45-59, histogram),
// launch plan from the histogram, bin_scatter_kernel (sorted descriptors), seq_pull_kernel (bases fetched from the
// pinned view), then fills on `stream` and traceback rounds on `tstream` over alternating scratch sets (three by
// default), result_index_kernel and the copies home on `stream3`.  FADEGPU_F_HOST_BINNING (submit_host_binning, on the
// caller's thread) evaluates the floor and the windows and sorts on the host, then plans from its histogram and runs
// the kernels on the same BinState.  A batch and a job are in flight (InFlight) from their submit to their wait.
// A pair or region call (fadegpu_align_* / fadegpu_score_*, or a job of fadegpu_submit_pairs / _regions) is a stage
// half on the caller's thread (stage_call: staging, upload, prep and classify on stream2) and a device half
// (launch_job: plan, scatter, kernels, results on stream3), which the ctx thread runs for jobs.  A device-binned submit
// and the two halves of a call run one binning sequence on their BinState.
// There is no CPU fallback: every compute entry point needs a CUDA device.
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <exception>
#include <mutex>
#include <thread>
#include <string>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif
#include "../../include/fadegpu.h"
#include "kernels.cuh"

using namespace fade;

static_assert(FADEGPU_MAX_OPS == OPS_CAP, "ABI ops capacity must match the kernels");
static_assert(sizeof(AlnOut) == 32 + 4 * OPS_CAP, "AlnOut layout");
static_assert(sizeof(AlnDesc) == 40, "AlnDesc layout");
static_assert(sizeof(PairResult) == sizeof(fadegpu_pair_result) && sizeof(fadegpu_pair_result) == 32, "fadegpu_pair_result layout");
static_assert(PAIR_R_OVERSIZE == FADEGPU_R_OVERSIZE, "oversize flag");

static thread_local std::string g_last_error;

constexpr int MAX_SETS = 4;

struct fadegpu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    fadegpu_params p{};
    SwConsts k{};
    // reference
    int32_t n_contigs = 0;
    std::vector<std::string> names;
    std::vector<int64_t> clen, coff;
    int64_t total_bases = 0, padded_bases = 0;
    uint32_t *d_two = nullptr, *d_n = nullptr, *d_x = nullptr;
    int64_t *d_xpos = nullptr;
    uint8_t *d_xchr = nullptr;
    int64_t n_x = 0;
    size_t ref_bytes = 0;
    // Fills run back to back on `stream`; the traceback rounds (and the generic kernel) of a launch
    // run on `tstream`, at higher priority, under the fill of the NEXT launch (of this batch or of
    // the following one): their many small, latency-bound grids take SM slots as fill blocks retire.
    // The scratch sets (three by default) take turns between consecutive launches, ordered by events.
    cudaStream_t tstream = nullptr;
    unsigned next_set = 0;
    struct ScratchSet {
        cudaEvent_t ev_fill = nullptr, ev_trace = nullptr;   // last fill / last traceback that used this scratch set
        bool used = false;
        uint32_t *d_ck = nullptr;        // fill checkpoints
        size_t ck_bytes = 0;
        uint8_t *d_gen = nullptr;        // generic kernel slots
        size_t gen_bytes = 0;
        unsigned int *d_cursor = nullptr;
        // traceback rounds: per-alignment state, request queues, trace tiles (sized per launch)
        uint8_t *d_trace = nullptr;
        size_t trace_bytes = 0;
        unsigned int *d_qcount = nullptr;
    } scratch[MAX_SETS];
    int n_sets = 3;                      // FADEGPU_SCRATCH_SETS=2..4 overrides (A/B measurements)
    uint32_t *d_alu = nullptr;
    int sm_count = 148;
    int host_threads = 1;
    cudaStream_t stream2 = nullptr;      // uploads + binning of the next batch while the previous one computes
    cudaStream_t stream3 = nullptr;      // result copies to the host, off the compute stream
    int64_t *d_clen = nullptr, *d_coff = nullptr;   // contig tables for the device-side binning
    std::string err;
    // asynchronous submits: fadegpu_submit queues the batch (fadegpu_submit_pairs / _regions the job), this thread
    // waits for the binning histogram, plans and launches; the caller goes on filling / reading other batches or jobs
    // a batch of n reads in input layout `mode` (SubmitMode; seq_bytes of compact inputs), or a job
    struct Queued { fadegpu_batch *b; int64_t n; int mode; int64_t seq_bytes; fadegpu_job *j; };
    std::thread worker;
    std::mutex q_mu;
    std::condition_variable q_cv, done_cv;
    std::deque<Queued> queue;
    bool worker_stop = false, worker_busy = false;
    std::mutex submit_mu;                 // one submit body at a time (they size shared scratch and order the streams)
    std::vector<fadegpu_batch *> batches; // the caller's batches (guarded by q_mu): fadegpu_align_pairs / _regions refuse to
                                          // run while one of them is in flight
    // fadegpu_align_* / fadegpu_score_* run on this job; fadegpu_job_create hands out the others (guarded by q_mu),
    // freed with the ctx.  jobs_in_flight counts those submitted and not yet waited for.
    fadegpu_job *sync_job = nullptr;
    std::vector<fadegpu_job *> jobs;
    int jobs_in_flight = 0;
};

// What a pair call and a region call do differently after the stage half of their shared body (stage_call), kept
// with the job until its device half has run.  Both stage the query offsets at byte 0 of the upload; the rest of the
// layout is the caller's.
struct StagedCall {
    const char *fn = nullptr, *item = nullptr;   // the call's and an item's name, for messages
    int64_t n = 0, qbytes = 0, n_over = 0;       // items, query letters, oversize items (counted by the host validation)
    int32_t max_ops = 0;
    bool score_only = false;                     // fadegpu_score_*: score and end cell, no traceback (max_ops is 0)
    size_t raw = 0;                              // bytes staged and uploaded
    size_t o_tbeg = 0, o_tend = 0;               // byte offsets of the int64 window bounds of every item in the upload
    // after the binning histogram is home: the reference the SW kernels read; counts its launches
    std::function<int(fadegpu_job *j, RefDev *ref, int *launches)> reference;
};

struct Launch {
    int R;            // 13/19/32 = packed kernels, 0 = generic list
    int aln_first, n_aln;
    int item_first, n_items;
    int tw_stride;
    int nblk_max;
    int qmax, tmax;   // generic only
};

// The device-binning core of an annotate batch and of a pair / region job: the binning inputs on the device, the
// histogram and the launch plan built from it, the sorted descriptors, the result records and the events that order
// them (alloc_bin_state, free_bin_state).
struct BinState {
    int64_t max_items = 0, max_seq_bytes = 0, cap_items = 0;   // (cap_items: warp items)
    // binning inputs; d_in_seq4: 16-byte slots that keep the source's alignment phase
    uint8_t *d_in_seq4 = nullptr;
    int64_t *d_in_seq_off = nullptr, *d_in_pos = nullptr;
    int32_t *d_in_lq = nullptr, *d_in_tid = nullptr, *d_in_alen = nullptr, *d_in_cl = nullptr, *d_in_cr = nullptr;
    // classify and scatter
    int32_t *d_key = nullptr, *d_tlen = nullptr, *d_hist = nullptr, *d_keybase = nullptr, *d_cursor = nullptr;
    int64_t *d_start = nullptr, *d_aln_start = nullptr, *d_src_off = nullptr;
    int32_t *d_over = nullptr, *h_over = nullptr;      // items left unaligned because their window exceeds 2^31 cells
    unsigned long long *d_stats = nullptr, *h_stats = nullptr;
    int32_t *h_hist = nullptr, *h_keybase = nullptr;   // (h_*: pinned)
    BinArgs ba{};                                      // the binning of the last submit (for replays); n == 0: none
    // launch plan, descriptors in sorted order, result records
    std::vector<Launch> plan;
    std::vector<int32_t> sorted_tlen;
    int64_t n_aln = 0, n_items = 0, n_generic = 0, scratch_bytes = 0;
    AlnDesc *d_aln = nullptr;
    WarpItem *h_items = nullptr, *d_items = nullptr;
    AlnOut *d_out = nullptr;
    uint32_t *d_flags = nullptr;
    uint2 *d_fillres = nullptr;
    // start of the uploads, first fill may start (compute stream), end of the kernels, results home,
    // inputs ready (upload stream), end of the last fill
    cudaEvent_t ev[6] = { nullptr, nullptr, nullptr, nullptr, nullptr, nullptr };
    cudaEvent_t ev_prep = nullptr, ev_ready = nullptr;   // histogram home / descriptors ready (upload stream)
    cudaEvent_t ev_kernels = nullptr;                    // end of the kernels (recorded on tstream)
};

// A batch's or a job's submit from the submit call to its wait (guarded by ctx->q_mu): `queued` while its device half
// waits for or runs on the ctx thread, which leaves that half's outcome here
struct InFlight {
    bool in_flight = false, queued = false;
    int rc = 0;
    std::string err;
};

// One pair or region call: its device-binning core, the staging of the raw inputs, the targets of a pair call packed
// as a reference of their own, the records and ops of the call in pinned memory (fadegpu_job_results_view).
// Everything grows with use.
struct fadegpu_job {
    fadegpu_ctx *ctx = nullptr;
    BinState bs;
    char *h_stage = nullptr, *d_raw = nullptr;          // pinned staging / device copy of offsets + ASCII
    size_t stage_bytes = 0, raw_bytes = 0;
    uint32_t *d_two = nullptr, *d_n = nullptr, *d_x = nullptr, *d_chunk_x = nullptr;
    size_t two_bytes = 0, n_bytes = 0, x_bytes = 0, chunk_bytes = 0;
    int64_t *d_xpos = nullptr, *d_clen = nullptr, *d_coff = nullptr;
    size_t xpos_bytes = 0, clen_bytes = 0, coff_bytes = 0;
    uint8_t *d_xchr = nullptr;
    size_t xchr_bytes = 0;
    uint32_t *d_spill = nullptr, *d_ops = nullptr;
    size_t spill_bytes = 0, ops_bytes = 0;
    fadegpu_pair_result *d_res = nullptr;
    size_t res_bytes = 0;
    int32_t *d_bad = nullptr, *h_bad = nullptr;         // lowest item index with a bad query letter (h_bad: pinned)
    fadegpu_pair_result *h_res = nullptr;               // pinned records and ops of the last submit
    uint32_t *h_ops = nullptr;
    size_t h_res_bytes = 0, h_ops_bytes = 0;
    // the call between its stage half and its wait: where the records go, what the device half needs, the stats
    StagedCall sc;
    PairArgs pa{};
    fadegpu_pair_result *out = nullptr;
    uint32_t *ops_out = nullptr;
    int n_prep = 0;
    int64_t h2d = 0;
    fadegpu_stats st{};
    int64_t n_res = -1;                                 // records of the last successful wait (-1: none)
    InFlight fl;
};

struct AlnTmp {       // a read that needs SW, captured in read order (sequential pass), before sorting
    int64_t start;    // window start inside the contig
    int64_t so;       // byte offset of its bases inside the caller's seq4
    int32_t read, tlen, qlen, tid, key;
    uint32_t clip_left, clip_right;
};

struct fadegpu_batch {
    fadegpu_ctx *ctx = nullptr;
    fadegpu_batch_view v{};
    BinState bs;
    AlnOut *h_out = nullptr;                   // [max_reads] pinned result records
    int64_t *h_aln_start = nullptr;            // [max_reads] pinned window start of each record
    int64_t n_reads = 0;
    fadegpu_stats st{};
    InFlight fl;
    // host binning: staging (pinned descriptors, allocated on first use; the bases go through h_c_seq4) and scratch
    AlnDesc *h_aln = nullptr;
    int64_t cap_seq = 0;
    std::vector<std::vector<AlnTmp>> tl_aln;   // per host thread
    std::vector<uint32_t> order;               // alignment indices sorted by (class, window length desc)
    int32_t *h_ridx = nullptr;                 // [max_reads] per read: index into the results, -1 = none
    std::vector<AlnTmp> all_aln;
    std::vector<int32_t> cnt;
    std::vector<int64_t> soff;
    // ---- device-side binning (submits from the pinned view) ----
    bool dev_binning = false;          // the last submit used it
    int32_t *d_ridx = nullptr;                         // per read: index into the results (built on the device, copied home)
    uint8_t *d_rflags = nullptr;
    uint8_t *d_gate = nullptr;                         // compact inputs: the one byte per read that is uploaded
    const uint4 *d_view_meta = nullptr;                // device address of the pinned view's 32-byte records
    // reads that pass the length floor, gathered by the host in read order (pinned, allocated on first use); h_c_seq4
    // also stages the bases of a host-binned submit
    uint8_t *h_c_seq4 = nullptr;
    int64_t *h_c_seq_off = nullptr, *h_c_pos = nullptr;
    int32_t *h_c_lq = nullptr, *h_c_tid = nullptr, *h_c_alen = nullptr, *h_c_cl = nullptr, *h_c_cr = nullptr, *h_c_read = nullptr;
    int32_t *d_in_read = nullptr;
    int64_t n_c = 0, seq_c = 0;                        // gathered reads / their sequence bytes
    bool pulled = false;
    const uint8_t *d_view_seq4 = nullptr;              // device address of the pinned view's seq4
    std::vector<int32_t> idx;                          // gather scratch
    AlnDesc *d_aln_scratch = nullptr;                  // replays scatter into these instead of the live descriptors
    int64_t *d_i64_scratch = nullptr;
};

extern "C" { static void drain_submits(fadegpu_ctx *c); }

namespace {

std::mutex g_err_mu;

int fail(fadegpu_ctx *ctx, int code, const std::string &msg)
{
    std::lock_guard<std::mutex> g(g_err_mu);
    if (ctx) ctx->err = msg;
    g_last_error = msg;
    return code;
}

int cuda_fail(fadegpu_ctx *ctx, cudaError_t e, const char *what)
{
    std::string m = std::string(what) + ": " + cudaGetErrorString(e);
    return fail(ctx, e == cudaErrorMemoryAllocation ? FADEGPU_E_OOM : FADEGPU_E_CUDA, m);
}

#define CU(ctx, call)                                              \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return cuda_fail(ctx, e__, #call); \
    } while (0)

template <typename T>
void free_host(T *&p) { if (p) cudaFreeHost(p); p = nullptr; }
template <typename T>
void free_dev(T *&p) { if (p) cudaFree(p); p = nullptr; }

void free_reference(fadegpu_ctx *c)
{
    free_dev(c->d_two); free_dev(c->d_n); free_dev(c->d_x); free_dev(c->d_xpos); free_dev(c->d_xchr);
    free_dev(c->d_clen); free_dev(c->d_coff);
    c->n_x = 0; c->ref_bytes = 0; c->n_contigs = 0; c->total_bases = c->padded_bases = 0;
    c->names.clear(); c->clen.clear(); c->coff.clear();
}

// an allocated core is freed once the ctx's streams are done with whatever they have queued
void free_bin_state(fadegpu_ctx *c, BinState &s)
{
    if (s.max_items) {
        cudaSetDevice(c->device);
        for (cudaStream_t q : { c->stream, c->tstream, c->stream2, c->stream3 }) if (q) cudaStreamSynchronize(q);
    }
    free_host(s.h_items); free_dev(s.d_aln); free_dev(s.d_items); free_dev(s.d_out); free_dev(s.d_flags); free_dev(s.d_fillres);
    free_dev(s.d_in_seq4); free_dev(s.d_in_seq_off); free_dev(s.d_in_pos); free_dev(s.d_in_lq); free_dev(s.d_in_tid);
    free_dev(s.d_in_alen); free_dev(s.d_in_cl); free_dev(s.d_in_cr); free_dev(s.d_key); free_dev(s.d_tlen); free_dev(s.d_start);
    free_dev(s.d_aln_start); free_dev(s.d_src_off); free_dev(s.d_hist); free_dev(s.d_keybase); free_dev(s.d_cursor);
    free_dev(s.d_over); free_host(s.h_over); free_dev(s.d_stats);
    free_host(s.h_hist); free_host(s.h_keybase); free_host(s.h_stats);
    for (cudaEvent_t e : { s.ev_prep, s.ev_ready, s.ev_kernels }) if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : s.ev) if (e) cudaEventDestroy(e);
    s = BinState{};
}

// Allocates the core and wires s.ba to its arrays (the caller sets the rest of s.ba before each classify); on failure
// nothing stays allocated.
int alloc_bin_state(fadegpu_ctx *c, BinState &s, int64_t max_items, int64_t max_seq_bytes)
{
    const size_t n = (size_t)max_items;
    s.cap_items = (max_items + 7) / 8 + 8;
    cudaError_t e = cudaSuccess;
    auto H = [&](auto **p, size_t bytes) { if (e == cudaSuccess) e = cudaHostAlloc((void **)p, std::max<size_t>(bytes, 16), cudaHostAllocDefault); };
    auto D = [&](auto **p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc((void **)p, std::max<size_t>(bytes, 16)); };
    H(&s.h_items, (size_t)s.cap_items * sizeof(WarpItem));
    D(&s.d_aln, n * sizeof(AlnDesc)); D(&s.d_items, (size_t)s.cap_items * sizeof(WarpItem));
    D(&s.d_out, n * sizeof(AlnOut)); D(&s.d_flags, n * 4);
    D(&s.d_fillres, (size_t)s.cap_items * 32 * sizeof(uint2));
    D(&s.d_in_seq4, (size_t)max_seq_bytes + 32 * n + 16); D(&s.d_in_seq_off, (n + 1) * 8); D(&s.d_in_pos, n * 8);
    D(&s.d_in_lq, n * 4); D(&s.d_in_tid, n * 4); D(&s.d_in_alen, n * 4); D(&s.d_in_cl, n * 4); D(&s.d_in_cr, n * 4);
    D(&s.d_key, n * 4); D(&s.d_tlen, n * 4); D(&s.d_start, n * 8); D(&s.d_aln_start, n * 8); D(&s.d_src_off, n * 8);
    D(&s.d_hist, (size_t)BIN_KEYS * 4); D(&s.d_keybase, (size_t)BIN_KEYS * 4); D(&s.d_cursor, (size_t)BIN_KEYS * 4);
    D(&s.d_over, (size_t)OVER_CAP * 4); H(&s.h_over, (size_t)OVER_CAP * 4); D(&s.d_stats, 128);
    H(&s.h_hist, (size_t)BIN_KEYS * 4); H(&s.h_keybase, (size_t)BIN_KEYS * 4); H(&s.h_stats, 128);
    if (e == cudaSuccess) e = cudaEventCreate(&s.ev_prep);
    if (e == cudaSuccess) e = cudaEventCreate(&s.ev_ready);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_kernels, cudaEventDisableTiming);
    for (auto &ev : s.ev) if (e == cudaSuccess) e = cudaEventCreate(&ev);
    if (e != cudaSuccess) {
        free_bin_state(c, s);
        return cuda_fail(c, e, "fadegpu_alloc_batch");   // (a job's core grows through the same allocation)
    }
    s.max_items = max_items; s.max_seq_bytes = max_seq_bytes;
    BinArgs &ba = s.ba;
    ba.seq4 = s.d_in_seq4; ba.seq_off = s.d_in_seq_off; ba.l_qseq = s.d_in_lq; ba.tid = s.d_in_tid; ba.pos = s.d_in_pos;
    ba.aligned_len = s.d_in_alen; ba.clip_left = s.d_in_cl; ba.clip_right = s.d_in_cr;
    ba.src_off = s.d_src_off; ba.over_list = s.d_over;
    ba.key = s.d_key; ba.tlen = s.d_tlen; ba.start = s.d_start; ba.hist = s.d_hist; ba.stats = s.d_stats;
    ba.keybase = s.d_keybase; ba.cursor = s.d_cursor; ba.aln = s.d_aln; ba.aln_start = s.d_aln_start;
    return 0;
}

// the job must not be queued; the ctx's streams are synchronised before anything is freed
void free_job(fadegpu_job *j)
{
    if (!j) return;
    free_bin_state(j->ctx, j->bs);
    free_host(j->h_stage); free_host(j->h_res); free_host(j->h_ops); free_host(j->h_bad);
    free_dev(j->d_raw); free_dev(j->d_two); free_dev(j->d_n); free_dev(j->d_x); free_dev(j->d_chunk_x);
    free_dev(j->d_xpos); free_dev(j->d_xchr); free_dev(j->d_clen); free_dev(j->d_coff); free_dev(j->d_spill);
    free_dev(j->d_ops); free_dev(j->d_res); free_dev(j->d_bad);
    delete j;
}

int upload_contig_tables(fadegpu_ctx *c)
{
    const size_t nb = std::max<size_t>(1, (size_t)c->n_contigs) * sizeof(int64_t);
    CU(c, cudaMalloc(&c->d_clen, nb)); CU(c, cudaMalloc(&c->d_coff, nb));
    if (c->n_contigs > 0) {
        CU(c, cudaMemcpy(c->d_clen, c->clen.data(), (size_t)c->n_contigs * 8, cudaMemcpyHostToDevice));
        CU(c, cudaMemcpy(c->d_coff, c->coff.data(), (size_t)c->n_contigs * 8, cudaMemcpyHostToDevice));
    }
    return 0;
}

RefDev ref_dev(const fadegpu_ctx *c)
{
    RefDev r;
    r.planes.two = c->d_two; r.planes.nmask = c->d_n; r.planes.xmask = c->d_x;
    r.xpos = c->d_xpos; r.xchr = c->d_xchr; r.n_x = c->n_x;
    return r;
}

size_t ck_words_of(int R) { return (size_t)(2 * R + 2); }

int ensure_dev(fadegpu_ctx *c, void **p, size_t *have, size_t bytes)
{
    if (bytes <= *have) return 0;
    if (*p) cudaFree(*p);               // (synchronises with whatever still uses it)
    *p = nullptr; *have = 0;
    CU(c, cudaMalloc(p, bytes));
    *have = bytes;
    return 0;
}

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// device bytes of the traceback-round scratch for a launch of n alignments of row class R
size_t trace_scratch_bytes(int R, int64_t n)
{
    return align256((size_t)n * sizeof(LaneCtl)) + 2 * align256((size_t)n * 8) +
           align256((size_t)((n + 1) / 2) * trace_tile_bytes(R));
}

constexpr int GEN_SLOTS_MAX = 8192;
constexpr size_t GEN_BUDGET = (size_t)4 << 30;

size_t gen_slot_bytes(int qmax, int tmax)
{
    size_t b = (size_t)8 * qmax + (((size_t)qmax + 15) & ~(size_t)15) + (size_t)qmax * tmax;
    return (b + 15) & ~(size_t)15;
}

// Launch plan from the sorted order: cls_first[rk] = first sorted position of row class rk (the
// generic list is rank N_ROW_CLASSES), s.sorted_tlen[pos] = window length at sorted position pos,
// s.h_stats[2..5] = the maxima of the binning.  Fills s.plan, s.h_items and grows the ctx scratch buffers.
int build_plan(fadegpu_ctx *c, BinState &s, const int64_t *cls_first)
{
    const int64_t n_aln = cls_first[N_ROW_CLASSES + 1];
    const int32_t *sorted_tlen = s.sorted_tlen.data();
    const int qmax_all = std::max(1, (int)s.h_stats[2]), tmax_all = std::max(1, (int)s.h_stats[3]);
    const int gen_qmax = std::max(1, (int)s.h_stats[4]), gen_tmax = std::max(1, (int)s.h_stats[5]);
    int64_t n_items = 0;
    size_t ck_needed = 0, gen_needed = 0, trace_needed = 0;
    s.plan.clear();
    s.n_generic = 0;
    for (int rk = 0; rk <= N_ROW_CLASSES; ++rk) {
        const int R = rk < N_ROW_CLASSES ? ROW_CLASSES[rk] : 0;
        const int64_t first_aln = cls_first[rk], last_aln = cls_first[rk + 1];
        if (last_aln <= first_aln) continue;
        if (R == 0) {
            Launch L{};
            L.R = 0; L.aln_first = (int)first_aln; L.n_aln = (int)(last_aln - first_aln); L.qmax = gen_qmax; L.tmax = gen_tmax;
            s.plan.push_back(L);
            gen_needed = std::max(gen_needed, gen_slot_bytes(gen_qmax, gen_tmax));
            s.n_generic += last_aln - first_aln;
            continue;
        }
        // warp items of 8 alignments; split into launches that fit the checkpoint scratch
        const size_t cw = ck_words_of(R);
        int64_t a0 = first_aln;
        while (a0 < last_aln) {
            Launch L{};
            L.R = R; L.aln_first = (int)a0; L.item_first = (int)n_items; L.qmax = qmax_all; L.tmax = tmax_all;
            size_t words = 0;
            int nblk_max = 1;
            int64_t a1 = a0;
            while (a1 < last_aln) {
                const int nblk = num_blocks(sorted_tlen[a1]);  // longest of the 8 (sorted descending)
                const size_t wds = (size_t)(nblk - 1) * cw * 32;
                if (a1 > a0 && (words + wds) * 4 > (size_t)c->p.scratch_bytes) break;
                if (n_items >= s.cap_items) return fail(c, FADEGPU_E_STATE, "fadegpu_submit: internal error (item capacity)");
                WarpItem &it = s.h_items[n_items++];
                it.ck_off = (int64_t)words;
                it.first = (int32_t)(a1 - a0);
                it.nblk = (int16_t)nblk;
                it.pad = 0;
                it.nsteps = sorted_tlen[a1] + FG - 1;
                words += wds;
                nblk_max = std::max(nblk_max, nblk);
                a1 = std::min<int64_t>(a1 + 8, last_aln);
            }
            L.n_aln = (int)(a1 - a0);
            L.n_items = (int)(n_items - L.item_first);
            L.tw_stride = tw_stride_for(nblk_max);
            L.nblk_max = nblk_max;
            ck_needed = std::max(ck_needed, words * 4);
            trace_needed = std::max(trace_needed, trace_scratch_bytes(R, L.n_aln));
            s.plan.push_back(L);
            a0 = a1;
        }
    }
    s.n_aln = n_aln; s.n_items = n_items;
    s.scratch_bytes = (int64_t)ck_needed;
    // a slot for wildcard alignments discovered on the device, sized for the largest problem
    if (n_aln > 0) gen_needed = std::max(gen_needed, gen_slot_bytes(qmax_all, tmax_all));
    for (int l = 0; l < (s.plan.empty() ? 0 : c->n_sets); ++l) {
        fadegpu_ctx::ScratchSet &ln = c->scratch[l];
        if (ck_needed) { int rc = ensure_dev(c, (void **)&ln.d_ck, &ln.ck_bytes, ck_needed); if (rc) return rc; }
        if (trace_needed) { int rc = ensure_dev(c, (void **)&ln.d_trace, &ln.trace_bytes, trace_needed); if (rc) return rc; }
        if (gen_needed) {
            const size_t want = std::min<size_t>(GEN_BUDGET, gen_needed * 1024);
            int rc = ensure_dev(c, (void **)&ln.d_gen, &ln.gen_bytes, std::max(want, gen_needed));
            if (rc) return rc;
        }
    }
    return 0;
}

// What a plan runs against: the resident reference (submits) or the packed targets of a pair call, the query bases its
// descriptors point into, whether alignments whose score rules out both predicates skip the traceback
// (FADEGPU_F_TAGS_ONLY), and the optional full-CIGAR spill rings (ops_cap words per alignment, in sorted order).
// end_only (score-only calls): no alignment is traced back; the traceback launches only find the end cell.
struct PlanTarget {
    RefDev ref;
    const uint8_t *seq;
    int tags_only;
    uint32_t *ops_spill;
    int ops_cap;
    bool end_only;
};

// an annotate batch's plan: both binnings stage its queries in the device mirror (d_in_seq4)
PlanTarget batch_target(const fadegpu_ctx *c, const fadegpu_batch *b)
{
    return PlanTarget{ ref_dev(c), b->bs.d_in_seq4, (c->p.flags & FADEGPU_F_TAGS_ONLY) ? 1 : 0, nullptr, 0, false };
}

// Queue every kernel of the plan: fills on c->stream (after `dep`: the inputs, or the start of a timed replay),
// traceback + generic on c->tstream, consecutive launches on alternating scratch sets.  On return bs.ev_kernels marks
// the end of the kernels; the caller joins it.  With stage timers every launch is synchronised.
int run_plan(fadegpu_ctx *c, BinState &bs, const PlanTarget &pt, float *fill_ms, float *trace_ms, float *gen_ms,
             int *launches, cudaEvent_t dep)
{
    const bool timed = fill_ms != nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr;
    if (timed) {
        CU(c, cudaEventCreate(&e0)); CU(c, cudaEventCreate(&e1)); CU(c, cudaEventCreate(&e2));
        *fill_ms = *trace_ms = *gen_ms = 0.f;
    }
    int nl = 0;
    cudaStream_t sf = c->stream, st = c->tstream;
    if (dep) CU(c, cudaStreamWaitEvent(sf, dep, 0));
    for (const Launch &L : bs.plan) {
        fadegpu_ctx::ScratchSet &ln = c->scratch[c->next_set++ % (unsigned)c->n_sets];
        // the scratch set is free again once its previous traceback is through
        if (ln.used) CU(c, cudaStreamWaitEvent(sf, ln.ev_trace, 0));
        ln.used = true;
        if (L.R != 0) {
            KernelArgs a;
            a.aln = bs.d_aln + L.aln_first;
            a.n_aln = L.n_aln;
            a.items = bs.d_items + L.item_first;
            a.n_items = L.n_items;
            a.seq = pt.seq;
            a.ref = pt.ref;
            a.ck = ln.d_ck;
            a.fillres = bs.d_fillres + (size_t)L.item_first * 32;
            a.aln_flags = bs.d_flags + L.aln_first;
            a.out = bs.d_out + L.aln_first;
            a.k = c->k;
            a.min_length = c->p.min_length;
            a.tw_stride = L.tw_stride;
            {
                uint8_t *p = ln.d_trace;
                a.state = reinterpret_cast<LaneCtl *>(p); p += align256((size_t)L.n_aln * sizeof(LaneCtl));
                a.queue[0] = reinterpret_cast<unsigned long long *>(p); p += align256((size_t)L.n_aln * 8);
                a.queue[1] = reinterpret_cast<unsigned long long *>(p); p += align256((size_t)L.n_aln * 8);
                a.tiles = reinterpret_cast<uint32_t *>(p);
                a.qcount = ln.d_qcount;
                a.round = 0;
                a.max_rounds = L.nblk_max + FG;   // each round scans one candidate block or walks one block
                a.tags_only = pt.tags_only;
            }
            a.ops_spill = pt.ops_spill ? pt.ops_spill + (size_t)L.aln_first * pt.ops_cap : nullptr;
            a.ops_cap = pt.ops_cap;
            CU(c, cudaMemsetAsync(a.aln_flags, 0, (size_t)L.n_aln * sizeof(uint32_t), sf));
            CU(c, cudaMemsetAsync(ln.d_qcount, 0, 2 * sizeof(unsigned int), sf));
            if (timed) CU(c, cudaEventRecord(e0, sf));
            CU(c, launch_fill(L.R, a, sf));
            if (timed) CU(c, cudaEventRecord(e1, sf));
            CU(c, cudaEventRecord(ln.ev_fill, sf));
            CU(c, cudaStreamWaitEvent(st, ln.ev_fill, 0));
            nl += 1;   // the fill kernel; launch_trace adds its own launches
            CU(c, launch_trace(L.R, a, pt.end_only, st, c->sm_count, &nl));
            // wildcard letters found by the packed kernels -> generic kernel over the flagged ones
            GenericArgs ga;
            ga.aln = a.aln; ga.n_aln = L.n_aln; ga.aln_flags = a.aln_flags; ga.seq = a.seq; ga.ref = a.ref;
            ga.out = a.out; ga.cursor = ln.d_cursor; ga.scratch = ln.d_gen;
            ga.qmax = L.qmax; ga.tmax = L.tmax;
            ga.slot_bytes = (int64_t)gen_slot_bytes(L.qmax, L.tmax);
            ga.n_slots = (int)std::max<size_t>(1, std::min<size_t>(GEN_SLOTS_MAX, ln.gen_bytes / (size_t)ga.slot_bytes));
            ga.chunk = 64;
            ga.open = c->p.gap_open; ga.extend = c->p.gap_extend; ga.match = c->p.match; ga.mismatch = c->p.mismatch;
            ga.min_length = c->p.min_length; ga.tags_only = pt.tags_only;
            ga.ops_spill = a.ops_spill; ga.ops_cap = a.ops_cap;
            if (timed) CU(c, cudaEventRecord(e2, st));
            CU(c, cudaMemsetAsync(ln.d_cursor, 0, sizeof(unsigned int), st));
            CU(c, launch_generic(ga, ga.n_slots, st));
            nl += 1;
            if (timed) {
                cudaEvent_t e3;
                CU(c, cudaEventCreate(&e3));
                CU(c, cudaEventRecord(e3, st));
                CU(c, cudaEventSynchronize(e3));
                float t;
                cudaEventElapsedTime(&t, e0, e1); *fill_ms += t;
                cudaEventElapsedTime(&t, e1, e2); *trace_ms += t;
                cudaEventElapsedTime(&t, e2, e3); *gen_ms += t;
                cudaEventDestroy(e3);
            }
            CU(c, cudaEventRecord(ln.ev_trace, st));
        } else {
            GenericArgs ga;
            ga.aln = bs.d_aln + L.aln_first; ga.n_aln = L.n_aln; ga.aln_flags = nullptr; ga.seq = pt.seq;
            ga.ref = pt.ref; ga.out = bs.d_out + L.aln_first; ga.cursor = ln.d_cursor; ga.scratch = ln.d_gen;
            ga.qmax = L.qmax; ga.tmax = L.tmax;
            ga.slot_bytes = (int64_t)gen_slot_bytes(L.qmax, L.tmax);
            ga.n_slots = (int)std::max<size_t>(1, std::min<size_t>(GEN_SLOTS_MAX, ln.gen_bytes / (size_t)ga.slot_bytes));
            ga.n_slots = std::min(ga.n_slots, std::max(L.n_aln, 1));
            ga.chunk = 1;
            ga.open = c->p.gap_open; ga.extend = c->p.gap_extend; ga.match = c->p.match; ga.mismatch = c->p.mismatch;
            ga.min_length = c->p.min_length; ga.tags_only = pt.tags_only;
            ga.ops_spill = pt.ops_spill ? pt.ops_spill + (size_t)L.aln_first * pt.ops_cap : nullptr;
            ga.ops_cap = pt.ops_cap;
            CU(c, cudaEventRecord(ln.ev_fill, sf));        // (orders tstream after dep and the set's previous traceback)
            CU(c, cudaStreamWaitEvent(st, ln.ev_fill, 0));
            if (timed) CU(c, cudaEventRecord(e0, st));
            CU(c, cudaMemsetAsync(ln.d_cursor, 0, sizeof(unsigned int), st));
            CU(c, launch_generic(ga, ga.n_slots, st));
            nl += 1;
            if (timed) {
                CU(c, cudaEventRecord(e1, st));
                CU(c, cudaEventSynchronize(e1));
                float t;
                cudaEventElapsedTime(&t, e0, e1); *gen_ms += t;
            }
            CU(c, cudaEventRecord(ln.ev_trace, st));
        }
    }
    if (timed) { cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2); }
    CU(c, cudaEventRecord(bs.ev[5], sf));          // end of the batch's last fill (timeline diagnostics)
    // every launch ends on tstream, in launch order: its tail is the batch's
    CU(c, cudaEventRecord(bs.ev_kernels, bs.plan.empty() ? sf : st));
    if (launches) *launches = nl;
    return 0;
}

// ---- The device-binning sequence of a device-binned submit and of a pair / region call, in the order the stream
// overlap of DESIGN.md 4.4 and 4.10 depends on: bin_zero, (caller's prep) bin_classify, (host waits for ev_prep)
// plan_from_histogram, bin_scatter, (caller records ev_ready) run_kernels. ----

// on stream2, before the classify kernel and anything else that counts into the stats
int bin_zero(fadegpu_ctx *c, BinState &s)
{
    CU(c, cudaMemsetAsync(s.d_hist, 0, (size_t)BIN_KEYS * 4, c->stream2));
    CU(c, cudaMemsetAsync(s.d_cursor, 0, (size_t)BIN_KEYS * 4, c->stream2));
    CU(c, cudaMemsetAsync(s.d_stats, 0, 128, c->stream2));
    return 0;
}

// Classify on stream2, then the histogram, the stats and `list_bytes` of the caller's list (a batch's over-list, a
// job's bad-letter slot) go home; ev_prep marks their arrival.
int bin_classify(fadegpu_ctx *c, BinState &s, void *h_list, const void *d_list, size_t list_bytes)
{
    cudaStream_t s2 = c->stream2;
    CU(c, launch_bin_classify(s.ba, c->sm_count, s2));
    CU(c, cudaMemcpyAsync(s.h_hist, s.d_hist, (size_t)BIN_KEYS * 4, cudaMemcpyDeviceToHost, s2));
    CU(c, cudaMemcpyAsync(s.h_stats, s.d_stats, 128, cudaMemcpyDeviceToHost, s2));
    CU(c, cudaMemcpyAsync(h_list, d_list, list_bytes, cudaMemcpyDeviceToHost, s2));
    CU(c, cudaEventRecord(s.ev_prep, s2));
    return 0;
}

// Launch plan from the binning histogram (s.h_hist, s.h_stats: from the device, or summed by the host binning) that
// classified n_aln alignments; also fills s.h_keybase, the first sorted position of every key, for the scatter.
int plan_from_histogram(fadegpu_ctx *c, BinState &s, int64_t n_aln)
{
    int64_t cls_first[N_ROW_CLASSES + 2];
    std::vector<int32_t> &stl = s.sorted_tlen;
    stl.resize((size_t)n_aln);
    int64_t run = 0;
    for (int rk = 0; rk <= N_ROW_CLASSES; ++rk) {
        cls_first[rk] = run;
        const int k0 = rk * KEYS_PER_CLASS, k1 = k0 + KEYS_PER_CLASS;
        for (int key = k0; key < k1; ++key) {
            const int32_t cnt = s.h_hist[key];
            s.h_keybase[key] = (int32_t)run;
            if (!cnt) continue;
            const int tl = rk == N_ROW_CLASSES ? (int)s.h_stats[5] : key_tlen(key - k0);
            std::fill(stl.begin() + run, stl.begin() + run + cnt, tl);
            run += cnt;
        }
    }
    cls_first[N_ROW_CLASSES + 1] = run;
    if (run != n_aln) return fail(c, FADEGPU_E_CUDA, "fadegpu_submit: internal error (histogram does not add up)");
    return build_plan(c, s, cls_first);
}

// After plan_from_histogram, on stream2: the keybase and the plan's warp items go up (BIN_KEYS * 4 +
// n_items * sizeof(WarpItem) bytes) and the scatter kernel writes the sorted descriptors
int bin_scatter(fadegpu_ctx *c, BinState &s)
{
    if (s.n_aln == 0) return 0;
    cudaStream_t s2 = c->stream2;
    CU(c, cudaMemcpyAsync(s.d_keybase, s.h_keybase, (size_t)BIN_KEYS * 4, cudaMemcpyHostToDevice, s2));
    if (s.n_items > 0)
        CU(c, cudaMemcpyAsync(s.d_items, s.h_items, (size_t)s.n_items * sizeof(WarpItem), cudaMemcpyHostToDevice, s2));
    CU(c, launch_bin_scatter(s.ba, c->sm_count, s2));
    return 0;
}

// Once the caller has recorded ev_ready on stream2: the compute stream waits for it and runs the plan against pt, and
// stream3 continues after the kernels; ev[1] and ev[2] bracket them.
int run_kernels(fadegpu_ctx *c, BinState &s, const PlanTarget &pt, int *launches)
{
    CU(c, cudaStreamWaitEvent(c->stream, s.ev_ready, 0));
    CU(c, cudaEventRecord(s.ev[1], c->stream));
    { int rc = run_plan(c, s, pt, nullptr, nullptr, nullptr, launches, s.ev_ready); if (rc) return rc; }
    CU(c, cudaStreamWaitEvent(c->stream3, s.ev_kernels, 0));
    CU(c, cudaEventRecord(s.ev[2], c->stream3));
    return 0;
}

}  // namespace

extern "C" {

int fadegpu_abi_version(void) { return FADEGPU_ABI_VERSION; }

int fadegpu_device_count(int *n)
{
    if (!n) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_device_count: null argument");
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) { *n = 0; return cuda_fail(nullptr, e, "cudaGetDeviceCount"); }
    *n = c;
    return FADEGPU_OK;
}

int fadegpu_default_params(fadegpu_params *p)
{
    if (!p) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_default_params: null argument");
    p->window_size = 300;  // source/app.d:18
    p->min_length = 5;     // source/app.d:17
    p->gap_open = 10;      // source/anno.d:36
    p->gap_extend = 2;
    p->match = 2;
    p->mismatch = -3;
    p->flags = 0;
    p->scratch_bytes = 0;
    p->host_threads = 0;
    p->reserved = 0;
    return FADEGPU_OK;
}

const char *fadegpu_last_error(const fadegpu_ctx *ctx)
{
    // copied under the lock into a buffer of the calling thread: the ctx thread may be rewriting ctx->err
    static thread_local std::string copy;
    std::lock_guard<std::mutex> g(g_err_mu);
    copy = ctx ? ctx->err : g_last_error;
    return copy.c_str();
}

int fadegpu_create(int device, const fadegpu_params *p, fadegpu_ctx **out)
{
    if (!out) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_create: null out");
    *out = nullptr;
    fadegpu_params pp;
    fadegpu_default_params(&pp);
    if (p) pp = *p;
    if (pp.gap_open < pp.gap_extend || pp.gap_extend <= 0 || pp.match <= 0 || pp.mismatch > 0 ||
        pp.match > 100 || pp.mismatch < -100 || pp.gap_open > 1000 || pp.window_size < 0)
        return fail(nullptr, FADEGPU_E_ARG, "fadegpu_create: unsupported scoring / window parameters");
    // the four streams of a ctx must be able to overlap: ask for more hardware queues than the default 8 unless the
    // process has chosen a value (only effective if no CUDA context exists yet)
    setenv("CUDA_DEVICE_MAX_CONNECTIONS", "32", 0);
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0)
        return fail(nullptr, FADEGPU_E_NODEV, std::string("fadegpu_create: no CUDA device (") +
                                                  (e != cudaSuccess ? cudaGetErrorString(e) : "count 0") + "); there is no CPU fallback");
    if (device < 0 || device >= n) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_create: bad device index");
    fadegpu_ctx *c = new (std::nothrow) fadegpu_ctx();
    if (!c) return fail(nullptr, FADEGPU_E_OOM, "fadegpu_create: out of host memory");
    c->device = device;
    c->p = pp;
    if (c->p.scratch_bytes <= 0) c->p.scratch_bytes = (int64_t)8 << 30;
    {
        int hw = 1;
#ifdef _OPENMP
        hw = std::max(1, omp_get_num_procs());
#endif
        c->host_threads = c->p.host_threads > 0 ? std::min(c->p.host_threads, 4 * hw) : hw;
    }
    c->k = make_consts(pp.gap_open, pp.gap_extend, pp.match, pp.mismatch);
    if (pp.flags & FADEGPU_F_NO_SHORTCUT) c->k.shortcut = 0;
    // Stream priorities (smaller = more urgent): uploads / binning / result copies (-2) above the traceback (-1) above
    // the fills (0).  Measured on 10 M reads (FADEGPU_PRIO="fill,trace,prep,out" overrides, A/B): this order 44.0 ms kernels /
    // 49.6 ms end to end; binning BELOW the fills (-1,-2,0,0) 44.3 / 52.7 (the next batch's inputs arrive late); all equal
    // 47.5 / 54.8 (the traceback rounds no longer slip under the next fill).
    int prio[4] = { 0, -1, -2, -2 };
    if (const char *pv = getenv("FADEGPU_PRIO")) sscanf(pv, "%d,%d,%d,%d", &prio[0], &prio[1], &prio[2], &prio[3]);
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio[0])) != cudaSuccess ||
        (e = cudaMalloc(&c->d_alu, 64)) != cudaSuccess ||
        (e = cudaStreamCreateWithPriority(&c->tstream, cudaStreamNonBlocking, prio[1])) != cudaSuccess ||
        (e = cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, prio[2])) != cudaSuccess ||
        (e = cudaStreamCreateWithPriority(&c->stream3, cudaStreamNonBlocking, prio[3])) != cudaSuccess ||
        (e = cudaDeviceGetAttribute(&c->sm_count, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess) {
        int rc = cuda_fail(nullptr, e, "fadegpu_create");
        delete c;
        return rc;
    }
    if (const char *ev = getenv("FADEGPU_SCRATCH_SETS")) c->n_sets = std::min(MAX_SETS, std::max(2, atoi(ev)));
    for (int l = 0; l < c->n_sets; ++l) {
        fadegpu_ctx::ScratchSet &ln = c->scratch[l];
        if ((e = cudaEventCreateWithFlags(&ln.ev_fill, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&ln.ev_trace, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaMalloc(&ln.d_cursor, sizeof(unsigned int))) != cudaSuccess ||
            (e = cudaMalloc(&ln.d_qcount, 2 * sizeof(unsigned int))) != cudaSuccess) {
            int rc = cuda_fail(nullptr, e, "fadegpu_create");
            fadegpu_destroy(c);
            return rc;
        }
    }
    *out = c;
    return FADEGPU_OK;
}

void fadegpu_destroy(fadegpu_ctx *c)
{
    if (!c) return;
    if (c->worker.joinable()) {
        { std::lock_guard<std::mutex> lk(c->q_mu); c->worker_stop = true; }
        c->q_cv.notify_all();
        c->worker.join();                 // finishes the queued submits first
    }
    cudaSetDevice(c->device);
    for (fadegpu_job *j : c->jobs) free_job(j);   // (each waits for the streams first)
    c->jobs.clear();
    free_job(c->sync_job);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->stream2) { cudaStreamSynchronize(c->stream2); cudaStreamDestroy(c->stream2); }
    if (c->stream3) { cudaStreamSynchronize(c->stream3); cudaStreamDestroy(c->stream3); }
    free_reference(c);
    if (c->tstream) { cudaStreamSynchronize(c->tstream); cudaStreamDestroy(c->tstream); }
    for (auto &ln : c->scratch) {
        if (ln.ev_fill) cudaEventDestroy(ln.ev_fill);
        if (ln.ev_trace) cudaEventDestroy(ln.ev_trace);
    }
    for (auto &ln : c->scratch) { free_dev(ln.d_ck); free_dev(ln.d_gen); free_dev(ln.d_cursor); free_dev(ln.d_trace); free_dev(ln.d_qcount); }
    free_dev(c->d_alu);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

int fadegpu_load_reference(fadegpu_ctx *c, int32_t n_contigs, const char *const *names,
                           const int64_t *lengths, const char *const *seqs)
{
    if (!c) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_load_reference: null ctx");
    if (n_contigs <= 0 || !lengths || !seqs) return fail(c, FADEGPU_E_ARG, "fadegpu_load_reference: bad arguments");
    drain_submits(c);
    std::lock_guard<std::mutex> submit_guard(c->submit_mu);
    CU(c, cudaSetDevice(c->device));
    { CU(c, cudaStreamSynchronize(c->stream)); CU(c, cudaStreamSynchronize(c->tstream)); }
    free_reference(c);
    c->n_contigs = n_contigs;
    int64_t off = 0, total = 0;
    for (int t = 0; t < n_contigs; ++t) {
        if (lengths[t] < 0 || !seqs[t]) { free_reference(c); return fail(c, FADEGPU_E_ARG, "fadegpu_load_reference: bad contig"); }
        c->names.emplace_back(names && names[t] ? names[t] : "");
        c->clen.push_back(lengths[t]);
        c->coff.push_back(off);
        total += lengths[t];
        off += (lengths[t] + 31) & ~(int64_t)31;  // every contig starts on a 32-base word boundary
    }
    c->total_bases = total;
    c->padded_bases = off + 32;
    const size_t w2 = (size_t)(c->padded_bases / 16), w1 = (size_t)(c->padded_bases / 32);
    std::vector<uint32_t> two, nm, xm;
    try { two.assign(w2, 0u); nm.assign(w1, 0u); xm.assign(w1, 0u); }
    catch (...) { free_reference(c); return fail(c, FADEGPU_E_OOM, "fadegpu_load_reference: out of host memory"); }
    // byte -> (2-bit code | 4 = N | 8 = wildcard)
    uint8_t lut[256];
    for (int i = 0; i < 256; ++i) lut[i] = 8;
    lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['T'] = lut['t'] = 2; lut['G'] = lut['g'] = 3;
    lut['N'] = lut['n'] = 4;
    for (int t = 0; t < n_contigs; ++t) {
        const unsigned char *s = reinterpret_cast<const unsigned char *>(seqs[t]);
        const int64_t len = lengths[t], base = c->coff[t];
        const int64_t nwords = (len + 31) / 32;
#pragma omp parallel for schedule(static) num_threads(std::max(1, c->host_threads))
        for (int64_t wd = 0; wd < nwords; ++wd) {
            uint32_t a0 = 0, a1 = 0, n = 0, x = 0;
            const int64_t p0 = wd * 32;
            const int lim = (int)std::min<int64_t>(32, len - p0);
            for (int b = 0; b < lim; ++b) {
                const uint8_t v = lut[s[p0 + b]];
                const uint32_t code = v & 3u;
                if (b < 16) a0 |= code << (2 * b); else a1 |= code << (2 * (b - 16));
                n |= (uint32_t)((v >> 2) & 1u) << b;
                x |= (uint32_t)((v >> 3) & 1u) << b;
            }
            const size_t gw = (size_t)((base + p0) / 32);
            two[2 * gw] = a0; two[2 * gw + 1] = a1; nm[gw] = n; xm[gw] = x;
        }
    }
    // sparse list of wildcard letters (upper-cased like source/analysis.d:63)
    std::vector<int64_t> xpos;
    std::vector<uint8_t> xchr;
    for (int t = 0; t < n_contigs; ++t) {
        const unsigned char *s = reinterpret_cast<const unsigned char *>(seqs[t]);
        const int64_t len = lengths[t], base = c->coff[t];
        for (int64_t wd = 0; wd * 32 < len; ++wd) {
            const uint32_t x = xm[(size_t)((base + wd * 32) / 32)];
            if (!x) continue;
            for (int b = 0; b < 32; ++b)
                if ((x >> b) & 1u) {
                    unsigned char ch = s[wd * 32 + b];
                    if (ch >= 'a' && ch <= 'z') ch = (unsigned char)(ch - 32);
                    xpos.push_back(base + wd * 32 + b);
                    xchr.push_back(ch);
                }
        }
    }
    c->n_x = (int64_t)xpos.size();
    cudaError_t e;
    if ((e = cudaMalloc(&c->d_two, w2 * 4)) != cudaSuccess || (e = cudaMalloc(&c->d_n, w1 * 4)) != cudaSuccess ||
        (e = cudaMalloc(&c->d_x, w1 * 4)) != cudaSuccess ||
        (e = cudaMalloc(&c->d_xpos, std::max<size_t>(1, xpos.size()) * 8)) != cudaSuccess ||
        (e = cudaMalloc(&c->d_xchr, std::max<size_t>(1, xchr.size()))) != cudaSuccess) {
        free_reference(c);
        return cuda_fail(c, e, "fadegpu_load_reference: cudaMalloc");
    }
    CU(c, cudaMemcpy(c->d_two, two.data(), w2 * 4, cudaMemcpyHostToDevice));
    CU(c, cudaMemcpy(c->d_n, nm.data(), w1 * 4, cudaMemcpyHostToDevice));
    CU(c, cudaMemcpy(c->d_x, xm.data(), w1 * 4, cudaMemcpyHostToDevice));
    if (!xpos.empty()) {
        CU(c, cudaMemcpy(c->d_xpos, xpos.data(), xpos.size() * 8, cudaMemcpyHostToDevice));
        CU(c, cudaMemcpy(c->d_xchr, xchr.data(), xchr.size(), cudaMemcpyHostToDevice));
    }
    c->ref_bytes = w2 * 4 + 2 * w1 * 4 + xpos.size() * 9;
    { int rc = upload_contig_tables(c); if (rc) return rc; }
    return FADEGPU_OK;
}

int fadegpu_share_reference(fadegpu_ctx *dst, const fadegpu_ctx *src)
{
    if (!dst || !src) return fail(dst, FADEGPU_E_ARG, "fadegpu_share_reference: null ctx");
    if (!src->d_two) return fail(dst, FADEGPU_E_STATE, "fadegpu_share_reference: source has no reference");
    drain_submits(dst);
    std::lock_guard<std::mutex> submit_guard(dst->submit_mu);
    CU(dst, cudaSetDevice(dst->device));
    { CU(dst, cudaStreamSynchronize(dst->stream)); CU(dst, cudaStreamSynchronize(dst->tstream)); }
    if (dst->device != src->device) {   // direct NVLink copies need peer access; without it the copy is staged through the host
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, dst->device, src->device) == cudaSuccess && can) {
            const cudaError_t pe = cudaDeviceEnablePeerAccess(src->device, 0);
            if (pe != cudaSuccess) cudaGetLastError();   // already enabled (or not possible): the copy still works
        }
    }
    free_reference(dst);
    dst->n_contigs = src->n_contigs; dst->names = src->names; dst->clen = src->clen; dst->coff = src->coff;
    dst->total_bases = src->total_bases; dst->padded_bases = src->padded_bases; dst->n_x = src->n_x;
    const size_t w2 = (size_t)(src->padded_bases / 16), w1 = (size_t)(src->padded_bases / 32);
    const size_t nx = std::max<size_t>(1, (size_t)src->n_x);
    CU(dst, cudaMalloc(&dst->d_two, w2 * 4)); CU(dst, cudaMalloc(&dst->d_n, w1 * 4)); CU(dst, cudaMalloc(&dst->d_x, w1 * 4));
    CU(dst, cudaMalloc(&dst->d_xpos, nx * 8)); CU(dst, cudaMalloc(&dst->d_xchr, nx));
    CU(dst, cudaMemcpyPeer(dst->d_two, dst->device, src->d_two, src->device, w2 * 4));
    CU(dst, cudaMemcpyPeer(dst->d_n, dst->device, src->d_n, src->device, w1 * 4));
    CU(dst, cudaMemcpyPeer(dst->d_x, dst->device, src->d_x, src->device, w1 * 4));
    if (src->n_x > 0) {
        CU(dst, cudaMemcpyPeer(dst->d_xpos, dst->device, src->d_xpos, src->device, (size_t)src->n_x * 8));
        CU(dst, cudaMemcpyPeer(dst->d_xchr, dst->device, src->d_xchr, src->device, (size_t)src->n_x));
    }
    dst->ref_bytes = src->ref_bytes;
    { int rc = upload_contig_tables(dst); if (rc) return rc; }
    return FADEGPU_OK;
}

int fadegpu_reference_info(const fadegpu_ctx *c, int32_t *n_contigs, int64_t *total_bases, int64_t *device_bytes)
{
    if (!c) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_reference_info: null ctx");
    if (n_contigs) *n_contigs = c->n_contigs;
    if (total_bases) *total_bases = c->total_bases;
    if (device_bytes) *device_bytes = (int64_t)c->ref_bytes;
    return FADEGPU_OK;
}

void fadegpu_free_batch(fadegpu_batch *b)
{
    if (!b) return;
    fadegpu_ctx *c = b->ctx;
    if (c) {
        std::unique_lock<std::mutex> lk(c->q_mu);
        c->done_cv.wait(lk, [&] { return !b->fl.queued; });
        c->batches.erase(std::remove(c->batches.begin(), c->batches.end(), b), c->batches.end());
    }
    free_bin_state(c, b->bs);
    fadegpu_batch_view &v = b->v;
    free_host(v.seq4); free_host(v.seq_off); free_host(v.l_qseq); free_host(v.tid); free_host(v.pos);
    free_host(v.aligned_len); free_host(v.clip_left); free_host(v.clip_right);
    free_host(v.gate); free_host(v.meta);
    free_host(v.flags); free_host(v.score); free_host(v.beg_query); free_host(v.end_query);
    free_host(v.beg_ref); free_host(v.end_ref); free_host(v.win_start); free_host(v.n_ops); free_host(v.ops);
    free_host(b->h_aln); free_host(b->h_out); free_host(b->h_ridx); free_host(b->h_aln_start);
    free_dev(b->d_ridx); free_dev(b->d_rflags); free_dev(b->d_gate);
    free_host(b->h_c_seq4); free_host(b->h_c_seq_off); free_host(b->h_c_pos); free_host(b->h_c_lq); free_host(b->h_c_tid);
    free_host(b->h_c_alen); free_host(b->h_c_cl); free_host(b->h_c_cr); free_host(b->h_c_read); free_dev(b->d_in_read);
    free_dev(b->d_aln_scratch); free_dev(b->d_i64_scratch);
    delete b;
}

int fadegpu_alloc_batch(fadegpu_ctx *c, int64_t max_reads, int64_t max_seq_bytes, fadegpu_batch **out)
{
    if (!c || !out) return fail(c, FADEGPU_E_ARG, "fadegpu_alloc_batch: null argument");
    *out = nullptr;
    if (max_reads <= 0 || max_seq_bytes <= 0 || max_reads > (int64_t)1 << 30)
        return fail(c, FADEGPU_E_ARG, "fadegpu_alloc_batch: bad sizes");
    CU(c, cudaSetDevice(c->device));
    fadegpu_batch *b = new (std::nothrow) fadegpu_batch();
    if (!b) return fail(c, FADEGPU_E_OOM, "fadegpu_alloc_batch: out of host memory");
    b->ctx = c;
    fadegpu_batch_view &v = b->v;
    v.max_reads = max_reads; v.max_seq_bytes = max_seq_bytes;
    const size_t n = (size_t)max_reads;
    b->cap_seq = max_seq_bytes + 16;
    cudaError_t e = cudaSuccess;
    auto H = [&](auto **p, size_t bytes) { if (e == cudaSuccess) e = cudaHostAlloc((void **)p, std::max<size_t>(bytes, 16), cudaHostAllocDefault); };
    auto D = [&](auto **p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc((void **)p, std::max<size_t>(bytes, 16)); };
    H(&v.seq4, (size_t)max_seq_bytes + 16); H(&v.seq_off, (n + 1) * 8); H(&v.l_qseq, n * 4); H(&v.tid, n * 4);
    H(&v.pos, n * 8); H(&v.aligned_len, n * 4); H(&v.clip_left, n * 4); H(&v.clip_right, n * 4);
    H(&v.flags, n); H(&v.gate, n); H(&v.meta, n * sizeof(fadegpu_read_meta));
    if (!(c->p.flags & FADEGPU_F_NO_SCATTER)) {   // the per-read output arrays are only filled without NO_SCATTER
        H(&v.score, n * 4); H(&v.beg_query, n * 4); H(&v.end_query, n * 4); H(&v.beg_ref, n * 4);
        H(&v.end_ref, n * 4); H(&v.win_start, n * 8); H(&v.n_ops, n * 4); H(&v.ops, n * 4 * FADEGPU_MAX_OPS);
    }
    H(&b->h_out, n * sizeof(AlnOut)); H(&b->h_ridx, n * 4); H(&b->h_aln_start, n * 8);
    // the host staging (h_aln, h_c_*) is allocated on first use
    // device-side binning beyond the core: gathered read indices, per-read result index and flags, gate bytes
    D(&b->d_in_read, n * 4); D(&b->d_ridx, n * 4); D(&b->d_rflags, n); D(&b->d_gate, n);
    if (e == cudaSuccess) e = cudaHostGetDevicePointer((void **)&b->d_view_seq4, v.seq4, 0);
    if (e == cudaSuccess) e = cudaHostGetDevicePointer((void **)&b->d_view_meta, v.meta, 0);
    const int rc = e != cudaSuccess ? cuda_fail(c, e, "fadegpu_alloc_batch") : alloc_bin_state(c, b->bs, max_reads, max_seq_bytes);
    if (rc) { fadegpu_free_batch(b); return rc; }
    { std::lock_guard<std::mutex> lk(c->q_mu); c->batches.push_back(b); }
    *out = b;
    return FADEGPU_OK;
}

int fadegpu_get_batch_view(fadegpu_batch *b, fadegpu_batch_view *view)
{
    if (!b || !view) return fail(b ? b->ctx : nullptr, FADEGPU_E_ARG, "fadegpu_get_batch_view: null argument");
    *view = b->v;
    return FADEGPU_OK;
}

// FADEGPU_F_HOST_BINNING, on the calling thread under submit_mu: the host evaluates the length floor and the windows
// (analysis.d:34,45-59), sorts by (row class, window length) and gathers descriptors and bases, fills the batch's
// histogram and stats as the classify kernel would and plans from them; uploads and kernels follow on the batch's
// BinState as for a device-binned submit.  The independent reference for the classify kernel's arithmetic.
static int submit_host_binning(fadegpu_ctx *c, fadegpu_batch *b, int64_t n, const fadegpu_inputs *in)
{
    if (!b->h_aln) CU(c, cudaHostAlloc((void **)&b->h_aln, (size_t)b->v.max_reads * sizeof(AlnDesc), cudaHostAllocDefault));
    if (!b->h_c_seq4) CU(c, cudaHostAlloc((void **)&b->h_c_seq4, (size_t)b->cap_seq + 16, cudaHostAllocDefault));
    BinState &bs = b->bs;
    b->n_reads = n;
    bs.plan.clear();
    bs.ba.n = 0;   // nothing binned on the device: replays run the plan only
    b->dev_binning = false;
    memset(&b->st, 0, sizeof(b->st));
    b->st.n_reads = n;

    // ---- 1. which reads need SW, their windows (analysis.d:34,45-59) and size class ----
    const auto t_begin = std::chrono::steady_clock::now();
    auto ms_since = [](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    const int nthr = std::max(1, c->host_threads);   // explicit: OMP_NUM_THREADS (torchrun sets it to 1) is ignored
    b->st.host_threads = nthr;
    if ((int)b->tl_aln.size() < nthr) b->tl_aln.resize((size_t)nthr);
    const uint32_t floor_u = (uint32_t)c->p.min_length;  // uint <= int compare of analysis.d:34
    const int64_t W = c->p.window_size;
    const int64_t seq_total = n > 0 ? in->seq_off[n] : 0;
    int64_t cells = 0, n_over = 0, seq_bytes = 0;
    int bad = 0, qmax = 0, tmax = 0, qmax_g = 0, tmax_g = 0;
#pragma omp parallel num_threads(nthr) reduction(+ : cells, seq_bytes) reduction(| : bad) reduction(max : qmax, tmax, qmax_g, tmax_g)
    {
        int tix = 0, tn = 1;
#ifdef _OPENMP
        tix = omp_get_thread_num(); tn = omp_get_num_threads();
#endif
        std::vector<AlnTmp> &loc = b->tl_aln[(size_t)tix];
        loc.clear();
        const int64_t lo = n * tix / tn, hi = n * (tix + 1) / tn;
        for (int64_t r = lo; r < hi; ++r) {
            const uint32_t cl = (uint32_t)in->clip_left[r], cr = (uint32_t)in->clip_right[r];
            const bool need = (cl != 0 && !(cl <= floor_u)) || (cr != 0 && !(cr <= floor_u));
            if (!need) continue;
            const int32_t tid = in->tid[r];
            const int32_t ql = in->l_qseq[r];
            if (tid < 0 || tid >= c->n_contigs || ql <= 0) continue;
            const int64_t so = in->seq_off[r];
            if (so < 0 || so + (ql + 1) / 2 > seq_total) { bad = 1; continue; }
            int64_t start = in->pos[r] - W;
            if (start < 0) start = 0;
            int64_t end = in->pos[r] + (int64_t)in->aligned_len[r] + W;
            if (end > c->clen[tid]) end = c->clen[tid];
            if (end <= start) continue;                              // empty window: nothing to align
            // a window this large (spliced alignment spanning megabases) would need a multi-GB trace
            // for ONE read in the reference as well; refuse it loudly instead of running for hours
            if (end - start > 0x7fffffff || (end - start) * (int64_t)ql > ((int64_t)1 << 31)) {
                // (the reference would need a multi-GB trace for this ONE read) left unaligned and reported
#pragma omp critical(fadegpu_oversize)
                { if (n_over < OVER_CAP) bs.h_over[n_over] = (int32_t)r; ++n_over; }
                continue;
            }
            const int tlen = (int)(end - start);
            const int rk = bin_rank(ql, tlen, c->p.flags & FADEGPU_F_FORCE_GENERIC);
            // key = class rank (row classes, then the generic list) then descending window length (generic: input order)
            loc.push_back(AlnTmp{ start, so, (int32_t)r, tlen, ql, tid, bin_key(rk, tlen), cl, cr });
            cells += (int64_t)ql * tlen;
            seq_bytes += (ql + 1) / 2;
            qmax = std::max(qmax, ql); tmax = std::max(tmax, tlen);
            if (rk == N_ROW_CLASSES) { qmax_g = std::max(qmax_g, ql); tmax_g = std::max(tmax_g, tlen); }
        }
    }
    if (bad & 1) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: seq_off / l_qseq inconsistent");
    b->st.cells = cells;
    b->st.n_oversize = n_over;
    b->st.host_classify_ms = ms_since(t_begin);
    // (they go up into bs.d_in_seq4, which holds max_seq_bytes + 32 n + 16 bytes)
    if (seq_bytes > b->cap_seq) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: read bases exceed max_seq_bytes");
    const auto t_sort = std::chrono::steady_clock::now();

    // ---- 2. bin by class, counting sort by window length (longest first), launch plan ----
    int64_t n_aln = 0;
    for (int t = 0; t < nthr; ++t) n_aln += (int64_t)b->tl_aln[(size_t)t].size();
    std::vector<AlnTmp> &all = b->all_aln;
    std::vector<uint32_t> &order = b->order;
    all.resize((size_t)n_aln);
    order.resize((size_t)n_aln);
    // parallel, stable counting sort of the INDICES: per-thread histograms over the thread's own
    // (read-ordered) slice, their sum planned like a device histogram, per-thread start of every key
    // (key, then thread), per-thread scatter
    const int KEYS = BIN_KEYS;
    std::vector<int32_t> &hist = b->cnt;
    hist.resize((size_t)nthr * (size_t)(KEYS + 1));
    std::vector<int64_t> toff((size_t)nthr + 1, 0);
    for (int t = 0; t < nthr; ++t) toff[(size_t)t + 1] = toff[(size_t)t] + (int64_t)b->tl_aln[(size_t)t].size();
#pragma omp parallel num_threads(nthr)
    {
        int t = 0;
#ifdef _OPENMP
        t = omp_get_thread_num();
#endif
        if (t < nthr) {
            const auto &loc = b->tl_aln[(size_t)t];
            int32_t *h = hist.data() + (size_t)t * (size_t)(KEYS + 1);
            memset(h, 0, (size_t)(KEYS + 1) * sizeof(int32_t));
            if (!loc.empty()) memcpy(all.data() + toff[(size_t)t], loc.data(), loc.size() * sizeof(AlnTmp));
            for (const AlnTmp &a : loc) ++h[a.key];
        }
    }
#pragma omp parallel for schedule(static) num_threads(nthr)
    for (int key = 0; key < KEYS; ++key) {
        int32_t sum = 0;
        for (int t = 0; t < nthr; ++t) sum += hist[(size_t)t * (size_t)(KEYS + 1) + (size_t)key];
        bs.h_hist[key] = sum;
    }
    memset(bs.h_stats, 0, 128);   // the layout bin_classify_kernel writes
    bs.h_stats[0] = (unsigned long long)cells; bs.h_stats[1] = (unsigned long long)n_aln;
    bs.h_stats[2] = qmax; bs.h_stats[3] = tmax; bs.h_stats[4] = qmax_g; bs.h_stats[5] = tmax_g;
    { int rc = plan_from_histogram(c, bs, n_aln); if (rc) return rc; }
    b->st.n_aligned = n_aln; b->st.n_generic = bs.n_generic; b->st.scratch_bytes = bs.scratch_bytes;
    for (int key = 0; key < KEYS; ++key) {
        if (!bs.h_hist[key]) continue;
        int32_t run = bs.h_keybase[key];
        for (int t = 0; t < nthr; ++t) {
            int32_t &hv = hist[(size_t)t * (size_t)(KEYS + 1) + (size_t)key];
            const int32_t c0 = hv;
            hv = run;
            run += c0;
        }
    }
#pragma omp parallel num_threads(nthr)
    {
        int t = 0;
#ifdef _OPENMP
        t = omp_get_thread_num();
#endif
        if (t < nthr) {
            int32_t *h = hist.data() + (size_t)t * (size_t)(KEYS + 1);
            const int64_t o0 = toff[(size_t)t], o1 = toff[(size_t)t + 1];
            for (int64_t kx = o0; kx < o1; ++kx) order[(size_t)h[all[(size_t)kx].key]++] = (uint32_t)kx;
        }
    }

    b->st.host_sort_ms = ms_since(t_sort);
    const auto t_gather = std::chrono::steady_clock::now();
    // ---- 3. descriptors + gathered read bases ----
    std::vector<int64_t> &soff = b->soff;
    soff.resize((size_t)n_aln);
    for (int64_t kx = 0, o = 0; kx < n_aln; ++kx) {
        soff[(size_t)kx] = o;
        o += (all[order[(size_t)kx]].qlen + 1) / 2;
    }
#pragma omp parallel for schedule(static) num_threads(nthr)
    for (int64_t kx = 0; kx < n_aln; ++kx) {
        const AlnTmp &a = all[order[(size_t)kx]];
        if (kx + 8 < n_aln) {   // the bases sit at random places of the caller's array: prefetch ahead
            const uint8_t *pf = in->seq4 + all[order[(size_t)kx + 8]].so;
            __builtin_prefetch(pf); __builtin_prefetch(pf + 64);
        }
        AlnDesc &d = b->h_aln[kx];
        const int ql = a.qlen;
        d.gstart = c->coff[a.tid] + a.start;
        d.seq_off = soff[(size_t)kx];
        d.tlen = a.tlen;
        d.qlen = ql;
        d.clip_left = a.clip_left;
        d.clip_right = a.clip_right;
        d.read = a.read;
        d.pad = 0;
        b->h_aln_start[kx] = a.start;
        memcpy(b->h_c_seq4 + d.seq_off, in->seq4 + a.so, (size_t)((ql + 1) / 2));
    }

    b->st.host_gather_ms = ms_since(t_gather);
    const int64_t n_items = bs.n_items;

    // ---- 4. queue copies and kernels ----
    // copies in on stream2, kernels on the compute stream, copies out on stream3: the DMA of one
    // batch overlaps the kernels of its neighbours
    CU(c, cudaEventRecord(bs.ev[0], c->stream2));
    if (n_aln > 0) {
        CU(c, cudaMemcpyAsync(bs.d_aln, b->h_aln, (size_t)n_aln * sizeof(AlnDesc), cudaMemcpyHostToDevice, c->stream2));
        if (n_items > 0)
            CU(c, cudaMemcpyAsync(bs.d_items, bs.h_items, (size_t)n_items * sizeof(WarpItem), cudaMemcpyHostToDevice, c->stream2));
        CU(c, cudaMemcpyAsync(bs.d_in_seq4, b->h_c_seq4, (size_t)seq_bytes, cudaMemcpyHostToDevice, c->stream2));
    }
    b->st.h2d_bytes = n_aln * (int64_t)sizeof(AlnDesc) + n_items * (int64_t)sizeof(WarpItem) + seq_bytes;
    CU(c, cudaEventRecord(bs.ev_ready, c->stream2));
    int nl = 0;
    { int rc = run_kernels(c, bs, batch_target(c, b), &nl); if (rc) return rc; }
    b->st.kernel_launches = nl;
    if (n_aln > 0)
        CU(c, cudaMemcpyAsync(b->h_out, bs.d_out, (size_t)n_aln * sizeof(AlnOut), cudaMemcpyDeviceToHost, c->stream3));
    b->st.d2h_bytes = n_aln * (int64_t)sizeof(AlnOut);
    CU(c, cudaEventRecord(bs.ev[3], c->stream3));
    b->st.host_submit_ms = ms_since(t_begin);
    return FADEGPU_OK;
}

// Stage A of a submit: the host keeps the reads that pass the length floor (analysis.d:34, unsigned
// compare) and copies their bases and per-read fields, in read order, into pinned staging.  One
// streaming pass over clip_left / clip_right plus ~110 B per kept read; the window arithmetic, the
// sort by window length and everything after it run on the device (stage B).
static int gather_reads(fadegpu_ctx *c, fadegpu_batch *b, int64_t n, const fadegpu_inputs &in)
{
    const auto t0 = std::chrono::steady_clock::now();
    if (!b->h_c_read) {   // (a host-binned submit may have allocated h_c_seq4 already)
        const size_t m = (size_t)b->v.max_reads;
        auto H = [&](auto **p, size_t bytes) { return *p ? cudaSuccess : cudaHostAlloc((void **)p, std::max<size_t>(bytes, 16), cudaHostAllocDefault); };
        CU(c, H(&b->h_c_seq4, (size_t)b->cap_seq + 16)); CU(c, H(&b->h_c_seq_off, (m + 1) * 8)); CU(c, H(&b->h_c_pos, m * 8));
        CU(c, H(&b->h_c_lq, m * 4)); CU(c, H(&b->h_c_tid, m * 4)); CU(c, H(&b->h_c_alen, m * 4));
        CU(c, H(&b->h_c_cl, m * 4)); CU(c, H(&b->h_c_cr, m * 4)); CU(c, H(&b->h_c_read, m * 4));
    }
    const uint32_t floor_u = (uint32_t)c->p.min_length;
    const int T = (int)std::max<int64_t>(1, std::min<int64_t>(std::min(c->host_threads, 64), n / 4096));
    std::vector<int64_t> cnt((size_t)T + 1, 0), bytes((size_t)T + 1, 0);
    b->idx.resize((size_t)std::max<int64_t>(n, 1));
    int32_t *const idx = b->idx.data();
    // pass 1, branch-free: indices of the reads that need SW (compacted per thread range) and their bytes
#pragma omp parallel for schedule(static, 1) num_threads(T)
    for (int t = 0; t < T; ++t) {
        const int64_t r0 = n * t / T, r1 = n * (t + 1) / T;
        int64_t k = 0, by = 0;
        int32_t *out = idx + r0;
        for (int64_t r = r0; r < r1; ++r) {
            const uint32_t cl = (uint32_t)in.clip_left[r], cr = (uint32_t)in.clip_right[r];
            const int nd = (int)(cl > floor_u) | (int)(cr > floor_u);     // == (cl != 0 && !(cl <= floor)) || ...
            const int ql = in.l_qseq[r];
            out[k] = (int32_t)r;
            k += nd;
            by += nd ? (int64_t)((ql > 0 ? ql + 1 : 0) >> 1) : 0;
        }
        cnt[(size_t)t + 1] = k; bytes[(size_t)t + 1] = by;
    }
    for (int t = 0; t < T; ++t) { cnt[(size_t)t + 1] += cnt[(size_t)t]; bytes[(size_t)t + 1] += bytes[(size_t)t]; }
    if (bytes[(size_t)T] > b->cap_seq) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: sequence bytes exceed max_seq_bytes");
    // pass 2: copy the kept reads; the loads are scattered over seven arrays, so prefetch ahead
    int bad = 0;
#pragma omp parallel for schedule(static, 1) reduction(| : bad) num_threads(T)
    for (int t = 0; t < T; ++t) {
        const int32_t *ix = idx + n * t / T;
        const int64_t m = cnt[(size_t)t + 1] - cnt[(size_t)t];
        int64_t k = cnt[(size_t)t], by = bytes[(size_t)t];
        constexpr int D = 12;
        for (int64_t i = 0; i < m; ++i) {
            if (i + 2 * D < m) {
                const int64_t rr = ix[i + 2 * D];
                __builtin_prefetch(&in.seq_off[rr]); __builtin_prefetch(&in.pos[rr]); __builtin_prefetch(&in.tid[rr]);
                __builtin_prefetch(&in.aligned_len[rr]); __builtin_prefetch(&in.l_qseq[rr]);
            }
            if (i + D < m) {
                const uint8_t *p = in.seq4 + in.seq_off[ix[i + D]];
                __builtin_prefetch(p); __builtin_prefetch(p + 64);
            }
            const int64_t r = ix[i];
            const int ql = in.l_qseq[r];
            const int64_t nb = ql > 0 ? (ql + 1) / 2 : 0;
            if (in.seq_off[r] < 0 || (nb > 0 && in.seq_off[r + 1] - in.seq_off[r] < nb)) bad = 1;
            else memcpy(b->h_c_seq4 + by, in.seq4 + in.seq_off[r], (size_t)nb);
            b->h_c_seq_off[k] = by; b->h_c_pos[k] = in.pos[r];
            b->h_c_lq[k] = ql; b->h_c_tid[k] = in.tid[r]; b->h_c_alen[k] = in.aligned_len[r];
            b->h_c_cl[k] = in.clip_left[r]; b->h_c_cr[k] = in.clip_right[r]; b->h_c_read[k] = (int32_t)r;
            ++k; by += nb;
        }
    }
    if (bad) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: seq_off / l_qseq inconsistent");
    b->n_c = cnt[(size_t)T]; b->seq_c = bytes[(size_t)T];
    b->h_c_seq_off[b->n_c] = b->seq_c;
    b->n_reads = n;
    b->st.host_gather_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    b->st.host_threads = T;
    return FADEGPU_OK;
}

// Where a queued submit finds its inputs
enum SubmitMode : int {
    MODE_GATHERED = 0,   // fadegpu_submit_inputs: the reads past the length floor, staged by gather_reads
    MODE_VIEW = 1,       // fadegpu_submit: the seven input arrays of the pinned view are DMA'd as they are (36 B / read)
    MODE_COMPACT = 2     // fadegpu_submit_compact: one gate byte per read is DMA'd, the GPU fetches the rest it needs
};

// Stage B: the inputs go to the GPU, a classify kernel applies the length floor (analysis.d:34) and the window
// arithmetic (analysis.d:45-59) and histograms the reads that need SW by (row class, window length), the host
// turns the 96 KB histogram into the launch plan, a scatter kernel writes the sorted descriptors, the GPU pulls the
// bases of those reads from the pinned view, the SW kernels follow on the compute stream and the result records
// come back on a third stream.  Uploads and binning of batch k+1 overlap the kernels of batch k.
static int submit_device_binning(fadegpu_ctx *c, fadegpu_batch *b, int64_t n_reads, int mode, int64_t seq_bytes)
{
    const auto t_begin = std::chrono::steady_clock::now();
    auto ms_since = [](std::chrono::steady_clock::time_point t0) {
        return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    };
    const bool pull = mode != MODE_GATHERED;
    BinState &bs = b->bs;
    b->n_reads = n_reads;
    bs.plan.clear();
    b->dev_binning = true;
    {
        const float g = pull ? 0.f : b->st.host_gather_ms; const int32_t th = pull ? 1 : b->st.host_threads;
        memset(&b->st, 0, sizeof(b->st));
        b->st.host_gather_ms = g; b->st.host_threads = th;
    }
    b->st.n_reads = n_reads;
    bs.n_aln = 0; bs.n_items = 0; bs.ba.n = 0;
    cudaStream_t s2 = c->stream2;
    CU(c, cudaEventRecord(bs.ev[0], s2));
    b->pulled = pull;
    const fadegpu_batch_view &v = b->v;
    const int64_t n = pull ? n_reads : b->n_c;
    const int64_t seq_total = mode == MODE_COMPACT ? seq_bytes : mode == MODE_VIEW ? (n > 0 ? v.seq_off[n] : 0) : b->seq_c;
    int64_t n_aln = 0, up_bytes = 0;
    memset(bs.h_stats, 0, 128);
    if (n > 0) {
        auto up = [&](void *d, const void *h, size_t bytes) { up_bytes += (int64_t)bytes; return cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, s2); };
        if (mode == MODE_COMPACT) CU(c, up(b->d_gate, v.gate, (size_t)n));
        else {
            if (!pull) CU(c, up(bs.d_in_seq4, b->h_c_seq4, (size_t)seq_total));
            CU(c, up(bs.d_in_seq_off, pull ? v.seq_off : b->h_c_seq_off, (size_t)(n + 1) * 8));
            CU(c, up(bs.d_in_lq, pull ? v.l_qseq : b->h_c_lq, (size_t)n * 4)); CU(c, up(bs.d_in_tid, pull ? v.tid : b->h_c_tid, (size_t)n * 4));
            CU(c, up(bs.d_in_pos, pull ? v.pos : b->h_c_pos, (size_t)n * 8)); CU(c, up(bs.d_in_alen, pull ? v.aligned_len : b->h_c_alen, (size_t)n * 4));
            CU(c, up(bs.d_in_cl, pull ? v.clip_left : b->h_c_cl, (size_t)n * 4)); CU(c, up(bs.d_in_cr, pull ? v.clip_right : b->h_c_cr, (size_t)n * 4));
            if (!pull) CU(c, up(b->d_in_read, b->h_c_read, (size_t)n * 4));
        }
        { int rc = bin_zero(c, bs); if (rc) return rc; }
        BinArgs &ba = bs.ba;
        ba.read = pull ? nullptr : b->d_in_read;
        ba.seq_cursor = pull ? bs.d_stats + 8 : nullptr;
        ba.gate = mode == MODE_COMPACT ? b->d_gate : nullptr; ba.host_meta = b->d_view_meta;
        ba.n = n; ba.seq_total = seq_total; ba.clen = c->d_clen; ba.coff = c->d_coff; ba.n_contigs = c->n_contigs;
        ba.window = c->p.window_size; ba.min_length = c->p.min_length; ba.flags = c->p.flags;
        { int rc = bin_classify(c, bs, bs.h_over, bs.d_over, (size_t)OVER_CAP * 4); if (rc) return rc; }
        CU(c, cudaEventSynchronize(bs.ev_prep));   // the previous batch keeps computing on c->stream meanwhile
        b->st.host_classify_ms = ms_since(t_begin);
        if (bs.h_stats[6] & 1ull) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: seq_off / l_qseq inconsistent");
        b->st.n_oversize = (int64_t)bs.h_stats[11];
        // ---- plan from the histogram ----
        const auto t_sort = std::chrono::steady_clock::now();
        n_aln = (int64_t)bs.h_stats[1];
        b->st.cells = (int64_t)bs.h_stats[0];
        { int rc = plan_from_histogram(c, bs, n_aln); if (rc) return rc; }
        b->st.host_sort_ms = ms_since(t_sort);
        b->st.n_aligned = n_aln; b->st.n_generic = bs.n_generic; b->st.scratch_bytes = bs.scratch_bytes;
        if (n_aln > 0) up_bytes += (int64_t)BIN_KEYS * 4 + bs.n_items * (int64_t)sizeof(WarpItem);
        { int rc = bin_scatter(c, bs); if (rc) return rc; }
        if (pull && n_aln > 0) CU(c, launch_seq_pull(b->d_view_seq4, bs.d_aln, bs.d_src_off, (int)n_aln, bs.d_in_seq4, c->sm_count, s2));
    }
    if (n_reads > 0) {
        CU(c, cudaMemsetAsync(b->d_rflags, 0, (size_t)n_reads, s2));
        CU(c, cudaMemsetAsync(b->d_ridx, 0xff, (size_t)n_reads * 4, s2));
    }
    CU(c, cudaEventRecord(bs.ev_ready, s2));
    CU(c, cudaEventRecord(bs.ev[4], s2));
    // ---- compute stream; results go home on stream3 while the next batch computes ----
    int nl = 0;
    { int rc = run_kernels(c, bs, batch_target(c, b), &nl); if (rc) return rc; }
    b->st.kernel_launches = nl + (n > 0 ? 1 : 0) + (n_aln > 0 ? (pull ? 3 : 2) : 0);
    cudaStream_t s3 = c->stream3;
    if (n_aln > 0) CU(c, launch_result_index(bs.d_out, (int)n_aln, n_reads, b->d_rflags, b->d_ridx, bs.d_stats + 7, c->sm_count, s3));
    if (n_reads > 0) {
        CU(c, cudaMemcpyAsync(b->v.flags, b->d_rflags, (size_t)n_reads, cudaMemcpyDeviceToHost, s3));
        CU(c, cudaMemcpyAsync(b->h_ridx, b->d_ridx, (size_t)n_reads * 4, cudaMemcpyDeviceToHost, s3));
    }
    if (n_aln > 0) CU(c, cudaMemcpyAsync(bs.h_stats + 7, bs.d_stats + 7, 8, cudaMemcpyDeviceToHost, s3));
    if (n_aln > 0) {
        CU(c, cudaMemcpyAsync(b->h_out, bs.d_out, (size_t)n_aln * sizeof(AlnOut), cudaMemcpyDeviceToHost, s3));
        CU(c, cudaMemcpyAsync(b->h_aln_start, bs.d_aln_start, (size_t)n_aln * 8, cudaMemcpyDeviceToHost, s3));
    }
    // (the bytes the GPU fetched itself -- bases, compact records -- are added from the device's counters)
    b->st.h2d_bytes = up_bytes + (pull ? (int64_t)bs.h_stats[10] * (int64_t)sizeof(fadegpu_read_meta) : 0);
    b->st.d2h_bytes = n_aln * (int64_t)(sizeof(AlnOut) + 8) + n_reads * 5 + (n > 0 ? (int64_t)BIN_KEYS * 4 + 128 + OVER_CAP * 4 : 0);
    if (pull && n_aln > 0) CU(c, cudaMemcpyAsync(bs.h_stats + 8, bs.d_stats + 8, 8, cudaMemcpyDeviceToHost, s3));   // bases pulled
    CU(c, cudaEventRecord(bs.ev[3], s3));
    b->st.host_submit_ms = ms_since(t_begin);
    return FADEGPU_OK;
}

static fadegpu_inputs view_inputs(const fadegpu_batch_view &v)
{
    fadegpu_inputs in;
    in.seq4 = v.seq4; in.seq_off = v.seq_off; in.l_qseq = v.l_qseq; in.tid = v.tid; in.pos = v.pos;
    in.aligned_len = v.aligned_len; in.clip_left = v.clip_left; in.clip_right = v.clip_right;
    return in;
}

static void worker_main(fadegpu_ctx *c);
static int launch_job(fadegpu_ctx *c, fadegpu_job *j);

// queue the device half of a batch (stage B) or of a staged job for the ctx thread, started on first use (caller holds
// q_mu)
static int queue_half(fadegpu_ctx *c, const fadegpu_ctx::Queued &q, const char *fn)
{
    if (!c->worker.joinable()) {
        try { c->worker = std::thread(worker_main, c); }
        catch (const std::exception &e) { return fail(c, FADEGPU_E_STATE, std::string(fn) + ": cannot start the submit thread: " + e.what()); }
    }
    InFlight &f = q.j ? q.j->fl : q.b->fl;
    f.queued = true; f.rc = 0;
    c->queue.push_back(q);
    c->q_cv.notify_one();
    return FADEGPU_OK;
}

static void worker_main(fadegpu_ctx *c)
{
    cudaSetDevice(c->device);
    std::unique_lock<std::mutex> lk(c->q_mu);
    for (;;) {
        c->q_cv.wait(lk, [&] { return c->worker_stop || !c->queue.empty(); });
        if (c->queue.empty()) return;
        const fadegpu_ctx::Queued q = c->queue.front();
        c->queue.pop_front();
        c->worker_busy = true;
        lk.unlock();
        int rc;
        std::string err;
        {
            std::lock_guard<std::mutex> g(c->submit_mu);
            rc = q.j ? launch_job(c, q.j) : submit_device_binning(c, q.b, q.n, q.mode, q.seq_bytes);
            if (rc) { std::lock_guard<std::mutex> ge(g_err_mu); err = c->err; }
        }
        lk.lock();
        InFlight &f = q.j ? q.j->fl : q.b->fl;
        f.rc = rc; f.err = err; f.queued = false;
        c->worker_busy = false;
        c->done_cv.notify_all();
    }
}

// every queued submit has been planned and launched
static void drain_submits(fadegpu_ctx *c)
{
    std::unique_lock<std::mutex> lk(c->q_mu);
    c->done_cv.wait(lk, [&] { return c->queue.empty() && !c->worker_busy; });
}

// The state every submit entry point checks, in this order: a reference is loaded, the batch is not in flight, and no
// job of the ctx is (annotate batches and jobs are not in flight together).  Messages under the entry point's name.
static int refuse_submit(fadegpu_ctx *c, const fadegpu_batch *b, bool compact)
{
    if (!c->d_two)
        return compact ? fail(c, FADEGPU_E_STATE, "fadegpu_submit_compact: no reference loaded")
                       : fail(c, FADEGPU_E_STATE, "fadegpu_submit: no reference loaded");
    std::lock_guard<std::mutex> lk(c->q_mu);
    if (b->fl.in_flight)
        return compact ? fail(c, FADEGPU_E_STATE, "fadegpu_submit_compact: batch already in flight (call fadegpu_wait)")
                       : fail(c, FADEGPU_E_STATE, "fadegpu_submit: batch already in flight (call fadegpu_wait)");
    const char *fn = compact ? "fadegpu_submit_compact" : "fadegpu_submit";
    if (c->jobs_in_flight > 0)
        return fail(c, FADEGPU_E_STATE, std::string(fn) + ": a job of this ctx is in flight (call fadegpu_job_wait)");
    return 0;
}

// The submit sequence of every input layout (`in`: the caller's arrays of MODE_GATHERED), after the entry point's
// checks.  Host-binned: the inputs binned on this thread, from the view's arrays (compact records expanded into them
// first) or the caller's.  Device-binned: the caller's arrays gathered on this thread, then stage B queued for the ctx
// thread, or run on this one with FADEGPU_F_SYNC_SUBMIT.
static int submit_batch(fadegpu_ctx *c, fadegpu_batch *b, int64_t n, int mode, int64_t seq_bytes, const fadegpu_inputs *in)
{
    if (c->p.flags & FADEGPU_F_HOST_BINNING) {
        fadegpu_batch_view &v = b->v;
        const fadegpu_inputs view = view_inputs(v);
        if (mode == MODE_COMPACT) {
            for (int64_t k = 0; k < n; ++k) {
                const fadegpu_read_meta &m = v.meta[k];
                v.seq_off[k] = m.seq_off; v.l_qseq[k] = m.l_qseq; v.tid[k] = m.tid; v.pos[k] = m.pos;
                v.aligned_len[k] = m.aligned_len; v.clip_left[k] = (int32_t)m.clip_left; v.clip_right[k] = (int32_t)m.clip_right;
            }
            v.seq_off[n] = seq_bytes;
        }
        std::lock_guard<std::mutex> g(c->submit_mu);
        CU(c, cudaSetDevice(c->device));
        int rc = submit_host_binning(c, b, n, mode == MODE_GATHERED ? in : &view);
        if (rc) return rc;
    } else {
        if (mode == MODE_GATHERED) {   // the caller's arrays are only read here
            CU(c, cudaSetDevice(c->device));
            int rc = gather_reads(c, b, n, *in);
            if (rc) return rc;
        }
        if (!(c->p.flags & FADEGPU_F_SYNC_SUBMIT)) {
            std::lock_guard<std::mutex> lk(c->q_mu);
            int rc = queue_half(c, { b, n, mode, seq_bytes, nullptr }, "fadegpu_submit");
            if (!rc) b->fl.in_flight = true;
            return rc;
        }
        std::lock_guard<std::mutex> g(c->submit_mu);
        if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, FADEGPU_E_CUDA, "fadegpu_submit: cudaSetDevice failed");
        int rc = submit_device_binning(c, b, n, mode, seq_bytes);
        if (rc) return rc;
    }
    std::lock_guard<std::mutex> lk(c->q_mu);
    b->fl.in_flight = true;
    return FADEGPU_OK;
}

int fadegpu_submit(fadegpu_ctx *c, fadegpu_batch *b, int64_t n_reads)
{
    if (!c || !b || b->ctx != c) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: bad ctx/batch");
    const fadegpu_batch_view &v = b->v;
    if (n_reads < 0 || n_reads > v.max_reads) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: n_reads out of range");
    if (n_reads > 0 && (v.seq_off[n_reads] < 0 || v.seq_off[n_reads] > v.max_seq_bytes))
        return fail(c, FADEGPU_E_ARG, "fadegpu_submit: seq_off[n] exceeds max_seq_bytes");
    { int rc = refuse_submit(c, b, false); if (rc) return rc; }
    return submit_batch(c, b, n_reads, MODE_VIEW, 0, nullptr);
}

int fadegpu_submit_compact(fadegpu_ctx *c, fadegpu_batch *b, int64_t n_reads, int64_t seq_bytes)
{
    if (!c || !b || b->ctx != c) return fail(c, FADEGPU_E_ARG, "fadegpu_submit_compact: bad ctx/batch");
    const fadegpu_batch_view &v = b->v;
    if (n_reads < 0 || n_reads > v.max_reads) return fail(c, FADEGPU_E_ARG, "fadegpu_submit_compact: n_reads out of range");
    if (seq_bytes < 0 || seq_bytes > v.max_seq_bytes || seq_bytes > (int64_t)0xffffffffll)
        return fail(c, FADEGPU_E_ARG, "fadegpu_submit_compact: seq_bytes out of range");
    { int rc = refuse_submit(c, b, true); if (rc) return rc; }
    return submit_batch(c, b, n_reads, MODE_COMPACT, seq_bytes, nullptr);
}

// (the state is checked before n_reads and the arrays: a call that fails both reports the state)
int fadegpu_submit_inputs(fadegpu_ctx *c, fadegpu_batch *b, int64_t n_reads, const fadegpu_inputs *in)
{
    if (!c || !b || b->ctx != c || !in) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: bad ctx/batch/inputs");
    { int rc = refuse_submit(c, b, false); if (rc) return rc; }
    if (n_reads < 0 || n_reads > b->v.max_reads) return fail(c, FADEGPU_E_ARG, "fadegpu_submit: n_reads out of range");
    if (n_reads > 0 && (!in->seq4 || !in->seq_off || !in->l_qseq || !in->tid || !in->pos || !in->aligned_len ||
                        !in->clip_left || !in->clip_right))
        return fail(c, FADEGPU_E_ARG, "fadegpu_submit: null input array");
    return submit_batch(c, b, n_reads, MODE_GATHERED, 0, in);
}

// At a wait: false if the submit is not in flight.  Otherwise, once the ctx thread is through with its queued half, the
// submit leaves flight (and the count *n_in_flight, if given), and *rc / *err receive that half's outcome.
static bool end_flight(fadegpu_ctx *c, InFlight &f, int *n_in_flight, int *rc, std::string *err)
{
    std::unique_lock<std::mutex> lk(c->q_mu);
    if (!f.in_flight) return false;
    c->done_cv.wait(lk, [&] { return !f.queued; });
    f.in_flight = false;
    if (n_in_flight) --*n_in_flight;
    *rc = f.rc; *err = f.err;
    f.rc = 0;
    return true;
}

int fadegpu_wait(fadegpu_ctx *c, fadegpu_batch *b)
{
    if (!c || !b || b->ctx != c) return fail(c, FADEGPU_E_ARG, "fadegpu_wait: bad ctx/batch");
    int rc;
    std::string err;
    if (!end_flight(c, b->fl, nullptr, &rc, &err)) return fail(c, FADEGPU_E_STATE, "fadegpu_wait: batch not submitted");
    if (rc) return fail(c, rc, err);   // (a queued submit reports its outcome here)
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaEventSynchronize(b->bs.ev[3]));
    float t;
    if (cudaEventElapsedTime(&t, b->bs.ev[1], b->bs.ev[2]) == cudaSuccess) b->st.kernel_ms = t;
    if (cudaEventElapsedTime(&t, b->bs.ev[0], b->bs.ev[3]) == cudaSuccess) b->st.total_ms = t;
    if (b->dev_binning && b->pulled) {
        if (b->bs.n_aln > 0) b->st.h2d_bytes += (int64_t)b->bs.h_stats[8];
        b->pulled = false;
    }
    // Device-binned submits: flags[] and the per-read index into the results were built on the device; only the
    // per-read output arrays (unless FADEGPU_F_NO_SCATTER) are filled here.  Host-binned submits: all of it here.
    const auto t_scatter = std::chrono::steady_clock::now();
    fadegpu_batch_view &v = b->v;
    const int64_t n = b->n_reads;
    const bool scatter = !(c->p.flags & FADEGPU_F_NO_SCATTER) && v.score != nullptr;
    // (no parallel region unless there is real work: its threads would spin for milliseconds afterwards on the
    // cores the ctx thread needs to queue the next batch)
    const bool walk = scatter || !b->dev_binning;
    const int nthr = walk ? (int)std::max<int64_t>(1, std::min<int64_t>(c->host_threads, b->bs.n_aln / 8192 + 1)) : 1;
    int64_t bad = 0;
    if (b->dev_binning) {
        if (b->bs.n_aln > 0 && (int64_t)b->bs.h_stats[7] != b->bs.n_aln) bad = 1;   // result records counted on the device
    } else {
        memset(v.flags, 0, (size_t)n);   // the other per-read outputs are defined only where FADEGPU_R_ALIGNED is set
        memset(b->h_ridx, 0xff, (size_t)n * sizeof(int32_t));
    }
#pragma omp parallel for schedule(static) reduction(+ : bad) num_threads(nthr) if (nthr > 1)
    for (int64_t k = 0; k < (walk ? b->bs.n_aln : 0); ++k) {
        const AlnOut &o = b->h_out[k];
        const int64_t r = o.read;
        if (r < 0 || r >= n || (o.flags & 0x80000000u) || !(o.flags & 1u) || (!b->dev_binning && b->h_aln[k].read != (int32_t)r)) { ++bad; continue; }
        if (!b->dev_binning) {
            v.flags[r] = (uint8_t)(o.flags & 0xff);
            b->h_ridx[r] = (int32_t)k;
        } else if (b->h_ridx[r] != (int32_t)k) { ++bad; continue; }
        if (!scatter) continue;
        v.score[r] = o.score; v.beg_query[r] = o.beg_query; v.end_query[r] = o.end_query;
        v.beg_ref[r] = o.beg_ref; v.end_ref[r] = o.end_ref; v.n_ops[r] = o.n_ops;
        v.win_start[r] = b->h_aln_start[k];
        memcpy(v.ops + (size_t)r * FADEGPU_MAX_OPS, o.ops, sizeof(o.ops));
    }
    for (int64_t k = 0; k < std::min<int64_t>(b->st.n_oversize, OVER_CAP); ++k) {
        const int64_t r = b->bs.h_over[k];
        if (r >= 0 && r < n) v.flags[r] = FADEGPU_R_OVERSIZE;
    }
    b->st.host_wait_ms = std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_scatter).count();
    if (bad) return fail(c, FADEGPU_E_CUDA, "fadegpu_wait: a kernel did not produce a result record (internal error)");
    return FADEGPU_OK;
}

int fadegpu_get_results(const fadegpu_batch *b, fadegpu_results_view *r)
{
    if (!b || !r) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_get_results: null argument");
    if (b->fl.in_flight) return fail(b->ctx, FADEGPU_E_STATE, "fadegpu_get_results: batch in flight (call fadegpu_wait)");
    static_assert(sizeof(fadegpu_result) == sizeof(AlnOut), "fadegpu_result must mirror AlnOut");
    r->n_results = b->bs.n_aln;
    r->results = reinterpret_cast<const fadegpu_result *>(b->h_out);
    r->win_start = b->h_aln_start;
    r->result_index = b->h_ridx;
    return FADEGPU_OK;
}

int fadegpu_get_stats(const fadegpu_batch *b, fadegpu_stats *s)
{
    if (!b || !s) return fail(nullptr, FADEGPU_E_ARG, "fadegpu_get_stats: null argument");
    *s = b->st;
    return FADEGPU_OK;
}

int fadegpu_get_timeline(const fadegpu_batch *b, const fadegpu_batch *origin, float ms[6])
{
    if (!b || !origin || !ms || b->ctx != origin->ctx) return fail(b ? b->ctx : nullptr, FADEGPU_E_ARG, "fadegpu_get_timeline: bad arguments");
    for (int k = 0; k < 6; ++k)
        if (cudaEventElapsedTime(&ms[k], origin->bs.ev[0], b->bs.ev[k]) != cudaSuccess) { cudaGetLastError(); ms[k] = -1.f; }
    return FADEGPU_OK;
}

// Replays re-run the device side of a submit on what it left resident in HBM: the binning kernels
// (length floor, window arithmetic, histogram, scatter of the descriptors -- into scratch, because the
// order among equal window lengths is not reproducible and the live descriptors point at the bases
// already fetched), then fills / traceback / generic.  No host work, no copies.
static int replay_binning(fadegpu_ctx *c, fadegpu_batch *b, cudaEvent_t *dep)
{
    *dep = nullptr;
    if (b->bs.ba.n == 0) return 0;
    const size_t n = (size_t)b->v.max_reads;
    if (!b->d_aln_scratch) {
        CU(c, cudaMalloc((void **)&b->d_aln_scratch, n * sizeof(AlnDesc)));
        CU(c, cudaMalloc((void **)&b->d_i64_scratch, 2 * n * sizeof(int64_t)));
    }
    BinState &bs = b->bs;
    cudaStream_t s2 = c->stream2;
    { int rc = bin_zero(c, bs); if (rc) return rc; }
    BinArgs ba = bs.ba;
    ba.gate = nullptr;        // compact inputs: the records fetched by the submit are resident in the device mirrors
    CU(c, launch_bin_classify(ba, c->sm_count, s2));
    if (bs.n_aln > 0) {
        ba.aln = b->d_aln_scratch; ba.aln_start = b->d_i64_scratch; ba.src_off = b->d_i64_scratch + n;
        if (ba.seq_cursor) ba.seq_cursor = bs.d_stats + 9;
        CU(c, launch_bin_scatter(ba, c->sm_count, s2));
    }
    CU(c, cudaEventRecord(bs.ev_ready, s2));
    *dep = bs.ev_ready;
    return 0;
}

static int replay_pass(fadegpu_ctx *c, fadegpu_batch *b)
{
    cudaEvent_t dep = nullptr;
    { int rc = replay_binning(c, b, &dep); if (rc) return rc; }
    { int rc = run_plan(c, b->bs, batch_target(c, b), nullptr, nullptr, nullptr, nullptr, dep); if (rc) return rc; }
    return 0;
}

int fadegpu_replay_batches(fadegpu_ctx *c, fadegpu_batch *const *batches, int32_t n_batches, int32_t iters, float *ms_out)
{
    if (!c || !batches || n_batches <= 0 || iters <= 0) return fail(c, FADEGPU_E_ARG, "fadegpu_replay_batches: bad arguments");
    for (int32_t i = 0; i < n_batches; ++i) {
        fadegpu_batch *b = batches[i];
        if (!b || b->ctx != c) return fail(c, FADEGPU_E_ARG, "fadegpu_replay_batches: bad batch");
        if (b->fl.in_flight) return fail(c, FADEGPU_E_STATE, "fadegpu_replay_batches: batch in flight");
        if (b->bs.plan.empty() && b->bs.n_aln > 0) return fail(c, FADEGPU_E_STATE, "fadegpu_replay_batches: nothing submitted");
    }
    drain_submits(c);
    std::lock_guard<std::mutex> submit_guard(c->submit_mu);
    CU(c, cudaSetDevice(c->device));
    cudaEvent_t e0, e1;
    CU(c, cudaEventCreate(&e0)); CU(c, cudaEventCreate(&e1));
    CU(c, cudaDeviceSynchronize());
    CU(c, cudaEventRecord(e0, c->stream));
    CU(c, cudaStreamWaitEvent(c->stream2, e0, 0));
    for (int32_t it = 0; it < iters; ++it)
        for (int32_t i = 0; i < n_batches; ++i) { int rc = replay_pass(c, batches[i]); if (rc) return rc; }
    // the ctx stream continues after the kernels of every batch; the streams are in order, so the last pass of every
    // batch covers the earlier ones
    for (int32_t i = 0; i < n_batches; ++i) CU(c, cudaStreamWaitEvent(c->stream, batches[i]->bs.ev_kernels, 0));
    CU(c, cudaEventRecord(e1, c->stream));
    CU(c, cudaEventSynchronize(e1));
    float ms = 0;
    CU(c, cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (ms_out) *ms_out = ms;
    return FADEGPU_OK;
}

int fadegpu_replay_kernels(fadegpu_ctx *c, fadegpu_batch *b, int32_t iters, float *ms_out)
{
    if (!c || !b || b->ctx != c || iters <= 0) return fail(c, FADEGPU_E_ARG, "fadegpu_replay_kernels: bad arguments");
    if (b->fl.in_flight) return fail(c, FADEGPU_E_STATE, "fadegpu_replay_kernels: batch in flight");
    if (b->bs.plan.empty() && b->bs.n_aln > 0) return fail(c, FADEGPU_E_STATE, "fadegpu_replay_kernels: nothing submitted");
    drain_submits(c);
    {   // one pass with per-stage events (serialising: fill / traceback / generic), then the timed passes
        std::lock_guard<std::mutex> submit_guard(c->submit_mu);
        CU(c, cudaSetDevice(c->device));
        float f = 0, t = 0, g = 0;
        int rc = run_plan(c, b->bs, batch_target(c, b), &f, &t, &g, nullptr, nullptr);
        if (rc) return rc;
        b->st.fill_ms = f; b->st.trace_ms = t; b->st.generic_ms = g;
    }
    fadegpu_batch *one[1] = { b };
    return fadegpu_replay_batches(c, one, 1, iters, ms_out);
}

// copy with the ctx's host threads (the caller's arrays are pageable; the staging is pinned)
static void parallel_copy(char *dst, const char *src, size_t bytes, int nthr)
{
    const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(1, nthr), bytes >> 20));
#pragma omp parallel for schedule(static, 1) num_threads(T) if (T > 1)
    for (int t = 0; t < T; ++t) {
        const size_t lo = bytes * (size_t)t / (size_t)T, hi = bytes * (size_t)(t + 1) / (size_t)T;
        memcpy(dst + lo, src + lo, hi - lo);
    }
}

static size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// FADEGPU_E_STATE while a batch of the ctx is submitted and not yet waited for
static int refuse_in_flight(fadegpu_ctx *c, const char *fn)
{
    std::lock_guard<std::mutex> lk(c->q_mu);
    for (const fadegpu_batch *b : c->batches)
        if (b->fl.in_flight)
            return fail(c, FADEGPU_E_STATE, std::string(fn) + ": a batch of this ctx is in flight (call fadegpu_wait)");
    return 0;
}

// The caller's part of a pair or region call: copy its arrays into the job's pinned staging
using StageFn = std::function<void(char *h_stage)>;
// on stream2, after the upload: the binning inputs and the queries of j->bs (failures reported to j->d_bad), and ba's
// contig table; counts its launches
using PrepFn = std::function<int(fadegpu_job *j, const char *d_raw, BinArgs &ba, int *launches)>;

// Stage half of a pair or region call, on the caller's thread: the raw inputs go to the device through the job's pinned
// staging on stream2, where the caller's prep kernels write the per-item binning inputs and the queries, and the binning
// classify kernel histograms them; the histogram is on its way home when this returns.  The device half (launch_job)
// does the rest.
static int stage_call(fadegpu_ctx *c, fadegpu_job *j, const StagedCall &sc, const StageFn &stage, const PrepFn &prep)
{
    j->sc = sc;
    j->st = fadegpu_stats{};
    j->st.n_reads = sc.n;
    j->st.n_oversize = sc.n_over;
    if (sc.n == 0) return FADEGPU_OK;
    const int64_t n = sc.n, qbytes = sc.qbytes;
    const int32_t max_ops = sc.max_ops;
    CU(c, cudaSetDevice(c->device));
    BinState &bs = j->bs;
    if (bs.max_items < n || bs.max_seq_bytes < qbytes + 16) {
        const int64_t nr = std::max(n, bs.max_items), sb = std::max(qbytes + 16, bs.max_seq_bytes);
        free_bin_state(c, bs);
        int rc = alloc_bin_state(c, bs, nr, sb);
        if (rc) return rc;
    }
    const size_t raw = sc.raw;
    if (j->stage_bytes < raw) {
        free_host(j->h_stage);
        j->stage_bytes = 0;
        CU(c, cudaHostAlloc((void **)&j->h_stage, raw, cudaHostAllocDefault));
        j->stage_bytes = raw;
    }
    stage(j->h_stage);
    {
        int rc = 0;
        auto grow = [&](auto **p, size_t *have, size_t bytes) { if (!rc) rc = ensure_dev(c, (void **)p, have, std::max<size_t>(bytes, 16)); };
        grow(&j->d_raw, &j->raw_bytes, raw);
        grow(&j->d_res, &j->res_bytes, (size_t)n * sizeof(fadegpu_pair_result));
        if (max_ops > 0) {
            grow(&j->d_spill, &j->spill_bytes, (size_t)n * (size_t)max_ops * 4);
            grow(&j->d_ops, &j->ops_bytes, (size_t)n * (size_t)max_ops * 4);
        }
        if (rc) return rc;
        if (!j->d_bad) CU(c, cudaMalloc((void **)&j->d_bad, sizeof(int32_t)));
        if (!j->h_bad) CU(c, cudaHostAlloc((void **)&j->h_bad, sizeof(int32_t), cudaHostAllocDefault));
    }
    // ---- upload, packing and binning on stream2 ----
    bs.plan.clear();
    bs.n_aln = 0; bs.n_items = 0;
    memset(bs.h_stats, 0, 128);
    cudaStream_t s2 = c->stream2;
    CU(c, cudaEventRecord(bs.ev[0], s2));
    CU(c, cudaMemcpyAsync(j->d_raw, j->h_stage, raw, cudaMemcpyHostToDevice, s2));
    j->h2d = (int64_t)raw;
    CU(c, cudaEventRecord(bs.ev[4], s2));
    { int rc = bin_zero(c, bs); if (rc) return rc; }
    CU(c, cudaMemsetAsync(j->d_bad, 0x7f, sizeof(int32_t), s2));   // > any item index
    BinArgs &ba = bs.ba;
    // window 0 and floor 0: the window of item k is exactly its target / interval, every non-empty item is aligned
    ba.n = n; ba.seq_total = qbytes; ba.window = 0; ba.min_length = 0; ba.flags = c->p.flags;
    j->n_prep = 0;
    { int rc = prep(j, j->d_raw, ba, &j->n_prep); if (rc) return rc; }
    return bin_classify(c, bs, j->h_bad, j->d_bad, sizeof(int32_t));
}

// Device half of a staged call, under submit_mu (it sizes the shared scratch): once the binning histogram is home, the
// launch plan and run_plan of a device-binned submit on the job's batch, with every alignment traced back and the full
// CIGARs spilled (score-only calls: only the end cell is found, nothing is spilled); the records come back in item
// order to j->out / j->ops_out on stream3.  Queued jobs run it on the ctx thread while the caller stages the next.
static int launch_job(fadegpu_ctx *c, fadegpu_job *j)
{
    const StagedCall &sc = j->sc;
    if (sc.n == 0) return FADEGPU_OK;
    const int64_t n = sc.n;
    const int32_t max_ops = sc.max_ops;
    BinState &bs = j->bs;
    CU(c, cudaSetDevice(c->device));
    CU(c, cudaEventSynchronize(bs.ev_prep));
    const int32_t bad = *j->h_bad;
    if (bad >= 0 && bad < n)
        return fail(c, FADEGPU_E_ARG, std::string(sc.fn) + ": the query of " + sc.item + " " + std::to_string(bad) +
                                          " holds a letter outside the BAM nt16 alphabet =ACMGRSVTWYHKDBN");
    if (bs.h_stats[6] & 1ull) return fail(c, FADEGPU_E_CUDA, std::string(sc.fn) + ": internal error (query offsets)");
    const int64_t n_aln = (int64_t)bs.h_stats[1];
    int n_prep = j->n_prep;
    int64_t h2d = j->h2d;
    PlanTarget pt{};
    { int rc = sc.reference(j, &pt.ref, &n_prep); if (rc) return rc; }
    { int rc = plan_from_histogram(c, bs, n_aln); if (rc) return rc; }
    if (n_aln > 0) h2d += (int64_t)BIN_KEYS * 4 + bs.n_items * (int64_t)sizeof(WarpItem);
    { int rc = bin_scatter(c, bs); if (rc) return rc; }
    CU(c, cudaEventRecord(bs.ev_ready, c->stream2));
    // ---- SW kernels: the plan against the caller's reference ----
    pt.seq = bs.d_in_seq4;
    pt.tags_only = 0;   // every item is traced back (or has its end cell found), whatever the ctx's FADEGPU_F_TAGS_ONLY
    pt.ops_spill = max_ops > 0 ? j->d_spill : nullptr;
    pt.ops_cap = max_ops;
    pt.end_only = sc.score_only;
    int nl = 0;
    { int rc = run_kernels(c, bs, pt, &nl); if (rc) return rc; }
    // ---- records in item order, home on stream3 ----
    cudaStream_t s3 = c->stream3;
    // the results kernel writes the ops of the aligned items only: empty and oversize items keep these zeros (rather
    // than whatever an earlier call of this job left there)
    if (max_ops > 0) CU(c, cudaMemsetAsync(j->d_ops, 0, (size_t)n * (size_t)max_ops * 4, s3));
    CU(c, launch_pair_results(n, reinterpret_cast<const int64_t *>(j->d_raw), reinterpret_cast<const int64_t *>(j->d_raw + sc.o_tbeg),
                              reinterpret_cast<const int64_t *>(j->d_raw + sc.o_tend), bs.d_aln, bs.d_out, (int)n_aln,
                              sc.score_only, j->d_spill, max_ops, reinterpret_cast<PairResult *>(j->d_res), j->d_ops,
                              bs.d_stats + 7, c->sm_count, s3));
    CU(c, cudaMemcpyAsync(j->out, j->d_res, (size_t)n * sizeof(fadegpu_pair_result), cudaMemcpyDeviceToHost, s3));
    if (max_ops > 0)
        CU(c, cudaMemcpyAsync(j->ops_out, j->d_ops, (size_t)n * (size_t)max_ops * 4, cudaMemcpyDeviceToHost, s3));
    CU(c, cudaMemcpyAsync(bs.h_stats + 7, bs.d_stats + 7, 8, cudaMemcpyDeviceToHost, s3));
    CU(c, cudaEventRecord(bs.ev[3], s3));
    fadegpu_stats &st = j->st;
    st.n_aligned = n_aln;
    st.n_generic = bs.n_generic;
    st.cells = (int64_t)bs.h_stats[0];
    st.h2d_bytes = h2d;
    st.d2h_bytes = n * (int64_t)(sizeof(fadegpu_pair_result) + 4 * (size_t)max_ops) + (int64_t)BIN_KEYS * 4 + 128 + 4 + 8;
    st.kernel_launches = nl + n_prep + 1 + (n_aln > 0 ? 2 : 1);
    st.scratch_bytes = bs.scratch_bytes;
    st.host_threads = c->host_threads;
    return FADEGPU_OK;
}

// The records of a launched call are home: the device's count of result records, and the device times
static int finish_job(fadegpu_ctx *c, fadegpu_job *j)
{
    if (j->sc.n == 0) return FADEGPU_OK;
    const BinState &bs = j->bs;
    CU(c, cudaEventSynchronize(bs.ev[3]));
    if ((int64_t)bs.h_stats[7] != j->st.n_aligned)
        return fail(c, FADEGPU_E_CUDA, std::string(j->sc.fn) + ": a kernel did not produce a result record (internal error)");
    float t;
    if (cudaEventElapsedTime(&t, bs.ev[1], bs.ev[2]) == cudaSuccess) j->st.kernel_ms = t;
    if (cudaEventElapsedTime(&t, bs.ev[0], bs.ev[3]) == cudaSuccess) j->st.total_ms = t;
    return FADEGPU_OK;
}

// A validated pair or region call.  Synchronous (job == nullptr): after the device halves of the jobs queued before it,
// both halves on the ctx's own job, the records straight into the caller's arrays.  A job: its pinned records, the
// stage half here and the device half queued for the ctx thread (here with FADEGPU_F_SYNC_SUBMIT).
static int run_call(fadegpu_ctx *c, fadegpu_job *job, const StagedCall &sc, const StageFn &stage, const PrepFn &prep,
                    fadegpu_pair_result *out, uint32_t *ops_out, fadegpu_stats *stats_out,
                    std::chrono::steady_clock::time_point t_begin)
{
    auto ms_since_begin = [&] {
        return std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    };
    if (!job) {
        drain_submits(c);
        std::lock_guard<std::mutex> submit_guard(c->submit_mu);
        if (!c->sync_job) {
            c->sync_job = new (std::nothrow) fadegpu_job();
            if (!c->sync_job) return fail(c, FADEGPU_E_OOM, std::string(sc.fn) + ": out of host memory");
            c->sync_job->ctx = c;
        }
        fadegpu_job *j = c->sync_job;
        j->out = out; j->ops_out = ops_out;
        int rc = stage_call(c, j, sc, stage, prep);
        if (!rc) rc = launch_job(c, j);
        if (!rc) rc = finish_job(c, j);
        if (rc) return rc;
        if (sc.n > 0) j->st.host_submit_ms = ms_since_begin();
        if (stats_out) *stats_out = j->st;
        return FADEGPU_OK;
    }
    fadegpu_job *j = job;
    j->n_res = -1;
    const size_t res_bytes = (size_t)sc.n * sizeof(fadegpu_pair_result), ops_bytes = (size_t)sc.n * (size_t)sc.max_ops * 4;
    CU(c, cudaSetDevice(c->device));
    if (j->h_res_bytes < res_bytes) {
        free_host(j->h_res);
        j->h_res_bytes = 0;
        CU(c, cudaHostAlloc((void **)&j->h_res, res_bytes, cudaHostAllocDefault));
        j->h_res_bytes = res_bytes;
    }
    if (j->h_ops_bytes < ops_bytes) {
        free_host(j->h_ops);
        j->h_ops_bytes = 0;
        CU(c, cudaHostAlloc((void **)&j->h_ops, ops_bytes, cudaHostAllocDefault));
        j->h_ops_bytes = ops_bytes;
    }
    j->out = j->h_res; j->ops_out = j->h_ops;
    { int rc = stage_call(c, j, sc, stage, prep); if (rc) return rc; }
    const bool here = (c->p.flags & FADEGPU_F_SYNC_SUBMIT) != 0;
    if (here) {
        std::lock_guard<std::mutex> submit_guard(c->submit_mu);
        int rc = launch_job(c, j);
        if (rc) return rc;
    }
    if (sc.n > 0) j->st.host_submit_ms = ms_since_begin();
    std::lock_guard<std::mutex> lk(c->q_mu);
    if (!here) { int rc = queue_half(c, { nullptr, 0, 0, 0, j }, sc.fn); if (rc) return rc; }
    j->fl.in_flight = true;
    ++c->jobs_in_flight;
    return FADEGPU_OK;
}

// Pairs: pair_prep_kernel writes the per-pair binning inputs and the queries (nt16, reverse-complemented),
// pair_pack_targets_kernel and pair_xlist_kernel pack the targets as a reference of their own, whose contigs the
// targets are.
static int pairs_call(fadegpu_ctx *c, const char *fn, bool score_only, int64_t n_pairs, const fadegpu_pairs *in,
                      int32_t max_ops, fadegpu_pair_result *out, uint32_t *ops_out, fadegpu_stats *stats_out,
                      fadegpu_job *job)
{
    const std::string at = std::string(fn) + ": ";
    if (!c) return fail(nullptr, FADEGPU_E_ARG, at + "null ctx");
    if (n_pairs < 0 || n_pairs > ((int64_t)1 << 30) || max_ops < 0)
        return fail(c, FADEGPU_E_ARG, at + "n_pairs or max_ops out of range");
    if (n_pairs > 0 && (!in || !in->query_off || !in->target_off || (!job && (!out || (max_ops > 0 && !ops_out)))))
        return fail(c, FADEGPU_E_ARG, at + "null argument");
    { int rc = refuse_in_flight(c, fn); if (rc) return rc; }
    const auto t_begin = std::chrono::steady_clock::now();
    const int64_t n = n_pairs;
    int64_t qbytes = 0, tbytes = 0, n_over = 0;
    if (n > 0) {
        const int64_t *qo = in->query_off, *to = in->target_off;
        if (qo[0] < 0 || to[0] < 0) return fail(c, FADEGPU_E_ARG, at + "negative offset");
        for (int64_t k = 0; k < n; ++k) {
            const int64_t ql = qo[k + 1] - qo[k], tl = to[k + 1] - to[k];
            if (ql < 0 || tl < 0)
                return fail(c, FADEGPU_E_ARG, at + "offsets decrease at pair " + std::to_string(k));
            if (ql > 0 && tl > 0 && (tl > 0x7fffffff || ql * tl > PAIR_MAX_CELLS)) ++n_over;
        }
        qbytes = qo[n] - qo[0]; tbytes = to[n] - to[0];
        if ((qbytes > 0 && !in->query) || (tbytes > 0 && !in->target))
            return fail(c, FADEGPU_E_ARG, at + "null sequence array");
    }
    // ---- staging: [query_off][target_off] rebased to 0, then the query and the target letters ----
    const size_t o_toff = align16((size_t)(n + 1) * 8), o_q = o_toff + align16((size_t)(n + 1) * 8);
    const size_t o_t = o_q + align16((size_t)qbytes);
    const int64_t n_words = n + (tbytes >> 5) + 2;   // target k starts at 32 * (k + toff[k] / 32)
    const int64_t n_chunks = (n_words + PAIR_CHUNK_WORDS - 1) / PAIR_CHUNK_WORDS;
    StagedCall sc;
    sc.fn = fn; sc.item = "pair";
    sc.n = n; sc.qbytes = qbytes; sc.n_over = n_over; sc.max_ops = max_ops; sc.score_only = score_only;
    sc.raw = o_t + align16((size_t)tbytes);
    sc.o_tbeg = o_toff; sc.o_tend = o_toff + 8;   // target k spans toff[k] .. toff[k + 1]
    auto stage = [&](char *h) {
        int64_t *hq = reinterpret_cast<int64_t *>(h), *ht = reinterpret_cast<int64_t *>(h + o_toff);
        const int64_t q0 = in->query_off[0], t0 = in->target_off[0];
        for (int64_t k = 0; k <= n; ++k) { hq[k] = in->query_off[k] - q0; ht[k] = in->target_off[k] - t0; }
        if (qbytes) parallel_copy(h + o_q, in->query + q0, (size_t)qbytes, c->host_threads);
        if (tbytes) parallel_copy(h + o_t, in->target + t0, (size_t)tbytes, c->host_threads);
    };
    auto prep = [&](fadegpu_job *j, const char *d, BinArgs &ba, int *launches) -> int {
        BinState &bs = j->bs;
        int rc = 0;
        auto grow = [&](auto **p, size_t *have, size_t bytes) { if (!rc) rc = ensure_dev(c, (void **)p, have, std::max<size_t>(bytes, 16)); };
        grow(&j->d_two, &j->two_bytes, (size_t)n_words * 8); grow(&j->d_n, &j->n_bytes, (size_t)n_words * 4);
        grow(&j->d_x, &j->x_bytes, (size_t)n_words * 4); grow(&j->d_chunk_x, &j->chunk_bytes, (size_t)n_chunks * 4);
        grow(&j->d_clen, &j->clen_bytes, (size_t)n * 8); grow(&j->d_coff, &j->coff_bytes, (size_t)n * 8);
        if (rc) return rc;
        PairArgs &pa = j->pa;
        pa = PairArgs{};
        pa.n = n;
        pa.qoff = reinterpret_cast<const int64_t *>(d); pa.toff = reinterpret_cast<const int64_t *>(d + o_toff);
        pa.query = d + o_q; pa.target = d + o_t;
        pa.seq_off = bs.d_in_seq_off; pa.pos = bs.d_in_pos; pa.l_qseq = bs.d_in_lq; pa.tid = bs.d_in_tid;
        pa.aligned_len = bs.d_in_alen; pa.clip_left = bs.d_in_cl; pa.clip_right = bs.d_in_cr;
        pa.clen = j->d_clen; pa.coff = j->d_coff; pa.seq4 = bs.d_in_seq4; pa.bad = j->d_bad;
        pa.two = j->d_two; pa.nmask = j->d_n; pa.xmask = j->d_x; pa.n_words = n_words;
        pa.chunk_x = j->d_chunk_x; pa.n_x = bs.d_stats + 12;
        CU(c, launch_pair_prep(pa, c->sm_count, c->stream2));
        CU(c, launch_pair_pack_targets(pa, c->stream2));
        *launches += 2;
        ba.clen = j->d_clen; ba.coff = j->d_coff; ba.n_contigs = (int32_t)n;   // contigs = targets
        return 0;
    };
    // (runs in the device half, possibly on the ctx thread: it captures nothing of this frame)
    sc.reference = [c](fadegpu_job *j, RefDev *ref, int *launches) -> int {
        PairArgs &pa = j->pa;
        const int64_t n_x = (int64_t)j->bs.h_stats[12];
        int rc = ensure_dev(c, (void **)&j->d_xpos, &j->xpos_bytes, std::max<size_t>(16, (size_t)n_x * 8));
        if (!rc) rc = ensure_dev(c, (void **)&j->d_xchr, &j->xchr_bytes, std::max<size_t>(16, (size_t)n_x));
        if (rc) return rc;
        pa.xpos = j->d_xpos; pa.xchr = j->d_xchr;
        if (n_x > 0) { CU(c, launch_pair_xlist(pa, c->stream2)); ++*launches; }
        ref->planes.two = j->d_two; ref->planes.nmask = j->d_n; ref->planes.xmask = j->d_x;
        ref->xpos = j->d_xpos; ref->xchr = j->d_xchr; ref->n_x = n_x;
        return 0;
    };
    return run_call(c, job, sc, stage, prep, out, ops_out, stats_out, t_begin);
}

int fadegpu_align_pairs(fadegpu_ctx *c, int64_t n_pairs, const fadegpu_pairs *in, int32_t max_ops,
                        fadegpu_pair_result *out, uint32_t *ops_out, fadegpu_stats *stats_out)
{
    return pairs_call(c, "fadegpu_align_pairs", false, n_pairs, in, max_ops, out, ops_out, stats_out, nullptr);
}

int fadegpu_score_pairs(fadegpu_ctx *c, int64_t n_pairs, const fadegpu_pairs *in, fadegpu_pair_result *out,
                        fadegpu_stats *stats_out)
{
    return pairs_call(c, "fadegpu_score_pairs", true, n_pairs, in, 0, out, nullptr, stats_out, nullptr);
}

// Regions: only the queries and the intervals are staged; region_prep_kernel writes the per-region binning inputs and
// the queries, the binning runs on the ctx's contig table and the SW kernels read the resident reference.
static int regions_call(fadegpu_ctx *c, const char *fn, bool score_only, int64_t n_regions, const fadegpu_regions *in,
                        int32_t max_ops, fadegpu_pair_result *out, uint32_t *ops_out, fadegpu_stats *stats_out,
                        fadegpu_job *job)
{
    const std::string at0 = std::string(fn) + ": ";
    if (!c) return fail(nullptr, FADEGPU_E_ARG, at0 + "null ctx");
    if (n_regions < 0 || n_regions > ((int64_t)1 << 30) || max_ops < 0)
        return fail(c, FADEGPU_E_ARG, at0 + "n_regions or max_ops out of range");
    if (n_regions > 0 && (!in || !in->query_off || !in->tid || !in->start || !in->end || !in->strand ||
                          (!job && (!out || (max_ops > 0 && !ops_out)))))
        return fail(c, FADEGPU_E_ARG, at0 + "null argument");
    { int rc = refuse_in_flight(c, fn); if (rc) return rc; }
    if (c->n_contigs <= 0) return fail(c, FADEGPU_E_STATE, at0 + "no reference is loaded");
    const auto t_begin = std::chrono::steady_clock::now();
    const int64_t n = n_regions;
    int64_t qbytes = 0, n_over = 0;
    if (n > 0) {
        const int64_t *qo = in->query_off;
        if (qo[0] < 0) return fail(c, FADEGPU_E_ARG, at0 + "negative offset");
        for (int64_t k = 0; k < n; ++k) {
            const int64_t ql = qo[k + 1] - qo[k];
            if (ql < 0) return fail(c, FADEGPU_E_ARG, at0 + "offsets decrease at region " + std::to_string(k));
            const int32_t tid = in->tid[k];
            const int64_t s = in->start[k], e = in->end[k];
            if (tid < 0 || tid >= c->n_contigs || s < 0 || s > e || e > c->clen[(size_t)tid] || in->strand[k] > 1) {
                const std::string at = at0 + "region " + std::to_string(k) + ": ";
                if (tid < 0 || tid >= c->n_contigs)
                    return fail(c, FADEGPU_E_ARG, at + "tid " + std::to_string(tid) + " is not a contig of the reference");
                if (s < 0 || s > e || e > c->clen[(size_t)tid])
                    return fail(c, FADEGPU_E_ARG, at + "[" + std::to_string(s) + ", " + std::to_string(e) +
                                                      ") is not an interval of contig " + std::to_string(tid) + " (length " +
                                                      std::to_string(c->clen[(size_t)tid]) + ")");
                return fail(c, FADEGPU_E_ARG, at + "strand " + std::to_string(in->strand[k]) + " is neither 0 nor 1");
            }
            const int64_t tl = e - s;
            if (ql > 0 && tl > 0 && (tl > 0x7fffffff || ql * tl > PAIR_MAX_CELLS)) ++n_over;
        }
        qbytes = qo[n] - qo[0];
        if (qbytes > 0 && !in->query) return fail(c, FADEGPU_E_ARG, at0 + "null sequence array");
    }
    // ---- staging: [query_off rebased to 0][tid][start][end][strand], then the query letters ----
    const size_t o_tid = align16((size_t)(n + 1) * 8), o_start = o_tid + align16((size_t)n * 4);
    const size_t o_end = o_start + align16((size_t)n * 8), o_strand = o_end + align16((size_t)n * 8);
    const size_t o_q = o_strand + align16((size_t)n);
    StagedCall sc;
    sc.fn = fn; sc.item = "region";
    sc.n = n; sc.qbytes = qbytes; sc.n_over = n_over; sc.max_ops = max_ops; sc.score_only = score_only;
    sc.raw = o_q + align16((size_t)qbytes);
    sc.o_tbeg = o_start; sc.o_tend = o_end;
    auto stage = [&](char *h) {
        int64_t *hq = reinterpret_cast<int64_t *>(h);
        const int64_t q0 = in->query_off[0];
        for (int64_t k = 0; k <= n; ++k) hq[k] = in->query_off[k] - q0;
        memcpy(h + o_tid, in->tid, (size_t)n * 4);
        memcpy(h + o_start, in->start, (size_t)n * 8);
        memcpy(h + o_end, in->end, (size_t)n * 8);
        memcpy(h + o_strand, in->strand, (size_t)n);
        if (qbytes) parallel_copy(h + o_q, in->query + q0, (size_t)qbytes, c->host_threads);
    };
    auto prep = [&](fadegpu_job *j, const char *d, BinArgs &ba, int *launches) -> int {
        BinState &bs = j->bs;
        RegionArgs ra{};
        ra.n = n;
        ra.query = d + o_q; ra.qoff = reinterpret_cast<const int64_t *>(d);
        ra.rtid = reinterpret_cast<const int32_t *>(d + o_tid);
        ra.start = reinterpret_cast<const int64_t *>(d + o_start); ra.end = reinterpret_cast<const int64_t *>(d + o_end);
        ra.strand = reinterpret_cast<const uint8_t *>(d + o_strand);
        ra.seq_off = bs.d_in_seq_off; ra.pos = bs.d_in_pos; ra.l_qseq = bs.d_in_lq; ra.tid = bs.d_in_tid;
        ra.aligned_len = bs.d_in_alen; ra.clip_left = bs.d_in_cl; ra.clip_right = bs.d_in_cr;
        ra.seq4 = bs.d_in_seq4; ra.bad = j->d_bad;
        CU(c, launch_region_prep(ra, c->sm_count, c->stream2));
        *launches += 1;
        // the intervals were validated above, so the window arithmetic clamps nothing: gstart = coff[tid] + start
        ba.clen = c->d_clen; ba.coff = c->d_coff; ba.n_contigs = c->n_contigs;
        return 0;
    };
    sc.reference = [c](fadegpu_job *, RefDev *ref, int *) -> int { *ref = ref_dev(c); return 0; };
    return run_call(c, job, sc, stage, prep, out, ops_out, stats_out, t_begin);
}

int fadegpu_align_regions(fadegpu_ctx *c, int64_t n_regions, const fadegpu_regions *in, int32_t max_ops,
                          fadegpu_pair_result *out, uint32_t *ops_out, fadegpu_stats *stats_out)
{
    return regions_call(c, "fadegpu_align_regions", false, n_regions, in, max_ops, out, ops_out, stats_out, nullptr);
}

int fadegpu_score_regions(fadegpu_ctx *c, int64_t n_regions, const fadegpu_regions *in, fadegpu_pair_result *out,
                          fadegpu_stats *stats_out)
{
    return regions_call(c, "fadegpu_score_regions", true, n_regions, in, 0, out, nullptr, stats_out, nullptr);
}

// ---- jobs: queued pair and region calls ----

int fadegpu_job_create(fadegpu_ctx *c, fadegpu_job **out)
{
    if (!c || !out) return fail(c, FADEGPU_E_ARG, "fadegpu_job_create: null argument");
    *out = nullptr;
    fadegpu_job *j = new (std::nothrow) fadegpu_job();
    if (!j) return fail(c, FADEGPU_E_OOM, "fadegpu_job_create: out of host memory");
    j->ctx = c;
    { std::lock_guard<std::mutex> lk(c->q_mu); c->jobs.push_back(j); }
    *out = j;
    return FADEGPU_OK;
}

void fadegpu_job_destroy(fadegpu_job *j)
{
    if (!j) return;
    fadegpu_ctx *c = j->ctx;
    {
        std::unique_lock<std::mutex> lk(c->q_mu);
        c->done_cv.wait(lk, [&] { return !j->fl.queued; });
        if (j->fl.in_flight) { j->fl.in_flight = false; --c->jobs_in_flight; }
        c->jobs.erase(std::remove(c->jobs.begin(), c->jobs.end(), j), c->jobs.end());
    }
    cudaSetDevice(c->device);
    free_job(j);
}

// what every submit checks before the call's own validation: the ctx, the job's state, the job flags
static int check_job_submit(fadegpu_ctx *c, fadegpu_job *j, const char *fn, int32_t max_ops, uint32_t job_flags)
{
    const std::string at = std::string(fn) + ": ";
    if (!c || !j) return fail(c, FADEGPU_E_ARG, at + "null ctx or job");
    if (j->ctx != c) return fail(c, FADEGPU_E_STATE, at + "the job belongs to another ctx");
    if (job_flags & ~FADEGPU_JOB_SCORE_ONLY) return fail(c, FADEGPU_E_ARG, at + "unknown job flags");
    if ((job_flags & FADEGPU_JOB_SCORE_ONLY) && max_ops != 0)
        return fail(c, FADEGPU_E_ARG, at + "max_ops must be 0 with FADEGPU_JOB_SCORE_ONLY");
    {
        std::lock_guard<std::mutex> lk(c->q_mu);
        if (!j->fl.in_flight) return 0;
    }
    return fail(c, FADEGPU_E_STATE, at + "job already in flight (call fadegpu_job_wait)");
}

int fadegpu_submit_pairs(fadegpu_ctx *c, fadegpu_job *j, int64_t n_pairs, const fadegpu_pairs *in, int32_t max_ops,
                         uint32_t job_flags)
{
    const char *fn = "fadegpu_submit_pairs";
    { int rc = check_job_submit(c, j, fn, max_ops, job_flags); if (rc) return rc; }
    return pairs_call(c, fn, (job_flags & FADEGPU_JOB_SCORE_ONLY) != 0, n_pairs, in, max_ops, nullptr, nullptr, nullptr, j);
}

int fadegpu_submit_regions(fadegpu_ctx *c, fadegpu_job *j, int64_t n_regions, const fadegpu_regions *in,
                           int32_t max_ops, uint32_t job_flags)
{
    const char *fn = "fadegpu_submit_regions";
    { int rc = check_job_submit(c, j, fn, max_ops, job_flags); if (rc) return rc; }
    return regions_call(c, fn, (job_flags & FADEGPU_JOB_SCORE_ONLY) != 0, n_regions, in, max_ops, nullptr, nullptr,
                        nullptr, j);
}

int fadegpu_job_wait(fadegpu_ctx *c, fadegpu_job *j, fadegpu_stats *stats_out)
{
    if (!c || !j) return fail(c, FADEGPU_E_ARG, "fadegpu_job_wait: null ctx or job");
    if (j->ctx != c) return fail(c, FADEGPU_E_STATE, "fadegpu_job_wait: the job belongs to another ctx");
    int rc;
    std::string err;
    if (!end_flight(c, j->fl, &c->jobs_in_flight, &rc, &err)) return fail(c, FADEGPU_E_STATE, "fadegpu_job_wait: job not submitted");
    if (rc) return fail(c, rc, err);   // (a queued device half reports its outcome here)
    CU(c, cudaSetDevice(c->device));
    { int r = finish_job(c, j); if (r) return r; }
    j->n_res = j->sc.n;
    if (stats_out) *stats_out = j->st;
    return FADEGPU_OK;
}

int fadegpu_job_results_view(const fadegpu_job *j, fadegpu_job_results *r)
{
    if (!j || !r) return fail(j ? j->ctx : nullptr, FADEGPU_E_ARG, "fadegpu_job_results_view: null argument");
    bool in_flight;
    { std::lock_guard<std::mutex> lk(j->ctx->q_mu); in_flight = j->fl.in_flight; }
    if (in_flight) return fail(j->ctx, FADEGPU_E_STATE, "fadegpu_job_results_view: job in flight (call fadegpu_job_wait)");
    const int64_t n = std::max<int64_t>(0, j->n_res);
    r->n = n;
    r->records = n > 0 ? j->h_res : nullptr;
    r->ops = n > 0 && j->sc.max_ops > 0 ? j->h_ops : nullptr;
    r->max_ops = j->n_res >= 0 ? j->sc.max_ops : 0;
    r->reserved = 0;
    return FADEGPU_OK;
}

int fadegpu_measure_alu_peak(fadegpu_ctx *c, double *ops_per_sec_out, double *sm_clock_mhz_out)
{
    if (!c || !ops_per_sec_out) return fail(c, FADEGPU_E_ARG, "fadegpu_measure_alu_peak: null argument");
    CU(c, cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CU(c, cudaGetDeviceProperties(&prop, c->device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    cudaEvent_t e0, e1;
    CU(c, cudaEventCreate(&e0)); CU(c, cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CU(c, cudaEventRecord(e0, c->stream));
        CU(c, launch_alu_peak(c->d_alu, iters, blocks, threads, c->stream));
        CU(c, cudaEventRecord(e1, c->stream));
        CU(c, cudaEventSynchronize(e1));
        float ms = 0;
        CU(c, cudaEventElapsedTime(&ms, e0, e1));
        const double ops = (double)blocks * threads * (double)iters * 64.0;  // thread-instructions
        if (rep > 0 && ms > 0) best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *ops_per_sec_out = best;
    if (sm_clock_mhz_out) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, c->device);
        *sm_clock_mhz_out = khz / 1000.0;
    }
    return FADEGPU_OK;
}

}  // extern "C"
