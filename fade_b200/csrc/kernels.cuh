// kernels.cuh -- sm_100a kernels of the realignment path and their launch descriptors.
//
//   sw_fill_kernel<R>    score-only packed-int16x2 wavefront + skewed checkpoints   (P1, P2)
//   sw_trace_kernel<R>   end cell (P3), block replay with trace, traceback, CIGAR,
//                        S padding and accept predicates                            (P3-P5, F9)
//   sw_generic_kernel    exact int32 fallback ON THE DEVICE for wildcard letters and sizes the
//                        packed kernels do not cover (thread per alignment)
//   pair_*_kernel        fadegpu_align_pairs: pack caller-supplied ASCII pairs into the read / reference formats
//                        above, and put the records back into pair order (also for regions and the score-only calls)
//   region_prep_kernel   fadegpu_align_regions: pack caller-supplied queries against intervals of the reference
//   alu_peak_kernel      INT16x2 ALU issue-rate microbenchmark (roofline denominator)
//
// Window gather (source/analysis.d:45-64) and reverse complement (source/util.d:18-34) happen
// inside the kernels from the device-resident packed reference and the BAM 4-bit read bases.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "sw_core.cuh"

namespace fade {

// one alignment = one read with at least one qualifying clip (the left and the right clip of a
// read are the same SW problem, source/analysis.d:40-67, so it is computed once)
struct AlnDesc {
    int64_t gstart;    // global base offset of the window start inside the packed reference
    int64_t seq_off;   // byte offset of the read's 4-bit bases inside the gathered buffer
    int32_t tlen;      // window length (end - start)
    int32_t qlen;      // l_qseq
    uint32_t clip_left, clip_right;
    int32_t read;      // index of the read inside the batch
    int32_t pad;
};

// one warp = 4 groups = 4 pairs = 8 consecutive alignments of the length-sorted list
struct WarpItem {
    int64_t ck_off;    // word offset of this warp's checkpoints inside the scratch
    int32_t first;     // index of its first alignment
    int16_t nblk;      // number of 32-step blocks (uniform over the warp)
    int16_t pad;
    int32_t nsteps;    // wavefront steps of the score-only pass: tmax + FG - 1
};

struct RefDev {
    RefPlanes planes;
    const int64_t *xpos;   // sorted global positions of wildcard bases
    const uint8_t *xchr;   // their upper-cased letters
    int64_t n_x;
};

struct KernelArgs {
    const AlnDesc *aln;
    int32_t n_aln;
    const WarpItem *items;
    int32_t n_items;
    const uint8_t *seq;        // gathered 4-bit read bases
    RefDev ref;
    uint32_t *ck;              // checkpoint scratch
    uint2 *fillres;            // [n_items*32] per thread: (running max M, first-reached block lo|hi<<16)
    uint32_t *aln_flags;       // [n_aln] bit0: needs the generic kernel (wildcard letter seen)
    AlnOut *out;               // [n_aln]
    SwConsts k;
    int32_t min_length;
    int32_t tw_stride;         // uint16 elements per group in shared memory
    // traceback rounds
    LaneCtl *state;            // [n_aln] per-alignment traceback state
    unsigned long long *queue[2];  // request queues (ping-pong): aln | blk << 32 | scanmask << 48
    unsigned int *qcount;      // [2]
    uint32_t *tiles;           // [ceil(n_aln/2)] trace tiles of the current round
    int32_t round, max_rounds;
    int32_t tags_only;         // FADEGPU_F_TAGS_ONLY
    uint32_t *ops_spill;       // [n_aln * ops_cap] full reversed-op ring per alignment (ctl_advance); nullptr = none
    int32_t ops_cap;
};

struct GenericArgs {
    const AlnDesc *aln;
    int32_t n_aln;
    const uint32_t *aln_flags; // nullptr = every alignment of the list
    const uint8_t *seq;
    RefDev ref;
    AlnOut *out;
    unsigned int *cursor;      // work counter
    uint8_t *scratch;          // n_slots * slot_bytes
    int64_t slot_bytes;
    int32_t qmax, tmax;
    int32_t n_slots;           // threads that own a scratch slot
    int32_t chunk;             // work items claimed per atomic
    int32_t open, extend, match, mismatch, min_length;
    int32_t tags_only;         // FADEGPU_F_TAGS_ONLY
    uint32_t *ops_spill;       // as KernelArgs::ops_spill
    int32_t ops_cap;
};

// ---- binning on the device (pinned-view submits): classify reads, histogram by (class, window
//      length), scatter the alignment descriptors into sorted order ----
struct BinArgs {
    // device mirrors of the batch inputs
    const uint8_t *seq4;
    int64_t *seq_off;
    int32_t *l_qseq, *tid;
    int64_t *pos;
    int32_t *aligned_len, *clip_left, *clip_right;
    const int32_t *read;            // [n] index of each entry in the caller's batch (nullptr = identity)
    int64_t n, seq_total;
    const int64_t *clen, *coff;     // contig lengths / global base offsets
    int32_t n_contigs, window, min_length;
    uint32_t flags;                 // FADEGPU_F_*
    // classify outputs
    int32_t *key;                   // [n] sort key, -1 = no SW for this read
    int32_t *tlen;                  // [n]
    int64_t *start;                 // [n] window start inside the contig
    int32_t *hist;                  // [BIN_KEYS]
    unsigned long long *stats;      // [0..6] cells, n_aln, qmax_all, tmax_all, qmax_generic, tmax_generic, bad;
                                    // [8] bytes of bases pulled, [10] records fetched (compact inputs)
    // scatter
    const int32_t *keybase;         // [BIN_KEYS] first sorted position of each key
    int32_t *cursor;                // [BIN_KEYS]
    AlnDesc *aln;
    int64_t *aln_start;
    // compact inputs (fadegpu_submit_compact): one gate byte per read on the device, the 32-byte records stay in
    // the caller's pinned view; the classify kernel fetches those of the reads that pass the length floor and
    // stores their fields into the (writable) device mirrors above
    int32_t *over_list;             // [OVER_CAP] reads whose window exceeds 2^31 DP cells (left unaligned, reported); count in stats[11]
    const uint8_t *gate;            // [n] device copy; nullptr = the seven input arrays above are complete
    const uint4 *host_meta;         // [2n] device-mapped address of the view's fadegpu_read_meta records
    // pull mode (the bases stay in the caller's pinned view until the GPU fetches the ones it needs)
    unsigned long long *seq_cursor; // device byte cursor into the compact sequence buffer; nullptr = seq_off is final
    int64_t *src_off;               // [n_aln] offset of each alignment's bases in the pinned view
};

// ---- pairs of caller-supplied sequences (fadegpu_align_pairs): the raw ASCII is packed on the device into the
//      formats the binning and the SW kernels read -- the targets become the "contigs" of a reference of their own ----
struct PairArgs {
    int64_t n;
    const char *query, *target;     // concatenated ASCII
    const int64_t *qoff, *toff;     // [n+1], starting at 0
    // per-pair inputs of the binning (tid = k, pos = 0, aligned_len = tlen, clip_left = qlen, clip_right = 0)
    int64_t *seq_off, *pos;
    int32_t *l_qseq, *tid, *aligned_len, *clip_left, *clip_right;
    int64_t *clen, *coff;           // contig table: target k starts at coff[k] = 32 * (k + toff[k] / 32)
    uint8_t *seq4;                  // queries as BAM nt16 nibbles, reverse-complemented, query k at byte qoff[k]
    int32_t *bad;                   // lowest pair whose query holds a letter outside nt16 (atomicMin; starts at n)
    // target planes (DESIGN 3) and the sorted wildcard list
    uint32_t *two, *nmask, *xmask;
    int64_t n_words;                // 32-base words of the planes
    uint32_t *chunk_x;              // [n_chunks] wildcard letters per chunk of PAIR_CHUNK_WORDS words
    unsigned long long *n_x;        // their total
    int64_t *xpos;
    uint8_t *xchr;
};
constexpr int PAIR_CHUNK_WORDS = 1024;
// qlen * tlen above this is not aligned (FADEGPU_R_OVERSIZE), as for reads
constexpr int64_t PAIR_MAX_CELLS = (int64_t)1 << 31;
constexpr uint32_t PAIR_R_OVERSIZE = 32u;   // FADEGPU_R_OVERSIZE
cudaError_t launch_pair_prep(const PairArgs &a, int sm_count, cudaStream_t s);
cudaError_t launch_pair_pack_targets(const PairArgs &a, cudaStream_t s);   // planes + chunk_x + n_x
cudaError_t launch_pair_xlist(const PairArgs &a, cudaStream_t s);          // xpos / xchr (after n_x is known)
// ---- caller-supplied queries against intervals of the resident reference (fadegpu_align_regions): only the queries
//      are packed; the binning runs on the ctx's own contig table ----
struct RegionArgs {
    int64_t n;
    const char *query;              // concatenated ASCII
    const int64_t *qoff;            // [n+1], starting at 0
    const int32_t *rtid;            // [n] contig of the interval
    const int64_t *start, *end;     // [n] interval [start, end) on the contig (validated by the host)
    const uint8_t *strand;          // [n] 0: the query as given, 1: its reverse complement
    // per-region inputs of the binning (pos = start, aligned_len = end - start, clip_left = qlen, clip_right = 0)
    int64_t *seq_off, *pos;
    int32_t *l_qseq, *tid, *aligned_len, *clip_left, *clip_right;
    uint8_t *seq4;                  // queries as BAM nt16 nibbles, stored so that the kernels' reverse complement gives
                                    // the strand's letters, query k at byte qoff[k]
    int32_t *bad;                   // lowest region whose query holds a letter outside nt16 (atomicMin; starts at n)
};
cudaError_t launch_region_prep(const RegionArgs &a, int sm_count, cudaStream_t s);
// item-ordered result records (pairs or regions): zeros (or FADEGPU_R_OVERSIZE) for every item k, whose query is
// qoff[k] .. qoff[k+1] and whose window spans t_beg[k] .. t_end[k] (pairs: toff, toff + 1; regions: start, end), then
// the records of the alignments with their full forward CIGARs assembled from the spill rings (score_only: score and end
// cell only, no spill rings, max_ops = 0); n_ok counts the records the SW kernels produced
struct PairResult {   // == fadegpu_pair_result
    int32_t score, end_query, end_ref, beg_query, beg_ref, n_ops;
    uint32_t flags;
    int32_t reserved;
};
cudaError_t launch_pair_results(int64_t n, const int64_t *qoff, const int64_t *t_beg, const int64_t *t_end,
                                const AlnDesc *aln, const AlnOut *out, int n_aln, bool score_only, const uint32_t *spill,
                                int max_ops, PairResult *res, uint32_t *ops, unsigned long long *n_ok, int sm_count,
                                cudaStream_t s);

constexpr int FILL_THREADS = 128;
constexpr int OVER_CAP = 256;        // oversize reads listed per batch (all of them are counted)
// row classes: R rows per thread x 8 threads cover reads of up to 104 / 152 / 200 / 256 / 304 bases
constexpr int N_ROW_CLASSES = 5;
__host__ __device__ constexpr int row_class(int k) { return k == 0 ? 13 : k == 1 ? 19 : k == 2 ? 25 : k == 3 ? 32 : 38; }
constexpr int ROW_CLASSES[N_ROW_CLASSES] = { row_class(0), row_class(1), row_class(2), row_class(3), row_class(4) };
constexpr int QMAX_FAST = FG * 38;   // rows covered by the largest packed instantiation
// Window lengths: up to TMAX_FAST every length is its own sort key; longer windows (spliced records: alignedLength
// spans the introns, analysis.d:53) share keys of TLONG_STEP columns up to TMAX_PACKED, beyond which only the generic
// kernel serves them.  TMAX_PACKED keeps block numbers (32 steps each) within 16 bits.
constexpr int TMAX_FAST = 4000;
constexpr int TLONG_STEP = 1024;
constexpr int TMAX_PACKED = 1000000;
constexpr int N_LONG_KEYS = (TMAX_PACKED - TMAX_FAST + TLONG_STEP - 1) / TLONG_STEP;
constexpr int KEYS_PER_CLASS = N_LONG_KEYS + TMAX_FAST + 2;
// The fill kernel keeps the target words of FILL_CHUNK_BLOCKS * 32 steps per pair in shared memory (2 KB) and
// restages them for longer windows, so that its occupancy does not depend on the longest window of a launch.
constexpr int FILL_CHUNK_BLOCKS = 32;

size_t fill_smem_bytes(int tw_stride);
size_t trace_tile_bytes(int R);
int tw_stride_for(int nblk_max);

constexpr int BIN_KEYS = (N_ROW_CLASSES + 1) * KEYS_PER_CLASS;
// sort key: class rank (ROW_CLASSES order, then the generic list) and descending window length
__host__ __device__ inline int bin_key(int rank, int tlen)
{
    if (rank == N_ROW_CLASSES) return rank * KEYS_PER_CLASS;
    return rank * KEYS_PER_CLASS + (tlen > TMAX_FAST ? (TMAX_PACKED - tlen) / TLONG_STEP : N_LONG_KEYS + TMAX_FAST - tlen);
}
// the window length a key stands for in the launch plan: exact up to TMAX_FAST, the upper end of the key's range beyond
__host__ __device__ inline int key_tlen(int key_in_class)
{
    return key_in_class < N_LONG_KEYS ? TMAX_PACKED - key_in_class * TLONG_STEP : TMAX_FAST - (key_in_class - N_LONG_KEYS);
}
__host__ __device__ inline int bin_rank(int qlen, int tlen, bool force_generic)
{
    if (force_generic || qlen > QMAX_FAST || tlen > TMAX_PACKED) return N_ROW_CLASSES;
    for (int k = 0; k < N_ROW_CLASSES; ++k) if (qlen <= FG * row_class(k)) return k;
    return N_ROW_CLASSES;
}
cudaError_t launch_bin_classify(const BinArgs &a, int sm_count, cudaStream_t s);
cudaError_t launch_bin_scatter(const BinArgs &a, int sm_count, cudaStream_t s);
cudaError_t launch_seq_pull(const uint8_t *host_seq4, const AlnDesc *aln, const int64_t *src_off, int n_aln, uint8_t *dst, int sm_count,
                            cudaStream_t s);
cudaError_t launch_result_index(const AlnOut *out, int n_aln, int64_t n_reads, uint8_t *flags, int32_t *ridx, unsigned long long *n_ok,
                                int sm_count, cudaStream_t s);
cudaError_t launch_fill(int R, const KernelArgs &a, cudaStream_t s);
// end_only (score-only calls): scan-only rounds that stop at the end cell, no traceback
cudaError_t launch_trace(int R, const KernelArgs &a, bool end_only, cudaStream_t s, int sm_count, int *launches);
cudaError_t launch_generic(const GenericArgs &a, int n_slots, cudaStream_t s);
cudaError_t launch_alu_peak(uint32_t *out, int iters, int blocks, int threads, cudaStream_t s);

}  // namespace fade
