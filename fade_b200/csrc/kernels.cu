// kernels.cu -- hand-written sm_100a kernels for the `fade annotate` realignment path.
// See kernels.cuh for the inventory and sw_core.cuh for the arithmetic they share with the CPU
// emulation.  Reference semantics: source/analysis.d:34-80,98-104 + parasail rules P1-P5.
#include "kernels.cuh"
#include <algorithm>
#include <cstdio>
#include <cstdlib>

namespace fade {

namespace {

constexpr unsigned FULL = 0xffffffffu;

// Footprint of the helper kernels that run UNDER a fill (binning of the next batch, traceback bookkeeping):
// 128 threads x <= 32 registers = 4096 registers, exactly what five resident fill blocks (5 x 128 x 96) leave
// free on an SM, so one such block per SM is resident at once without waiting for a fill block to retire.
#define FADE_SMALL_KERNEL __launch_bounds__(128, 16)


// Stage one pair: target selector words (window gather from the packed reference,
// source/analysis.d:45-64) into shared memory, query selector words (reverse complement of the
// BAM 4-bit bases, source/util.d:18-34) into registers.  `wild` gets bit0/bit1 when alignment
// a/b contains a letter outside ACGTN (those go to the generic kernel).
// Target selector words of the steps [step0, step0 + nsteps) of one pair: columns step0 - FG .. step0 + nsteps - 1 at
// tw[0 ..], i.e. column j at tw[j - step0 + FG].  Windows longer than FILL_CHUNK_STEPS are staged chunk by chunk.
__device__ __forceinline__ uint32_t stage_targets(const KernelArgs &a, const AlnDesc &da, const AlnDesc &db, int g,
                                                  int step0, int nsteps, uint16_t *tw)
{
    const int TW = nsteps + FG + 1;
    uint32_t w = 0;
    for (int idx = g; idx < TW; idx += FG) {
        const int j = step0 + idx - FG;
        int ca = C_TPAD, cb = C_TPAD;
        if (j >= 0 && j < da.tlen) ca = ref_code(a.ref.planes, da.gstart + j);
        if (j >= 0 && j < db.tlen) cb = ref_code(a.ref.planes, db.gstart + j);
        w |= (ca == C_WILD ? 1u : 0u) | (cb == C_WILD ? 2u : 0u);
        tw[idx] = (uint16_t)t_sel(ca, cb);
    }
    return w;
}

// STEP: query words of that score-only step (score_step, sw_core.cuh)
template <int R, int STEP>
__device__ __forceinline__ void stage_pair(const KernelArgs &a, const AlnDesc &da, const AlnDesc &db,
                                           int g, int nblk, uint16_t *tw, uint32_t (&qs)[query_words<R, STEP>()],
                                           uint8_t *qc, uint32_t &wild)
{
    uint32_t w = stage_targets(a, da, db, g, 0, FBLK * min(nblk, FILL_CHUNK_BLOCKS), tw);
    const uint8_t *sa = a.seq + da.seq_off, *sb = a.seq + db.seq_off;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int i = g * R + r;
        int ca = C_QPAD, cb = C_QPAD;
        if (i < da.qlen) ca = rc_query_code(sa, da.qlen, i);
        if (i < db.qlen) cb = rc_query_code(sb, db.qlen, i);
        w |= (ca == C_WILD ? 1u : 0u) | (cb == C_WILD ? 2u : 0u);
        set_query<STEP>(qs, r, ca, cb);
        if (qc) qc[i] = (uint8_t)(ca | (cb << 4));
    }
    wild = w;
}

__device__ __forceinline__ AlnDesc load_desc(const KernelArgs &a, int idx)
{
    AlnDesc d;
    if (idx < a.n_aln) d = a.aln[idx];
    else { d.gstart = 0; d.seq_off = 0; d.tlen = 0; d.qlen = 0; d.clip_left = d.clip_right = 0; d.read = -1; d.pad = 0; }
    return d;
}

// ------------------------------------------------------------------------------------------------
// score-only wavefront with checkpoints
// ------------------------------------------------------------------------------------------------
template <int R, int STEP>
__global__ void __launch_bounds__(FILL_THREADS, (R <= 19 ? 5 : 1)) sw_fill_kernel(const KernelArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = lane & (FG - 1), q = lane >> 3;
    const int w = blockIdx.x * (FILL_THREADS / 32) + wib;
    if (w >= a.n_items) return;
    const WarpItem item = a.items[w];
    const int ia = item.first + 2 * q, ib = ia + 1;
    const AlnDesc da = load_desc(a, ia), db = load_desc(a, ib);
    uint16_t *tw = reinterpret_cast<uint16_t *>(smem_raw) + (size_t)(wib * 4 + q) * a.tw_stride;
    const int nblk = item.nblk;
    const SwConsts k = a.k;

    uint32_t H[R], E[R], qs[query_words<R, STEP>()];
    uint32_t wild;
    stage_pair<R, STEP>(a, da, db, g, nblk, tw, qs, nullptr, wild);
#pragma unroll
    for (int r = 0; r < R; ++r) { H[r] = 0u; E[r] = k.neg_o; }
    uint32_t hu_prev = 0u, fout = k.neg_o, M = 0u, Mprev = 0u;
    int blk_lo = 0, blk_hi = 0;
    __syncwarp();

    constexpr int CW = ck_words<R>();
    uint32_t *ckw = a.ck + item.ck_off + lane;
    const uint16_t *twp = tw + (FG - g);
    const int nsteps = item.nsteps;   // tmax + FG - 1: the last block may be partial
    for (int c = 0; c < nblk; ++c) {
        if (c > 0 && (c % FILL_CHUNK_BLOCKS) == 0) {
            // a window longer than the staged chunk: the group replaces its target words by the next chunk's
            __syncwarp();
            wild |= stage_targets(a, da, db, g, c * FBLK, FBLK * min(nblk - c, FILL_CHUNK_BLOCKS), tw);
            twp = tw + (FG - g) - c * FBLK;
            __syncwarp();
        }
        const int ulim = min(FBLK, nsteps - c * FBLK);
#pragma unroll 2
        for (int u = 0; u < ulim; ++u) {
            const int t = c * FBLK + u;
            uint32_t hu = __shfl_up_sync(FULL, H[R - 1], 1, FG);
            uint32_t fin = __shfl_up_sync(FULL, fout, 1, FG);
            if (g == 0) { hu = 0u; fin = k.neg_o; }
            const uint32_t ts = twp[t];
            score_step<R, STEP>(H, E, qs, M, ts, hu_prev, fin, fout, k);
            hu_prev = hu;
        }
        if (c + 1 < nblk) {
            uint32_t *p = ckw + (size_t)c * CW * 32;
#pragma unroll
            for (int r = 0; r < R; ++r) { p[r * 32] = H[r]; p[(R + r) * 32] = E[r]; }
            p[(2 * R) * 32] = hu_prev;
            p[(2 * R + 1) * 32] = fout;
        }
        if (M != Mprev) {
            if ((M ^ Mprev) & 0xffffu) blk_lo = c;
            if ((M ^ Mprev) >> 16) blk_hi = c;
            Mprev = M;
        }
    }
    a.fillres[(size_t)w * 32 + lane] = make_uint2(M, (uint32_t)blk_lo | ((uint32_t)blk_hi << 16));
    if ((wild & 1u) && ia < a.n_aln) a.aln_flags[ia] = 1u;
    if ((wild & 2u) && ib < a.n_aln) a.aln_flags[ib] = 1u;
}

// ------------------------------------------------------------------------------------------------
// end cell + traceback by block replay, organised as rounds over a device-side request queue:
//   trace_init_kernel     per alignment: collect the per-thread maxima of the score-only pass,
//                         pick the first block to replay, enqueue (alignment, block, scan mask)
//   trace_replay_kernel   per PAIR OF REQUESTS (any two alignments): reload the wavefront state of
//                         the requested block from the checkpoints, re-run its 32 steps with
//                         (tagged) trace recording, write the trace tile, report scan hits
//   trace_advance_kernel  per request: end-cell selection / traceback walk through the tile;
//                         either finishes the alignment (CIGAR, predicates, AlnOut) or enqueues
//                         the next block it needs
// Requests are paired by queue position, so every replay does useful work for two alignments and
// no thread waits for a slower neighbour.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long pack_req(int aln, int blk, uint32_t scanmask)
{
    return (unsigned long long)(uint32_t)aln | ((unsigned long long)(uint32_t)(blk & 0xffff) << 32) |
           ((unsigned long long)(scanmask & 0xffu) << 48);
}

struct GlobalAcc {
    const uint8_t *seq;
    int qlen;
    RefPlanes planes;
    int64_t gstart;
    __device__ __forceinline__ int qcode(int i) const { return rc_query_code(seq, qlen, i); }
    __device__ __forceinline__ int tcode(int j) const { return ref_code(planes, gstart + j); }
};

template <int R>
__global__ void FADE_SMALL_KERNEL trace_init_kernel(const KernelArgs a)
{
    for (int aln = blockIdx.x * blockDim.x + threadIdx.x; aln < a.n_aln; aln += gridDim.x * blockDim.x) {
        a.out[aln].read = -1;              // "no result yet": fadegpu_wait refuses such a record
        a.out[aln].flags = 0x80000000u;
        if (a.aln_flags[aln] & 1u) continue;   // wildcard letter: the generic kernel produces it
        const AlnDesc d = a.aln[aln];
        LaneCtl &c = a.state[aln];
        const int w = aln >> 3, q = (aln & 7) >> 1, half = aln & 1;
        const uint2 *fr = a.fillres + (size_t)w * 32 + q * FG;
        for (int g = 0; g < FG; ++g) {
            const uint2 v = fr[g];
            c.best[g] = half ? lane_hi(v.x) : lane_lo(v.x);
            c.blk[g] = half ? (int)(v.y >> 16) : (int)(v.y & 0xffffu);
        }
        ctl_init(c, d.qlen, d.tlen);
        if (c.phase != 2 && a.tags_only && !score_may_accept(c.S, d.clip_left, d.clip_right, a.min_length)) {
            // FADEGPU_F_TAGS_ONLY: the score already rules out both accept predicates (analysis.d:76,100): no end cell, no
            // traceback; the record carries the score and FADEGPU_R_SCORE_ONLY
            AlnOut o;
            o.score = c.S; o.end_query = o.end_ref = o.beg_query = o.beg_ref = 0; o.n_ops = 0;
            o.flags = R_ALIGNED | R_SCORE_ONLY; o.read = d.read;
            for (int k = 0; k < OPS_CAP; ++k) o.ops[k] = 0;
            a.out[aln] = o;
        } else if (c.phase == 2) {
            AlnOut o;
            finalize_result(c, o, d.read, d.clip_left, d.clip_right, a.min_length);
            a.out[aln] = o;
        } else {
            const unsigned slot = atomicAdd(&a.qcount[0], 1u);
            a.queue[0][slot] = pack_req(aln, c.next_blk, ctl_scanmask(c));
        }
    }
}

// MODE 0: tagged trace recording, 1: plain trace recording, 2: scan only (round 0: find the end cell,
// no trace tile; the traceback then tries the ungapped-diagonal proof before asking for a traced replay)
// with the score-only step STEP (score_step)
template <int R, int MODE, int STEP = 0>
__device__ __forceinline__ void replay_round(const KernelArgs &a, int round, unsigned warp0, unsigned nwarps,
                                             uint16_t (*tws_all)[40])
{
    constexpr bool TAGGED = MODE == 0;
    constexpr bool SCAN_ONLY = MODE == 2;
    constexpr int RW = trace_words<R>();
    constexpr int CW = ck_words<R>();
    constexpr int MUL = TAGGED ? 16 : 1;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int g = lane & (FG - 1), q = lane >> 3;
    const int rin = round & 1;
    const unsigned cnt = a.qcount[rin];
    const unsigned long long *queue = a.queue[rin];
    const unsigned npairs = (cnt + 1u) >> 1;
    const unsigned nquads = (npairs + 3u) >> 2;
    const SwConsts k = a.k;
    const uint32_t e_init = TAGGED ? k.neg_o16 : k.neg_o;
    uint16_t *tws = tws_all[wib * 4 + q];
    for (unsigned quad = warp0; quad < nquads; quad += nwarps) {
        const unsigned pair = quad * 4u + (unsigned)q;
        // ---- the two requests of this group ----
        int aln[2], blk[2], half[2], S[2];
        uint32_t smask[2];
        AlnDesc d[2];
        const uint32_t *ckp[2];
#pragma unroll
        for (int L = 0; L < 2; ++L) {
            const unsigned ri = pair * 2u + (unsigned)L;
            if (ri < cnt) {
                const unsigned long long rq = queue[ri];
                aln[L] = (int)(uint32_t)(rq & 0xffffffffu);
                blk[L] = (int)((rq >> 32) & 0xffffu);
                smask[L] = (uint32_t)((rq >> 48) & 0xffu);
                d[L] = a.aln[aln[L]];
                const WarpItem it = a.items[aln[L] >> 3];
                ckp[L] = a.ck + it.ck_off + (((aln[L] & 7) >> 1) * FG + g);
                half[L] = aln[L] & 1;
                S[L] = a.state[aln[L]].S * MUL;
            } else {
                aln[L] = -1; blk[L] = 0; smask[L] = 0; half[L] = 0; S[L] = -1; ckp[L] = a.ck;
                d[L].gstart = 0; d[L].seq_off = 0; d[L].tlen = 0; d[L].qlen = 0;
            }
        }
        // ---- wavefront state of the requested blocks (checkpoints are in the plain domain) ----
        uint32_t H[R], E[R], qs[query_words<R, STEP>()], hu_prev, fout;
        {
            const uint32_t *p0 = ckp[0] + (size_t)(blk[0] > 0 ? blk[0] - 1 : 0) * CW * 32;
            const uint32_t *p1 = ckp[1] + (size_t)(blk[1] > 0 ? blk[1] - 1 : 0) * CW * 32;
            const bool z0 = blk[0] == 0, z1 = blk[1] == 0;
            const int sh0 = half[0] * 16, sh1 = half[1] * 16;
            auto mix = [&](uint32_t w0, uint32_t w1) {
                const uint32_t w = ((w0 >> sh0) & 0xffffu) | ((w1 >> sh1) << 16);
                return TAGGED ? to_tagged(w) : w;
            };
#pragma unroll
            for (int r = 0; r < R; ++r) {
                H[r] = mix(z0 ? 0u : p0[r * 32], z1 ? 0u : p1[r * 32]);
                E[r] = mix(z0 ? k.neg_o : p0[(R + r) * 32], z1 ? k.neg_o : p1[(R + r) * 32]);
            }
            hu_prev = mix(z0 ? 0u : p0[(2 * R) * 32], z1 ? 0u : p1[(2 * R) * 32]);
            fout = mix(z0 ? k.neg_o : p0[(2 * R + 1) * 32], z1 ? k.neg_o : p1[(2 * R + 1) * 32]);
        }
        // ---- query rows (reverse complement of the BAM nibbles) and the 39 target columns ----
        {
            const uint8_t *s0 = a.seq + d[0].seq_off, *s1 = a.seq + d[1].seq_off;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const int i = g * R + r;
                const int ca = i < d[0].qlen ? rc_query_code(s0, d[0].qlen, i) : C_QPAD;
                const int cb = i < d[1].qlen ? rc_query_code(s1, d[1].qlen, i) : C_QPAD;
                set_query<STEP>(qs, r, ca, cb);
            }
            __syncwarp();   // previous iteration's readers of tws are done
            for (int x = g; x < FBLK + FG - 1; x += FG) {
                const int j0 = blk[0] * FBLK - (FG - 1) + x, j1 = blk[1] * FBLK - (FG - 1) + x;
                const int ca = (j0 >= 0 && j0 < d[0].tlen) ? ref_code(a.ref.planes, d[0].gstart + j0) : C_TPAD;
                const int cb = (j1 >= 0 && j1 < d[1].tlen) ? ref_code(a.ref.planes, d[1].gstart + j1) : C_TPAD;
                tws[x] = (uint16_t)t_sel(ca, cb);
            }
            __syncwarp();
        }
        // ---- replay ----
        uint32_t *tile = a.tiles + (size_t)pair * tile_words<R>();
        const bool store = aln[0] >= 0;      // a pair without requests computes padding only
        bool need0 = (smask[0] >> g) & 1u, need1 = (smask[1] >> g) & 1u;
        const uint16_t *twp = tws + (FG - 1 - g);
        for (int u = 0; u < FBLK; ++u) {
            uint32_t hu = __shfl_up_sync(FULL, H[R - 1], 1, FG);
            uint32_t fin = __shfl_up_sync(FULL, fout, 1, FG);
            if (g == 0) { hu = 0u; fin = e_init; }
            const uint32_t ts = twp[u];
            uint32_t cmax = 0u;
            if constexpr (SCAN_ONLY) {
                score_step<R, STEP>(H, E, qs, cmax, ts, hu_prev, fin, fout, k);
            } else {
                uint32_t trw[RW];
                if (TAGGED) trace_step_tagged<R>(H, E, qs, ts, hu_prev, fin, fout, k, trw, cmax);
                else trace_step_plain<R>(H, E, qs, ts, hu_prev, fin, fout, k, trw, cmax);
                if (store) {
#pragma unroll
                    for (int w = 0; w < RW; ++w) tile[tile_index<R>(u, g, w)] = trw[w];
                }
            }
            hu_prev = hu;
            if (need0 && lane_lo(cmax) == S[0]) {
                need0 = false;
                int fr = 0;
#pragma unroll
                for (int r = R - 1; r >= 0; --r) if (lane_lo(H[r]) == S[0]) fr = r;
                a.state[aln[0]].fj[g] = blk[0] * FBLK + u - g;
                a.state[aln[0]].fr[g] = fr;
            }
            if (need1 && lane_hi(cmax) == S[1]) {
                need1 = false;
                int fr = 0;
#pragma unroll
                for (int r = R - 1; r >= 0; --r) if (lane_hi(H[r]) == S[1]) fr = r;
                a.state[aln[1]].fj[g] = blk[1] * FBLK + u - g;
                a.state[aln[1]].fr[g] = fr;
            }
            if (SCAN_ONLY && !__any_sync(FULL, need0 || need1)) break;   // every end-cell candidate found
        }
    }
}

template <int R, int MODE, int STEP = 0>
__global__ void __launch_bounds__(128) trace_replay_kernel(const KernelArgs a)
{
    __shared__ uint16_t tws_all[16][40];
    if (blockIdx.x == 0 && threadIdx.x == 0) a.qcount[(a.round & 1) ^ 1] = 0u;   // next round's queue starts empty
    replay_round<R, MODE, STEP>(a, a.round, blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5),
                                gridDim.x * (blockDim.x >> 5), tws_all);
}

// One WARP per request.  The traceback is a pointer chase; to avoid one L2 round trip per step the
// 32 lanes fetch the trace nibbles (and symbol codes) of the next 32 cells of the DIAGONAL through
// the current cell at once, speculating that the path keeps going diagonally (gaps cost >= 10, so
// it almost always does); a prefix sum of the step scores gives every lane the H value its cell
// would have, the first lane whose step is not "DIAG with H > 0" ends the batch.  Gap steps are
// taken one at a time.  Semantics are exactly those of ctl_advance (sw_core.cuh).
struct AdvanceSmem {
    LaneCtl ctl;     // staged copy of the alignment's traceback state
    AlnOut out;      // result record, written out coalesced
};
static_assert(sizeof(LaneCtl) % 4 == 0 && sizeof(AlnOut) % 4 == 0, "word-copyable");

// SPILL: the launch may carry a full-CIGAR spill ring (a.ops_spill, checked at run time); without it the walker is
// compiled exactly as for the annotate path.  END_ONLY (score-only calls): an alignment is done once its end cell is
// selected -- no walk, no traced replay requested, a finalize_end record.
template <int R, bool SPILL, bool END_ONLY = false>
__device__ __forceinline__ void advance_round(const KernelArgs &a, int round, unsigned warp0, unsigned nwarps,
                                              AdvanceSmem *smem_all)
{
    constexpr int RW = trace_words<R>();
    constexpr int CTLW = (int)(sizeof(LaneCtl) / 4), OUTW = (int)(sizeof(AlnOut) / 4);
    AdvanceSmem &sm = smem_all[threadIdx.x >> 5];
    const int rin = round & 1;
    const unsigned cnt = a.qcount[rin];
    const unsigned long long *queue = a.queue[rin];
    const int l = threadIdx.x & 31;
    const SwConsts &k = a.k;
    const bool tile_valid = !(round == 0 && k.shortcut);   // round 0 only scans for the end cell
    for (unsigned idx = warp0; idx < cnt; idx += nwarps) {
        const int aln = (int)(uint32_t)(queue[idx] & 0xffffffffu);
        const AlnDesc d = a.aln[aln];
        // stage the state in shared memory: one coalesced round trip instead of dozens of dependent ones
        LaneCtl &c = sm.ctl;
        {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(&a.state[aln]);
            uint32_t *dst = reinterpret_cast<uint32_t *>(&c);
            for (int w = l; w < CTLW; w += 32) dst[w] = src[w];
        }
        __syncwarp();
        const uint32_t *tile = a.tiles + (size_t)(idx >> 1) * tile_words<R>();
        const int sh = 16 * (int)(idx & 1u);
        GlobalAcc acc;
        acc.seq = a.seq + d.seq_off; acc.qlen = d.qlen; acc.planes = a.ref.planes; acc.gstart = d.gstart;
        // ---- phase 0 bookkeeping by lane 0, then every lane reads the (uniform) state ----
        int go = 1;
        if (l == 0) {
            c.cur_blk = c.next_blk;
            if (c.phase == 0 && !ctl_select_end<R>(c)) go = 0;
            if constexpr (END_ONLY) {
                if (go) { c.phase = 2; c.next_blk = -1; go = 0; }
            }
        }
        go = __shfl_sync(FULL, go, 0);
        __syncwarp();
        bool done = false;
        int need = -1;
        if (go) {
            int i = 0, j = 0, mode = 0, hval = 0, gval = 0, nrev = 0, cur_blk_ = 0;
            uint32_t cur = 0;
            if (l == 0) {
                i = c.i; j = c.j; mode = c.mode; hval = c.hval; gval = c.gval; nrev = c.nrev; cur = c.cur;
                cur_blk_ = c.cur_blk;
            }
            i = __shfl_sync(FULL, i, 0); j = __shfl_sync(FULL, j, 0); mode = __shfl_sync(FULL, mode, 0);
            hval = __shfl_sync(FULL, hval, 0); gval = __shfl_sync(FULL, gval, 0); nrev = __shfl_sync(FULL, nrev, 0);
            cur = __shfl_sync(FULL, cur, 0);
            const int cur_blk = __shfl_sync(FULL, cur_blk_, 0);
            auto push_n = [&](uint32_t op, int n) {
                if (cur != 0 && (cur & 0xf) == op) { cur += 16u * (uint32_t)n; return; }
                if (cur != 0) {
                    if (l == 0) {
                        c.ring[nrev % OPS_CAP] = cur;
                        if (SPILL && a.ops_spill) a.ops_spill[(size_t)aln * a.ops_cap + nrev % a.ops_cap] = cur;
                    }
                    ++nrev;
                }
                cur = ((uint32_t)n << 4) | op;
            };
            int forced = 0;   // > 0: the next `forced` steps are DIAG by the ungapped-diagonal proof
            for (;;) {
                if (i < 0 || j < 0) { done = true; break; }
                if (mode == 0 && hval <= 0) { done = true; break; }   // ZERO
                if (mode == 0) {
                    // speculative diagonal batch: lane l looks at cell (i-l, j-l)
                    const int ii = i - l, jj = j - l;
                    const bool valid = ii >= 0 && jj >= 0;
                    const int g = valid ? ii / R : 0, r = valid ? ii - g * R : 0;
                    const int t = jj + g;
                    const bool inblk = valid && tile_valid && (t / FBLK) == cur_blk;
                    uint32_t nib = 0;
                    int sc = 0;
                    bool eq = false;
                    if (valid && (inblk || forced > 0)) {
                        eq = acc.qcode(ii) == acc.tcode(jj);
                        sc = eq ? k.match : k.mismatch;
                    }
                    if (inblk && forced == 0)
                        nib = (tile[tile_index<R>(t % FBLK, g, r >> 2)] >> (sh + 4 * (r & 3))) & 0xfu;
                    const bool diag = forced > 0 ? (valid && l < forced) : (inblk && (nib >> 2) == 2u);
                    if (!diag) sc = 0;
                    int pre = sc;                       // inclusive prefix sum over lanes
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int v = __shfl_up_sync(FULL, pre, o);
                        if (l >= o) pre += v;
                    }
                    const int hv = hval - (pre - sc);   // H of this lane's cell if all earlier steps were DIAG
                    const bool ok = diag && hv > 0;
                    const unsigned bad = __ballot_sync(FULL, !ok);
                    const int L = bad ? __ffs(bad) - 1 : 32;
                    if (L > 0) {
                        const unsigned lim = L == 32 ? 0xffffffffu : ((1u << L) - 1u);
                        const unsigned eqm = __ballot_sync(FULL, eq) & lim;
                        int kx = 0;
                        while (kx < L) {
                            const unsigned bit = (eqm >> kx) & 1u;
                            const unsigned diff = ((bit ? ~eqm : eqm) & lim) >> kx;   // first position that differs
                            int run = diff ? __ffs(diff) - 1 : L - kx;
                            push_n(bit ? OP_EQ : OP_X, run);
                            kx += run;
                        }
                        // H after L diagonal steps = H of lane L's cell (lane L-1's value minus its step)
                        const int hlast = __shfl_sync(FULL, hv - sc, L - 1);
                        hval = hlast;
                        i -= L; j -= L;
                        if (forced > 0) forced -= L;
                        continue;
                    }
                    // lane 0's own cell is not a diagonal step
                    if (!__shfl_sync(FULL, (int)inblk, 0)) {
                        // Out of the replayed block in state H with the exact H known: try the ungapped-
                        // diagonal proof (see ctl_advance in sw_core.cuh) before asking for a replay.
                        bool proven = false;
                        int steps = 0;
                        if (k.shortcut) {
                            int rem = hval, pi = i, pj = j;
                            for (;;) {
                                const int qi = pi - l, qj = pj - l;
                                const bool v2 = qi >= 0 && qj >= 0;
                                int s2 = 0;
                                if (v2) s2 = acc.qcode(qi) == acc.tcode(qj) ? k.match : k.mismatch;
                                int p2 = s2;
#pragma unroll
                                for (int o = 1; o < 32; o <<= 1) {
                                    const int v = __shfl_up_sync(FULL, p2, o);
                                    if (l >= o) p2 += v;
                                }
                                const int rl = rem - p2;     // remainder after this lane's step
                                const unsigned hit = __ballot_sync(FULL, v2 && rl <= 0);
                                const unsigned inv = __ballot_sync(FULL, !v2);
                                const int fh = hit ? __ffs(hit) - 1 : 32, fi = inv ? __ffs(inv) - 1 : 32;
                                if (fh < fi) {
                                    proven = __shfl_sync(FULL, rl, fh) == 0;
                                    steps += fh + 1;
                                    break;
                                }
                                if (fi < 32) break;          // the diagonal leaves the matrix: nothing proven
                                rem = __shfl_sync(FULL, rl, 31);
                                steps += 32; pi -= 32; pj -= 32;
                            }
                        }
                        if (proven) { forced = steps; continue; }
                        const int g0 = i / R;
                        need = (j + g0) / FBLK;
                        break;
                    }
                    const uint32_t n0 = __shfl_sync(FULL, nib, 0);
                    if ((n0 >> 2) == 1u) { push_n(OP_I, 1); --i; mode = 1; gval = hval; }
                    else { push_n(OP_D, 1); --j; mode = 2; gval = hval; }
                } else {
                    const int g = i / R, r = i - g * R;
                    const int t = j + g;
                    if (t / FBLK != cur_blk || !tile_valid) { need = t / FBLK; break; }
                    const uint32_t nib = (tile[tile_index<R>(t % FBLK, g, r >> 2)] >> (sh + 4 * (r & 3))) & 0xfu;
                    if (mode == 1) {
                        if (!(nib & 2u)) { hval = gval + k.open; mode = 0; }
                        else { push_n(OP_I, 1); --i; gval += k.extend; }
                    } else {
                        if (!(nib & 1u)) { hval = gval + k.open; mode = 0; }
                        else { push_n(OP_D, 1); --j; gval += k.extend; }
                    }
                }
            }
            if (done && cur != 0) {
                if (l == 0) {
                    c.ring[nrev % OPS_CAP] = cur;
                    if (SPILL && a.ops_spill) a.ops_spill[(size_t)aln * a.ops_cap + nrev % a.ops_cap] = cur;
                }
                ++nrev; cur = 0;
            }
            if (l == 0) {
                c.i = i; c.j = j; c.mode = mode; c.hval = hval; c.gval = gval; c.cur = cur; c.nrev = nrev;
                if (done) { c.phase = 2; c.next_blk = -1; } else c.next_blk = need;
            }
        }
        __syncwarp();
        const bool fin = c.phase == 2;
        if (l == 0) {
            if (fin) {
                if constexpr (END_ONLY) finalize_end(c, sm.out, d.read);
                else finalize_result(c, sm.out, d.read, d.clip_left, d.clip_right, a.min_length);
            } else if (round + 1 < a.max_rounds) {
                const unsigned slot = atomicAdd(&a.qcount[rin ^ 1], 1u);
                a.queue[rin ^ 1][slot] = pack_req(aln, c.next_blk, ctl_scanmask(c));
            }   // else: out[aln] keeps its "no result" marker and fadegpu_wait reports the error
        }
        __syncwarp();
        if (fin) {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(&sm.out);
            uint32_t *dst = reinterpret_cast<uint32_t *>(&a.out[aln]);
            for (int w = l; w < OUTW; w += 32) dst[w] = src[w];
        } else {
            const uint32_t *src = reinterpret_cast<const uint32_t *>(&c);
            uint32_t *dst = reinterpret_cast<uint32_t *>(&a.state[aln]);
            for (int w = l; w < CTLW; w += 32) dst[w] = src[w];
        }
        __syncwarp();
    }
}

template <int R, bool SPILL, bool END_ONLY = false>
__global__ void FADE_SMALL_KERNEL trace_advance_kernel(const KernelArgs a)
{
    __shared__ AdvanceSmem adv[4];
    advance_round<R, SPILL, END_ONLY>(a, a.round, blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), gridDim.x * (blockDim.x >> 5), adv);
}

// The few alignments still unfinished after the full-grid rounds (very long paths): one block
// runs the remaining rounds back to back, separated by block barriers instead of launches.
template <int R, bool TAGGED>
__global__ void __launch_bounds__(128) trace_tail_kernel(const KernelArgs a)
{
    __shared__ uint16_t tws_all[16][40];
    __shared__ AdvanceSmem adv[4];
    for (int r = a.round; r < a.max_rounds; ++r) {
        if (a.qcount[r & 1] == 0u) break;          // uniform: every thread reads the same counter
        __syncthreads();
        if (threadIdx.x == 0) a.qcount[(r & 1) ^ 1] = 0u;
        __syncthreads();
        replay_round<R, TAGGED ? 0 : 1>(a, r, threadIdx.x >> 5, blockDim.x >> 5, tws_all);
        __threadfence_block();
        __syncthreads();
        advance_round<R, true>(a, r, threadIdx.x >> 5, blockDim.x >> 5, adv);   // (rarely reached: spill checked at run time)
        __threadfence_block();
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// generic exact kernel: one thread per alignment, int32, arbitrary letters and sizes
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int map_char(int c)
{
    switch (c) {
    case 'A': return 0;
    case 'C': return 1;
    case 'T': return 2;
    case 'G': return 3;
    case 'N': return 4;
    default: return 5;
    }
}

// upper-cased reference letter at global position p (source/analysis.d:63 .toUpper)
__device__ int ref_char(const RefDev &rf, int64_t p)
{
    const int c = ref_code(rf.planes, p);
    if (c < 4) return "ACTG"[c];
    if (c == C_N) return 'N';
    int64_t lo = 0, hi = rf.n_x - 1;
    while (lo <= hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int64_t v = rf.xpos[mid];
        if (v == p) return rf.xchr[mid];
        if (v < p) lo = mid + 1; else hi = mid - 1;
    }
    return '?';
}

__global__ void __launch_bounds__(128) sw_generic_kernel(const GenericArgs a)
{
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= a.n_slots) return;
    uint8_t *sc = a.scratch + (size_t)slot * a.slot_bytes;
    int32_t *Hc = reinterpret_cast<int32_t *>(sc);
    int32_t *Ec = Hc + a.qmax;
    uint8_t *qch = reinterpret_cast<uint8_t *>(Ec + a.qmax);
    uint8_t *trc = qch + ((a.qmax + 15) & ~15);
    const int o = a.open, e = a.extend;
    const char nt16[] = "=ACMGRSVTWYHKDBN";
    const uint8_t comp16[16] = { 0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15 };
    unsigned idx = 0, idx_end = 0;
    for (;;) {
        if (idx >= idx_end) {
            idx = atomicAdd(a.cursor, (unsigned)a.chunk);
            if (idx >= (unsigned)a.n_aln) break;
            idx_end = min(idx + (unsigned)a.chunk, (unsigned)a.n_aln);
        }
        const unsigned cur_idx = idx++;
        if (a.aln_flags && !(a.aln_flags[cur_idx] & 1u)) continue;
        const AlnDesc d = a.aln[cur_idx];
        const int qlen = d.qlen, tlen = d.tlen;
        AlnOut out;
        out.read = d.read;
        for (int kk = 0; kk < OPS_CAP; ++kk) out.ops[kk] = 0;
        if (qlen <= 0 || tlen <= 0 || qlen > a.qmax || tlen > a.tmax) {
            out.score = out.end_query = out.end_ref = out.beg_query = out.beg_ref = out.n_ops = 0;
            out.flags = R_ALIGNED | R_GENERIC;
            a.out[cur_idx] = out;
            continue;
        }
        const uint8_t *s4 = a.seq + d.seq_off;
        for (int i = 0; i < qlen; ++i) {   // source/util.d:23-34
            qch[i] = (uint8_t)nt16[comp16[nt16_at(s4, qlen - 1 - i)]];
            Hc[i] = 0;
            Ec[i] = -(1 << 28);
        }
        int best = 0, bi = 0, bj = 0;
        for (int j = 0; j < tlen; ++j) {
            const int tch = ref_char(a.ref, d.gstart + j);
            const int tcd = map_char(tch);
            int hdiag = 0, hup = 0, f = -(1 << 28);
            for (int i = 0; i < qlen; ++i) {
                const int hleft = Hc[i];
                const int e_opn = hleft - o, e_ext = Ec[i] - e;
                int tb = 0, ev, fv;
                if (e_opn > e_ext) { ev = e_opn; tb |= T_EOPEN; } else ev = e_ext;
                const int f_opn = hup - o, f_ext = f - e;
                if (f_opn > f_ext) { fv = f_opn; tb |= T_FOPEN; } else fv = f_ext;
                const int qcd = map_char(qch[i]);
                const int s = (qcd == 5 || tcd == 5) ? 0 : (qcd == tcd ? a.match : a.mismatch);
                int hd = hdiag + s;
                if (hd < 0) hd = 0;
                int h = hd;
                if (ev > h) h = ev;
                if (fv > h) h = fv;
                if (h == hd) tb |= (h == 0) ? T_ZERO : T_DIAG;
                else tb |= (h == fv) ? T_F : T_E;
                // here bits 2/3 describe how E[i][j] / F[i][j] THEMSELVES were derived
                trc[(size_t)i * tlen + j] = (uint8_t)tb;
                hdiag = hleft; hup = h; f = fv;
                Ec[i] = ev; Hc[i] = h;
                if (h > best) { best = h; bi = i; bj = j; }  // P3: first column, then first row
            }
        }
        out.score = best;
        if (best > 0 && a.tags_only && !score_may_accept(best, d.clip_left, d.clip_right, a.min_length)) {
            out.end_query = out.end_ref = out.beg_query = out.beg_ref = out.n_ops = 0;
            out.flags = R_ALIGNED | R_GENERIC | R_SCORE_ONLY;
            a.out[cur_idx] = out;
            continue;
        }
        if (best <= 0) {
            out.end_query = out.end_ref = out.beg_query = out.beg_ref = out.n_ops = 0;
            out.flags = R_ALIGNED | R_GENERIC;
            a.out[cur_idx] = out;
            continue;
        }
        // P4 traceback, reversed RLE ops into a ring (same convention as LaneCtl)
        uint32_t ring[OPS_CAP];
        int nrev = 0;
        uint32_t cur = 0;
        int i = bi, j = bj, state = 0;
        while (i >= 0 && j >= 0) {
            const int tb = trc[(size_t)i * tlen + j];
            uint32_t op;
            if (state == 0) {
                const int src = tb & 3;
                if (src == T_ZERO) break;
                if (src == T_DIAG) {
                    op = (qch[i] == (uint8_t)ref_char(a.ref, d.gstart + j)) ? OP_EQ : OP_X;
                    --i; --j;
                } else if (src == T_F) { state = 1; continue; }
                else { state = 2; continue; }
            } else if (state == 1) {
                op = OP_I; --i;
                if (tb & T_FOPEN) state = 0;
            } else {
                op = OP_D; --j;
                if (tb & T_EOPEN) state = 0;
            }
            if (cur != 0 && (cur & 0xf) == op) cur += 16;
            else {
                if (cur != 0) {
                    ring[nrev % OPS_CAP] = cur;
                    if (a.ops_spill) a.ops_spill[(size_t)cur_idx * a.ops_cap + nrev % a.ops_cap] = cur;
                    ++nrev;
                }
                cur = (1u << 4) | op;
            }
        }
        if (cur != 0) {
            ring[nrev % OPS_CAP] = cur;
            if (a.ops_spill) a.ops_spill[(size_t)cur_idx * a.ops_cap + nrev % a.ops_cap] = cur;
            ++nrev;
        }
        out.end_query = bi; out.end_ref = bj; out.beg_query = i + 1; out.beg_ref = j + 1;
        const int lead = i + 1, trail = qlen - 1 - bi;
        const int n = (lead > 0) + nrev + (trail > 0);
        out.n_ops = n;
        int wq = 0;
        if (lead > 0) out.ops[wq++] = ((uint32_t)lead << 4) | OP_S;
        for (int kk = nrev - 1; kk >= 0 && wq < OPS_CAP; --kk) {
            if (nrev - kk > OPS_CAP) break;
            out.ops[wq++] = ring[kk % OPS_CAP];
        }
        if (trail > 0 && wq < OPS_CAP && wq == n - 1) out.ops[wq++] = ((uint32_t)trail << 4) | OP_S;
        uint32_t flags = R_ALIGNED | R_GENERIC;
        if (n > OPS_CAP) flags |= R_OPS_TRUNC;
        const uint32_t first_op = lead > 0 ? (uint32_t)OP_S : (ring[(nrev - 1) % OPS_CAP] & 0xf);
        const uint32_t last_op = trail > 0 ? (uint32_t)OP_S : (ring[0] & 0xf);
        if (accept_side(true, best, n, first_op, last_op, lead, trail, d.clip_left, a.min_length)) flags |= R_ART_LEFT;
        if (accept_side(false, best, n, first_op, last_op, lead, trail, d.clip_right, a.min_length)) flags |= R_ART_RIGHT;
        out.flags = flags;
        a.out[cur_idx] = out;
    }
}

// ------------------------------------------------------------------------------------------------
// binning on the device (submits from the pinned view): the per-read part of align_clip that the
// host path evaluates while building descriptors -- length floor (analysis.d:34), window
// arithmetic (analysis.d:45-59) -- plus the length binning, without touching host cores
// ------------------------------------------------------------------------------------------------
__global__ void FADE_SMALL_KERNEL bin_classify_kernel(const BinArgs a)
{
    const uint32_t floor_u = (uint32_t)a.min_length;   // uint <= int compare of analysis.d:34
    unsigned long long cells = 0, bad = 0;
    int qmax = 0, tmax = 0, qmax_g = 0, tmax_g = 0, cnt = 0, fetched = 0;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n; r += (int64_t)gridDim.x * blockDim.x) {
        int key = -1;
        uint32_t cl, cr;
        bool need;
        if (a.gate) {
            // compact inputs: gate = min(255, max clip).  Below 255 it decides the floor exactly; at 255 (or with a
            // floor of 255 and more) the record itself does.
            const uint32_t g = a.gate[r];
            need = floor_u < 255u ? g > floor_u : g == 255u;
            cl = cr = 0;
            if (need) {
                const uint4 m0 = a.host_meta[2 * r], m1 = a.host_meta[2 * r + 1];   // one 32-byte PCIe read
                ++fetched;
                a.pos[r] = (int64_t)(((unsigned long long)m0.y << 32) | m0.x);
                a.seq_off[r] = (int64_t)m0.z;
                a.l_qseq[r] = (int32_t)m0.w;
                a.tid[r] = (int32_t)m1.x;
                a.aligned_len[r] = (int32_t)m1.y;
                a.clip_left[r] = (int32_t)(cl = m1.z);
                a.clip_right[r] = (int32_t)(cr = m1.w);
                need = (cl != 0 && !(cl <= floor_u)) || (cr != 0 && !(cr <= floor_u));
            } else {
                a.clip_left[r] = 0; a.clip_right[r] = 0;   // so that a replay from the device mirrors skips the read as well
            }
        } else {
            cl = (uint32_t)a.clip_left[r]; cr = (uint32_t)a.clip_right[r];
            need = (cl != 0 && !(cl <= floor_u)) || (cr != 0 && !(cr <= floor_u));
        }
        if (need) {
            const int tid = a.tid[r], ql = a.l_qseq[r];
            if (tid >= 0 && tid < a.n_contigs && ql > 0) {
                const int64_t so = a.seq_off[r];
                if (so < 0 || so + (ql + 1) / 2 > a.seq_total) bad |= 1ull;
                else {
                    int64_t start = a.pos[r] - a.window;
                    if (start < 0) start = 0;
                    int64_t end = a.pos[r] + (int64_t)a.aligned_len[r] + a.window;
                    if (end > a.clen[tid]) end = a.clen[tid];
                    if (end > start) {
                        if (end - start > 0x7fffffff || (end - start) * (int64_t)ql > ((int64_t)1 << 31)) {
                            // a window of more than 2^31 DP cells (a spliced record spanning megabases): the read is left
                            // unaligned and reported, the batch goes on
                            const unsigned long long slot = atomicAdd(&a.stats[11], 1ull);
                            if (slot < (unsigned long long)OVER_CAP) a.over_list[slot] = a.read ? a.read[r] : (int32_t)r;
                        } else {
                            const int tl = (int)(end - start);
                            const int rk = bin_rank(ql, tl, (a.flags & 1u) != 0);
                            key = bin_key(rk, tl);
                            a.tlen[r] = tl;
                            a.start[r] = start;
                            atomicAdd(&a.hist[key], 1);
                            cells += (unsigned long long)ql * (unsigned long long)tl;
                            ++cnt;
                            qmax = max(qmax, ql); tmax = max(tmax, tl);
                            if (rk == N_ROW_CLASSES) { qmax_g = max(qmax_g, ql); tmax_g = max(tmax_g, tl); }
                        }
                    }
                }
            }
        }
        a.key[r] = key;
    }
    // one set of atomics per warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        cells += __shfl_xor_sync(FULL, cells, o);
        bad |= __shfl_xor_sync(FULL, bad, o);
        cnt += __shfl_xor_sync(FULL, cnt, o);
        fetched += __shfl_xor_sync(FULL, fetched, o);
        qmax = max(qmax, __shfl_xor_sync(FULL, qmax, o)); tmax = max(tmax, __shfl_xor_sync(FULL, tmax, o));
        qmax_g = max(qmax_g, __shfl_xor_sync(FULL, qmax_g, o)); tmax_g = max(tmax_g, __shfl_xor_sync(FULL, tmax_g, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (cells) atomicAdd(&a.stats[0], cells);
        if (cnt) atomicAdd(&a.stats[1], (unsigned long long)cnt);
        if (qmax) atomicMax(&a.stats[2], (unsigned long long)qmax);
        if (tmax) atomicMax(&a.stats[3], (unsigned long long)tmax);
        if (qmax_g) atomicMax(&a.stats[4], (unsigned long long)qmax_g);
        if (tmax_g) atomicMax(&a.stats[5], (unsigned long long)tmax_g);
        if (bad) atomicOr(&a.stats[6], bad);
        if (fetched) atomicAdd(&a.stats[10], (unsigned long long)fetched);
    }
}

__global__ void FADE_SMALL_KERNEL bin_scatter_kernel(const BinArgs a)
{
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < a.n; r += (int64_t)gridDim.x * blockDim.x) {
        const int key = a.key[r];
        if (key < 0) continue;
        const int slot = a.keybase[key] + atomicAdd(&a.cursor[key], 1);
        AlnDesc d;
        d.gstart = a.coff[a.tid[r]] + a.start[r];
        d.seq_off = a.seq_off[r];
        if (a.seq_cursor) {
            // a 16-byte aligned slot that keeps the source's alignment phase, so that seq_pull_kernel copies whole uint4s
            const int64_t so = d.seq_off;
            const int ph = (int)(so & 15);
            const unsigned long long bytes = (unsigned long long)((ph + (a.l_qseq[r] + 1) / 2 + 15) & ~15);
            d.seq_off = (int64_t)atomicAdd(a.seq_cursor, bytes) + ph;
            a.src_off[slot] = so;
        }
        d.tlen = a.tlen[r];
        d.qlen = a.l_qseq[r];
        d.clip_left = (uint32_t)a.clip_left[r];
        d.clip_right = (uint32_t)a.clip_right[r];
        d.read = a.read ? a.read[r] : (int32_t)r;
        d.pad = 0;
        a.aln[slot] = d;
        a.aln_start[slot] = a.start[r];
    }
}

// The GPU fetches the bases of the reads it aligns straight from the caller's pinned (mapped) view:
// 8 lanes per alignment, one aligned uint4 each per pass, i.e. one 128-byte PCIe read per pass.
// Only ~20 % of a batch's bases are ever needed (SURVEY 6.2), so the other 80 % never cross PCIe
// and no host core touches any of them.
__global__ void FADE_SMALL_KERNEL seq_pull_kernel(const uint8_t *__restrict__ host_seq4, const AlnDesc *__restrict__ aln,
                                                       const int64_t *__restrict__ src_off, int n_aln, uint8_t *__restrict__ dst)
{
    const int lane = threadIdx.x & 7;
    for (int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 3; k < n_aln; k += (gridDim.x * blockDim.x) >> 3) {
        const int64_t so = src_off[k];
        const int ph = (int)(so & 15);
        const int chunks = (ph + (aln[k].qlen + 1) / 2 + 15) >> 4;
        const uint4 *s = reinterpret_cast<const uint4 *>(host_seq4 + (so - ph));
        uint4 *d = reinterpret_cast<uint4 *>(dst + (aln[k].seq_off - ph));
        for (int i = lane; i < chunks; i += 8) d[i] = s[i];
    }
}

// per-read flags and index into the compact results: the random stores of the scatter cost a host core milliseconds
// per batch (the records arrive in window-length order) and the device microseconds, so they are made here and 5
// bytes per read are copied home
__global__ void FADE_SMALL_KERNEL result_index_kernel(const AlnOut *out, int n_aln, int64_t n_reads, uint8_t *flags, int32_t *ridx,
                                                      unsigned long long *n_ok)
{
    int ok = 0;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n_aln; k += gridDim.x * blockDim.x) {
        const int r = out[k].read;
        const uint32_t f = out[k].flags;
        if (r >= 0 && (int64_t)r < n_reads && (f & 1u) && !(f & 0x80000000u)) { flags[r] = (uint8_t)(f & 0xffu); ridx[r] = k; ++ok; }
    }
    // records written by the SW kernels, counted so that the host need not walk them to validate
    ok = __reduce_add_sync(FULL, ok);
    if ((threadIdx.x & 31) == 0 && ok) atomicAdd(n_ok, (unsigned long long)ok);
}

// ------------------------------------------------------------------------------------------------
// pairs of caller-supplied sequences (fadegpu_align_pairs): pack the raw ASCII into the formats the
// binning and the SW kernels read, then put the records back into pair order
// ------------------------------------------------------------------------------------------------
// ASCII -> BAM nt16 code of "=ACMGRSVTWYHKDBN" (either case), 16 = not in the alphabet
__device__ __forceinline__ int nt16_of_ascii(int ch)
{
    if (ch >= 'a' && ch <= 'z') ch -= 32;
    switch (ch) {
    case '=': return 0; case 'A': return 1; case 'C': return 2; case 'M': return 3;
    case 'G': return 4; case 'R': return 5; case 'S': return 6; case 'V': return 7;
    case 'T': return 8; case 'W': return 9; case 'Y': return 10; case 'H': return 11;
    case 'K': return 12; case 'D': return 13; case 'B': return 14; case 'N': return 15;
    default: return 16;
    }
}

// The lanes of a warp write the qlen ASCII letters q as nt16 nibbles, two bases per byte, at dst: in REVERSE
// COMPLEMENT when rc.  True when the lane met a letter outside nt16.
__device__ __forceinline__ bool pack_query_nt16(const char *q, int64_t qlen, bool rc, uint8_t *dst, int l)
{
    const uint8_t comp16[16] = { 0, 8, 4, 12, 2, 10, 6, 14, 1, 9, 5, 13, 3, 11, 7, 15 };
    bool bad = false;
    for (int64_t b = l; b < (qlen + 1) / 2; b += 32) {
        uint32_t byte = 0;
        for (int h = 0; h < 2; ++h) {
            const int64_t i = 2 * b + h;   // base i of the reverse complement = complement of base qlen-1-i
            if (i >= qlen) break;
            const int c = nt16_of_ascii((unsigned char)q[rc ? qlen - 1 - i : i]);
            bad |= c > 15;
            byte |= (uint32_t)(rc ? comp16[c & 15] : c & 15) << (h ? 0 : 4);
        }
        dst[b] = (uint8_t)byte;
    }
    return bad;
}

// One warp per pair: lane 0 writes the pair's binning inputs, the lanes write the query as nt16 nibbles in REVERSE
// COMPLEMENT, two bases per byte.  The kernels reverse-complement a read as they load it (source/util.d:18-34), which
// restores the forward query; nt16 complement is an involution, so IUPAC letters come back unchanged.
__global__ void FADE_SMALL_KERNEL pair_prep_kernel(const PairArgs a)
{
    const int l = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < a.n; k += nwarps) {
        const int64_t q0 = a.qoff[k], qlen = a.qoff[k + 1] - q0;
        const int64_t t0 = a.toff[k], tlen = a.toff[k + 1] - t0;
        const bool over = tlen > 0x7fffffff || qlen * tlen > PAIR_MAX_CELLS;   // left unaligned, reported
        if (l == 0) {
            a.seq_off[k] = q0;
            a.pos[k] = 0;
            a.l_qseq[k] = (int32_t)qlen;
            a.tid[k] = (int32_t)k;
            a.aligned_len[k] = over ? 0 : (int32_t)tlen;
            a.clip_left[k] = over ? 0 : (int32_t)qlen;   // the length floor (0) passes every non-empty query
            a.clip_right[k] = 0;
            a.clen[k] = tlen;
            a.coff[k] = 32 * (k + (t0 >> 5));
        }
        const bool bad = pack_query_nt16(a.query + q0, qlen, true, a.seq4 + q0, l);
        if (__any_sync(0xffffffffu, bad) && l == 0) atomicMin(a.bad, (int32_t)k);
    }
}

// One warp per region, as pair_prep_kernel: the window of region k is [start, end) of contig tid (window 0 in the
// binning).  Strand 0 stores the query reverse-complemented and strand 1 as given, so that the kernels' reverse
// complement aligns the query itself or its reverse complement.
__global__ void FADE_SMALL_KERNEL region_prep_kernel(const RegionArgs a)
{
    const int l = threadIdx.x & 31;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t k = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < a.n; k += nwarps) {
        const int64_t q0 = a.qoff[k], qlen = a.qoff[k + 1] - q0;
        const int64_t tlen = a.end[k] - a.start[k];
        const bool over = tlen > 0x7fffffff || qlen * tlen > PAIR_MAX_CELLS;   // left unaligned, reported
        if (l == 0) {
            a.seq_off[k] = q0;
            a.pos[k] = a.start[k];
            a.l_qseq[k] = (int32_t)qlen;
            a.tid[k] = a.rtid[k];
            a.aligned_len[k] = over ? 0 : (int32_t)tlen;
            a.clip_left[k] = over ? 0 : (int32_t)qlen;   // the length floor (0) passes every non-empty query
            a.clip_right[k] = 0;
        }
        const bool bad = pack_query_nt16(a.query + q0, qlen, a.strand[k] == 0, a.seq4 + q0, l);
        if (__any_sync(0xffffffffu, bad) && l == 0) atomicMin(a.bad, (int32_t)k);
    }
}

// the pair whose target holds global base p (targets start on 32-base boundaries, coff strictly increasing)
__device__ __forceinline__ int64_t pair_of_base(const PairArgs &a, int64_t p)
{
    int64_t lo = 0, hi = a.n - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (a.coff[mid] <= p) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// One block per chunk of PAIR_CHUNK_WORDS 32-base words (4 consecutive words per thread): the 2-bit, N and wildcard
// planes of the targets, as fadegpu_load_reference packs contigs, and the chunk's number of wildcard letters.
constexpr int PAIR_WORDS_PER_THREAD = PAIR_CHUNK_WORDS / 256;
__global__ void __launch_bounds__(256) pair_pack_targets_kernel(const PairArgs a)
{
    __shared__ int warp_x[8];
    int nx = 0;
    for (int u = 0; u < PAIR_WORDS_PER_THREAD; ++u) {
        const int64_t w = (int64_t)blockIdx.x * PAIR_CHUNK_WORDS + threadIdx.x * PAIR_WORDS_PER_THREAD + u;
        if (w >= a.n_words) break;
        uint32_t a0 = 0, a1 = 0, nm = 0, xm = 0;
        if (a.n > 0) {
            const int64_t p0 = 32 * w, k = pair_of_base(a, p0);
            const int64_t local = p0 - a.coff[k], tlen = a.clen[k];
            if (local >= 0 && local < tlen) {
                const char *t = a.target + a.toff[k] + local;
                const int lim = (int)min((int64_t)32, tlen - local);
                for (int b = 0; b < lim; ++b) {
                    int ch = (unsigned char)t[b];
                    if (ch >= 'a' && ch <= 'z') ch -= 32;
                    const uint32_t code = ch == 'A' ? 0u : ch == 'C' ? 1u : ch == 'T' ? 2u : ch == 'G' ? 3u : 0u;
                    if (b < 16) a0 |= code << (2 * b); else a1 |= code << (2 * (b - 16));
                    if (ch == 'N') nm |= 1u << b;
                    else if (ch != 'A' && ch != 'C' && ch != 'G' && ch != 'T') xm |= 1u << b;
                }
            }
        }
        a.two[2 * w] = a0; a.two[2 * w + 1] = a1; a.nmask[w] = nm; a.xmask[w] = xm;
        nx += __popc(xm);
    }
    nx = __reduce_add_sync(FULL, nx);
    if ((threadIdx.x & 31) == 0) warp_x[threadIdx.x >> 5] = nx;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int i = 0; i < 8; ++i) t += warp_x[i];
        a.chunk_x[blockIdx.x] = (uint32_t)t;
        if (t) atomicAdd(a.n_x, (unsigned long long)t);
    }
}

// exclusive prefix of v over a block of 256 threads; *total receives the sum
__device__ __forceinline__ uint32_t block_exclusive_256(uint32_t v, uint32_t *total)
{
    __shared__ uint32_t warp_sum[8];
    const int l = threadIdx.x & 31, wi = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(FULL, inc, o);
        if (l >= o) inc += y;
    }
    if (l == 31) warp_sum[wi] = inc;
    __syncthreads();
    uint32_t before = 0, all = 0;
    for (int i = 0; i < 8; ++i) { if (i < wi) before += warp_sum[i]; all += warp_sum[i]; }
    __syncthreads();
    *total = all;
    return before + inc - v;
}

// Order-preserving compaction of the wildcard letters into the sorted (position, upper-cased letter) list that the
// generic kernel searches (RefDev::xpos / xchr).  Chunk b starts at the sum of chunk_x over the chunks before it.
__global__ void __launch_bounds__(256) pair_xlist_kernel(const PairArgs a)
{
    __shared__ uint32_t chunk_base;
    if (a.chunk_x[blockIdx.x] == 0) return;   // (uniform over the block)
    if (threadIdx.x == 0) chunk_base = 0;
    __syncthreads();
    {   // chunk_x is small (one word per 32768 target bases): the block adds up its predecessors
        uint32_t part = 0;
        for (int64_t c = threadIdx.x; c < blockIdx.x; c += blockDim.x) part += a.chunk_x[c];
        part = __reduce_add_sync(FULL, part);
        if ((threadIdx.x & 31) == 0 && part) atomicAdd(&chunk_base, part);
    }
    __syncthreads();
    const int64_t w0 = (int64_t)blockIdx.x * PAIR_CHUNK_WORDS + threadIdx.x * PAIR_WORDS_PER_THREAD;
    uint32_t xm[PAIR_WORDS_PER_THREAD], cnt = 0;
    for (int u = 0; u < PAIR_WORDS_PER_THREAD; ++u) {
        xm[u] = w0 + u < a.n_words ? a.xmask[w0 + u] : 0u;
        cnt += __popc(xm[u]);
    }
    uint32_t total;
    int64_t slot = (int64_t)chunk_base + block_exclusive_256(cnt, &total);
    for (int u = 0; u < PAIR_WORDS_PER_THREAD; ++u) {
        if (!xm[u]) continue;
        const int64_t p0 = 32 * (w0 + u), k = pair_of_base(a, p0);
        const char *t = a.target + a.toff[k] + (p0 - a.coff[k]);
        for (uint32_t m = xm[u]; m; m &= m - 1) {
            const int b = __ffs(m) - 1;
            int ch = (unsigned char)t[b];
            if (ch >= 'a' && ch <= 'z') ch -= 32;
            a.xpos[slot] = p0 + b;
            a.xchr[slot] = (uint8_t)ch;
            ++slot;
        }
    }
}

__global__ void FADE_SMALL_KERNEL pair_results_init_kernel(int64_t n, const int64_t *qoff, const int64_t *t_beg,
                                                           const int64_t *t_end, PairResult *res)
{
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t qlen = qoff[k + 1] - qoff[k], tlen = t_end[k] - t_beg[k];
        PairResult r;
        r.score = r.end_query = r.end_ref = r.beg_query = r.beg_ref = r.n_ops = 0;
        r.reserved = 0;
        r.flags = (qlen > 0 && tlen > 0 && (tlen > 0x7fffffff || qlen * tlen > PAIR_MAX_CELLS)) ? PAIR_R_OVERSIZE : 0u;
        res[k] = r;
    }
}

// one thread per alignment: its record goes to the pair's slot, its forward CIGAR (P5) is assembled from the spill ring
__global__ void FADE_SMALL_KERNEL pair_results_kernel(const AlnDesc *aln, const AlnOut *out, int n_aln, int64_t n,
                                                      const uint32_t *spill, int max_ops, PairResult *res, uint32_t *ops,
                                                      unsigned long long *n_ok)
{
    int ok = 0;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n_aln; idx += gridDim.x * blockDim.x) {
        const AlnOut o = out[idx];
        const int64_t k = o.read;
        if (k < 0 || k >= n || !(o.flags & R_ALIGNED) || (o.flags & 0x80000000u)) continue;
        ++ok;
        PairResult r;
        r.score = o.score; r.end_query = o.end_query; r.end_ref = o.end_ref; r.beg_query = o.beg_query; r.beg_ref = o.beg_ref;
        r.n_ops = o.n_ops;
        r.flags = (o.flags & (R_ALIGNED | R_GENERIC)) | (o.n_ops > max_ops ? R_OPS_TRUNC : 0u);
        r.reserved = 0;
        res[k] = r;
        if (max_ops > 0) {
            uint32_t *dst = ops + (size_t)k * max_ops;
            if (o.n_ops == 0) {
                for (int w = 0; w < max_ops; ++w) dst[w] = 0;
            } else {
                const int lead = o.beg_query, trail = aln[idx].qlen - 1 - o.end_query;
                const int nrev = o.n_ops - (lead > 0) - (trail > 0);
                forward_ops(spill + (size_t)idx * max_ops, max_ops, nrev, lead, trail, dst);
            }
        }
    }
    ok = __reduce_add_sync(FULL, ok);
    if ((threadIdx.x & 31) == 0 && ok) atomicAdd(n_ok, (unsigned long long)ok);
}

// score-only calls: the same, without the begin cell and the CIGAR (the generic kernel's are dropped here)
__global__ void FADE_SMALL_KERNEL pair_score_results_kernel(const AlnOut *out, int n_aln, int64_t n, PairResult *res,
                                                            unsigned long long *n_ok)
{
    int ok = 0;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < n_aln; idx += gridDim.x * blockDim.x) {
        const AlnOut o = out[idx];
        const int64_t k = o.read;
        if (k < 0 || k >= n || !(o.flags & R_ALIGNED) || (o.flags & 0x80000000u)) continue;
        ++ok;
        PairResult r;
        r.score = o.score; r.end_query = o.end_query; r.end_ref = o.end_ref;
        r.beg_query = r.beg_ref = r.n_ops = 0;
        r.flags = o.flags & (R_ALIGNED | R_GENERIC);
        r.reserved = 0;
        res[k] = r;
    }
    ok = __reduce_add_sync(FULL, ok);
    if ((threadIdx.x & 31) == 0 && ok) atomicAdd(n_ok, (unsigned long long)ok);
}

// ------------------------------------------------------------------------------------------------
// INT16x2 ALU issue-rate microbenchmark: 8 independent VIADDMNMX.S16x2 chains per thread
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) alu_peak_kernel(uint32_t *out, int iters)
{
    uint32_t x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    const uint32_t c = 0x00010003u + blockIdx.x, d = 0xfffefffdu;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            x0 = __viaddmax_s16x2(x0, c, d); x1 = __viaddmax_s16x2(x1, c, d);
            x2 = __viaddmax_s16x2(x2, c, d); x3 = __viaddmax_s16x2(x3, c, d);
            x4 = __viaddmax_s16x2(x4, c, d); x5 = __viaddmax_s16x2(x5, c, d);
            x6 = __viaddmax_s16x2(x6, c, d); x7 = __viaddmax_s16x2(x7, c, d);
        }
    }
    const uint32_t r = x0 ^ x1 ^ x2 ^ x3 ^ x4 ^ x5 ^ x6 ^ x7;
    if (r == 0x12345678u) out[0] = r;  // keep the chains alive
}

}  // namespace

int tw_stride_for(int nblk_max) { return (FBLK * std::min(nblk_max, FILL_CHUNK_BLOCKS) + FG + 1 + 7) & ~7; }

size_t fill_smem_bytes(int tw_stride) { return (size_t)(FILL_THREADS / FG) * tw_stride * 2; }

template <int R, int STEP>
static cudaError_t launch_fill_tf(const KernelArgs &a, cudaStream_t s)
{
    const size_t smem = fill_smem_bytes(a.tw_stride);
    cudaError_t e = cudaFuncSetAttribute(sw_fill_kernel<R, STEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int wpb = FILL_THREADS / 32;
    const int grid = (a.n_items + wpb - 1) / wpb;
    sw_fill_kernel<R, STEP><<<grid, FILL_THREADS, smem, s>>>(a);
    return cudaGetLastError();
}

template <int R>
static cudaError_t launch_fill_t(const KernelArgs &a, cudaStream_t s)
{
    switch (score_step_for(a.k)) {
    case 2: return launch_fill_tf<R, 2>(a, s);
    case 1: return launch_fill_tf<R, 1>(a, s);
    default: return launch_fill_tf<R, 0>(a, s);
    }
}

template <int R, bool TAGGED>
static cudaError_t launch_trace_tt(KernelArgs a, cudaStream_t s, int sm_count, int *launches)
{
    // init: one thread per alignment
    const int n = a.n_aln;
    int grid = std::min((n + 127) / 128, sm_count * 8);
    trace_init_kernel<R><<<grid, 128, 0, s>>>(a);
    int nl = 1;
    constexpr int FULL_ROUNDS = 10;  // covers paths up to ~9 blocks (any 2x250 read); the rest goes to the tail kernel
    const int quads = (n + 7) / 8;
    int r = 0;
    for (; r < a.max_rounds && r < FULL_ROUNDS; ++r) {
        a.round = r;
        // the queue shrinks quickly: smaller grid-stride grids for the later rounds
        const int g1 = std::min((quads + 3) / 4, r < 3 ? sm_count * 4 : sm_count);
        const int g2 = std::min((n + 3) / 4, r < 3 ? sm_count * 16 : sm_count * 2);   // a warp per request
        if (getenv("FADEGPU_DEBUG_ROUNDS")) {   // development aid: requests per round (synchronising!)
            unsigned int qc[2] = { 0, 0 };
            cudaStreamSynchronize(s);
            cudaMemcpy(qc, a.qcount, sizeof(qc), cudaMemcpyDeviceToHost);
            fprintf(stderr, "[fadegpu] round %d: %u requests (n_aln %d)\n", r, qc[r & 1], n);
        }
        if (r == 0 && a.k.shortcut) {
            const int step = score_step_for(a.k);
            if (step == 2) trace_replay_kernel<R, 2, 2><<<std::max(g1, 1), 128, 0, s>>>(a);
            else if (step == 1) trace_replay_kernel<R, 2, 1><<<std::max(g1, 1), 128, 0, s>>>(a);
            else trace_replay_kernel<R, 2, 0><<<std::max(g1, 1), 128, 0, s>>>(a);
        }
        else trace_replay_kernel<R, TAGGED ? 0 : 1><<<std::max(g1, 1), 128, 0, s>>>(a);
        if (a.ops_spill) trace_advance_kernel<R, true><<<std::max(g2, 1), 128, 0, s>>>(a);
        else trace_advance_kernel<R, false><<<std::max(g2, 1), 128, 0, s>>>(a);
        nl += 2;
    }
    if (r < a.max_rounds) {
        a.round = r;
        trace_tail_kernel<R, TAGGED><<<1, 128, 0, s>>>(a);
        nl += 1;
    }
    if (launches) *launches += nl;
    return cudaGetLastError();
}

// Score-only calls: trace_init_kernel as above, then rounds of scan-only replays (MODE 2, no trace tile) and advances
// that stop at the end cell.  Each round scans one candidate block of every unfinished alignment and marks every
// candidate thread whose maximum was first reached in it; an alignment has at most FG candidate threads, so FG rounds
// finish all of them and no tail kernel is needed.
template <int R, int STEP>
static cudaError_t launch_end_scan_ts(KernelArgs a, cudaStream_t s, int sm_count, int *launches)
{
    const int n = a.n_aln;
    trace_init_kernel<R><<<std::min((n + 127) / 128, sm_count * 8), 128, 0, s>>>(a);
    const int quads = (n + 7) / 8;
    a.max_rounds = FG;   // an alignment left after them keeps its "no result" marker, and the call reports it
    for (int r = 0; r < a.max_rounds; ++r) {
        a.round = r;
        const int g1 = std::min((quads + 3) / 4, r < 3 ? sm_count * 4 : sm_count);
        const int g2 = std::min((n + 3) / 4, r < 3 ? sm_count * 16 : sm_count * 2);
        trace_replay_kernel<R, 2, STEP><<<std::max(g1, 1), 128, 0, s>>>(a);
        trace_advance_kernel<R, false, true><<<std::max(g2, 1), 128, 0, s>>>(a);
    }
    if (launches) *launches += 1 + 2 * a.max_rounds;
    return cudaGetLastError();
}

template <int R>
static cudaError_t launch_trace_t(const KernelArgs &a, bool end_only, cudaStream_t s, int sm_count, int *launches)
{
    if (end_only) {
        switch (score_step_for(a.k)) {
        case 2: return launch_end_scan_ts<R, 2>(a, s, sm_count, launches);
        case 1: return launch_end_scan_ts<R, 1>(a, s, sm_count, launches);
        default: return launch_end_scan_ts<R, 0>(a, s, sm_count, launches);
        }
    }
    return a.k.tagged_ok ? launch_trace_tt<R, true>(a, s, sm_count, launches)
                         : launch_trace_tt<R, false>(a, s, sm_count, launches);
}

cudaError_t launch_fill(int R, const KernelArgs &a, cudaStream_t s)
{
    if (a.n_items <= 0) return cudaSuccess;
    switch (R) {
    case 13: return launch_fill_t<13>(a, s);
    case 19: return launch_fill_t<19>(a, s);
    case 25: return launch_fill_t<25>(a, s);
    case 32: return launch_fill_t<32>(a, s);
    case 38: return launch_fill_t<38>(a, s);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_trace(int R, const KernelArgs &a, bool end_only, cudaStream_t s, int sm_count, int *launches)
{
    if (a.n_items <= 0) return cudaSuccess;
    switch (R) {
    case 13: return launch_trace_t<13>(a, end_only, s, sm_count, launches);
    case 19: return launch_trace_t<19>(a, end_only, s, sm_count, launches);
    case 25: return launch_trace_t<25>(a, end_only, s, sm_count, launches);
    case 32: return launch_trace_t<32>(a, end_only, s, sm_count, launches);
    case 38: return launch_trace_t<38>(a, end_only, s, sm_count, launches);
    default: return cudaErrorInvalidValue;
    }
}

size_t trace_tile_bytes(int R)
{
    switch (R) {
    case 13: return (size_t)tile_words<13>() * 4;
    case 19: return (size_t)tile_words<19>() * 4;
    case 25: return (size_t)tile_words<25>() * 4;
    case 32: return (size_t)tile_words<32>() * 4;
    default: return (size_t)tile_words<38>() * 4;
    }
}

cudaError_t launch_bin_classify(const BinArgs &a, int sm_count, cudaStream_t s)
{
    if (a.n <= 0) return cudaSuccess;
    const int grid = (int)std::min<int64_t>((a.n + 127) / 128, (int64_t)sm_count * 16);
    bin_classify_kernel<<<grid, 128, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_bin_scatter(const BinArgs &a, int sm_count, cudaStream_t s)
{
    if (a.n <= 0) return cudaSuccess;
    const int grid = (int)std::min<int64_t>((a.n + 127) / 128, (int64_t)sm_count * 16);
    bin_scatter_kernel<<<grid, 128, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_seq_pull(const uint8_t *host_seq4, const AlnDesc *aln, const int64_t *src_off, int n_aln, uint8_t *dst, int sm_count,
                            cudaStream_t s)
{
    if (n_aln <= 0) return cudaSuccess;
    const int grid = std::min((n_aln * 8 + 127) / 128, sm_count * 16);
    seq_pull_kernel<<<grid, 128, 0, s>>>(host_seq4, aln, src_off, n_aln, dst);
    return cudaGetLastError();
}

cudaError_t launch_result_index(const AlnOut *out, int n_aln, int64_t n_reads, uint8_t *flags, int32_t *ridx, unsigned long long *n_ok,
                                int sm_count, cudaStream_t s)
{
    if (n_aln <= 0) return cudaSuccess;
    result_index_kernel<<<std::min((n_aln + 127) / 128, sm_count * 16), 128, 0, s>>>(out, n_aln, n_reads, flags, ridx, n_ok);
    return cudaGetLastError();
}

cudaError_t launch_generic(const GenericArgs &a, int n_slots, cudaStream_t s)
{
    if (a.n_aln <= 0 || n_slots <= 0) return cudaSuccess;
    const int threads = 128;
    const int grid = (n_slots + threads - 1) / threads;
    if (a.n_slots != n_slots || a.chunk <= 0) return cudaErrorInvalidValue;
    sw_generic_kernel<<<grid, threads, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pair_prep(const PairArgs &a, int sm_count, cudaStream_t s)
{
    if (a.n <= 0) return cudaSuccess;
    const int grid = (int)std::min<int64_t>((a.n * 32 + 127) / 128, (int64_t)sm_count * 16);
    pair_prep_kernel<<<grid, 128, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pair_pack_targets(const PairArgs &a, cudaStream_t s)
{
    if (a.n_words <= 0) return cudaSuccess;
    pair_pack_targets_kernel<<<(unsigned)((a.n_words + PAIR_CHUNK_WORDS - 1) / PAIR_CHUNK_WORDS), 256, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pair_xlist(const PairArgs &a, cudaStream_t s)
{
    if (a.n_words <= 0) return cudaSuccess;
    pair_xlist_kernel<<<(unsigned)((a.n_words + PAIR_CHUNK_WORDS - 1) / PAIR_CHUNK_WORDS), 256, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_region_prep(const RegionArgs &a, int sm_count, cudaStream_t s)
{
    if (a.n <= 0) return cudaSuccess;
    const int grid = (int)std::min<int64_t>((a.n * 32 + 127) / 128, (int64_t)sm_count * 16);
    region_prep_kernel<<<grid, 128, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pair_results(int64_t n, const int64_t *qoff, const int64_t *t_beg, const int64_t *t_end,
                                const AlnDesc *aln, const AlnOut *out, int n_aln, bool score_only, const uint32_t *spill,
                                int max_ops, PairResult *res, uint32_t *ops, unsigned long long *n_ok, int sm_count,
                                cudaStream_t s)
{
    if (n <= 0) return cudaSuccess;
    pair_results_init_kernel<<<(int)std::min<int64_t>((n + 127) / 128, (int64_t)sm_count * 16), 128, 0, s>>>(n, qoff, t_beg,
                                                                                                             t_end, res);
    if (n_aln > 0 && score_only)
        pair_score_results_kernel<<<std::min((n_aln + 127) / 128, sm_count * 16), 128, 0, s>>>(out, n_aln, n, res, n_ok);
    else if (n_aln > 0)
        pair_results_kernel<<<std::min((n_aln + 127) / 128, sm_count * 16), 128, 0, s>>>(aln, out, n_aln, n, spill, max_ops,
                                                                                       res, ops, n_ok);
    return cudaGetLastError();
}

cudaError_t launch_alu_peak(uint32_t *out, int iters, int blocks, int threads, cudaStream_t s)
{
    alu_peak_kernel<<<blocks, threads, 0, s>>>(out, iters);
    return cudaGetLastError();
}

}  // namespace fade
