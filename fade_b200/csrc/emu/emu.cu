// emu.cu -- HOST lock-step emulation of one 8-thread group of the realignment kernels.
//
// TEST INFRASTRUCTURE ONLY: built into libfadeemu.so and loaded only by tests/ (CPU, no GPU) to
// check the shared arithmetic core (sw_core.cuh: packed DP step, checkpoint/replay geometry,
// end-cell rule, traceback state machine, accept predicates) against the oracle.  The product
// library (libfadegpu.so) never links or loads this file; its orchestration of the same core is
// the CUDA code in kernels.cu.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "../sw_core.cuh"

using namespace fade;

namespace {

template <int R>
struct ThreadState {
    uint32_t H[R], E[R], qs[R], qf[R], qp[(R + 1) / 2];   // qf / qp: query words of fill_step_f16 / fill_step_f16x2
    uint32_t hu_prev, fout, M;
};

template <int R>
int align_pair(const uint8_t *qa, int qlen_a, const uint8_t *ta, int tlen_a,
               const uint8_t *qb, int qlen_b, const uint8_t *tb, int tlen_b,
               const SwConsts &k, int extra_blocks, int tagged, int32_t min_length,
               uint32_t clipl_a, uint32_t clipr_a, uint32_t clipl_b, uint32_t clipr_b,
               AlnOut *out_a, AlnOut *out_b, int ops_cap = 0, uint32_t *ops_a = nullptr, uint32_t *ops_b = nullptr,
               int32_t *scan_info = nullptr)
{
    const int rows = FG * R;
    if (qlen_a > rows || qlen_b > rows) return -1;
    const int tmax = tlen_a > tlen_b ? tlen_a : tlen_b;
    const int nblk = num_blocks(tmax) + extra_blocks;
    const int TW = FBLK * nblk + FG + 1;
    std::vector<uint16_t> tw(TW);
    for (int idx = 0; idx < TW; ++idx) {
        const int j = idx - FG;
        const int ca = (j >= 0 && j < tlen_a) ? ta[j] : C_TPAD;
        const int cb = (j >= 0 && j < tlen_b) ? tb[j] : C_TPAD;
        tw[idx] = (uint16_t)t_sel(ca, cb);
    }
    std::vector<uint8_t> qc(rows);
    std::vector<ThreadState<R>> st(FG);
    for (int g = 0; g < FG; ++g)
        for (int r = 0; r < R; ++r) {
            const int i = g * R + r;
            const int ca = i < qlen_a ? qa[i] : C_QPAD;
            const int cb = i < qlen_b ? qb[i] : C_QPAD;
            st[g].qs[r] = q_sel(ca, cb);
            set_query<1>(st[g].qf, r, ca, cb);
            set_query<2>(st[g].qp, r, ca, cb);
            qc[i] = (uint8_t)(ca | (cb << 4));
        }
    auto init_state = [&](ThreadState<R> &s) {
        for (int r = 0; r < R; ++r) { s.H[r] = 0; s.E[r] = k.neg_o; }
        s.hu_prev = 0; s.fout = k.neg_o; s.M = 0;
    };
    for (int g = 0; g < FG; ++g) init_state(st[g]);

    // ---- score-only pass with checkpoints (the step make_consts chose, as on the device) ----
    const int step = (tagged & 8) ? 0 : ((tagged & 16) && k.f16_ok ? 1 : score_step_for(k));
    const int CW = ck_words<R>();
    std::vector<uint32_t> ck((size_t)nblk * FG * CW);
    LaneCtl ctl[2];
    memset(ctl, 0, sizeof(ctl));
    uint32_t Mprev[FG];
    for (int g = 0; g < FG; ++g) Mprev[g] = 0;
    for (int c = 0; c < nblk; ++c) {
        for (int u = 0; u < FBLK; ++u) {
            const int t = c * FBLK + u;
            uint32_t hu[FG], fin[FG];
            for (int g = 0; g < FG; ++g) {
                hu[g] = g == 0 ? 0u : st[g - 1].H[R - 1];   // __shfl_up of the bottom-row H
                fin[g] = g == 0 ? k.neg_o : st[g - 1].fout; // __shfl_up of the running F
            }
            for (int g = 0; g < FG; ++g) {
                const uint32_t ts = tw[t - g + FG];
                const uint32_t hd = st[g].hu_prev;
                if (step == 2) score_step<R, 2>(st[g].H, st[g].E, st[g].qp, st[g].M, ts, hd, fin[g], st[g].fout, k);
                else if (step == 1) score_step<R, 1>(st[g].H, st[g].E, st[g].qf, st[g].M, ts, hd, fin[g], st[g].fout, k);
                else score_step<R, 0>(st[g].H, st[g].E, st[g].qs, st[g].M, ts, hd, fin[g], st[g].fout, k);
                st[g].hu_prev = hu[g];
            }
        }
        for (int g = 0; g < FG; ++g) {
            uint32_t *p = &ck[((size_t)c * FG + g) * CW];
            for (int r = 0; r < R; ++r) { p[r] = st[g].H[r]; p[R + r] = st[g].E[r]; }
            p[2 * R] = st[g].hu_prev;
            p[2 * R + 1] = st[g].fout;
            if (st[g].M != Mprev[g]) {
                if (lane_lo(st[g].M) != lane_lo(Mprev[g])) ctl[0].blk[g] = c;
                if (lane_hi(st[g].M) != lane_hi(Mprev[g])) ctl[1].blk[g] = c;
                Mprev[g] = st[g].M;
            }
        }
    }
    for (int g = 0; g < FG; ++g) { ctl[0].best[g] = lane_lo(st[g].M); ctl[1].best[g] = lane_hi(st[g].M); }

    // ---- traceback: replay blocks with trace recording ----
    ctl_init(ctl[0], qlen_a, tlen_a);
    ctl_init(ctl[1], qlen_b, tlen_b);
    constexpr int RW = trace_words<R>();
    std::vector<uint32_t> tr((size_t)tile_words<R>());
    // bit 5 of `tagged`: score-only calls -- every replay is a scan with the score-only step (no trace), the walkers stop
    // at the end cell; scan_info[2 L ..] receives lane L's number of scan replays and its first candidate block
    const bool end_only = (tagged & 32) != 0;
    const bool tg_trace = !end_only && (tagged & 1) && k.tagged_ok;
    int32_t scans[2] = { 0, 0 }, first_blk[2];
    for (int L = 0; L < 2; ++L) first_blk[L] = ctl[L].phase == 0 ? ctl[L].next_blk : -1;
    // ops_cap > 0: the walkers also spill every op into rings of ops_cap words, as the device does for
    // fadegpu_align_pairs, and ops_a / ops_b receive the first ops_cap forward ops assembled from them
    std::vector<uint32_t> spill[2];
    for (auto &v : spill) v.assign((size_t)(ops_cap > 0 ? ops_cap : 1), 0u);
    uint32_t *sp0 = ops_cap > 0 ? spill[0].data() : nullptr, *sp1 = ops_cap > 0 ? spill[1].data() : nullptr;
    int guard = 0;
    bool first_iter = true;
    while (ctl[0].phase != 2 || ctl[1].phase != 2) {
        if (++guard > 4 * nblk + 16) return -2;
        // bit 2 of `tagged`: the first replay is a scan with the score-only step in the plain / fp16 domain and records
        // no trace, like round 0 on the device (trace_replay_kernel<R, 2, STEP>)
        const bool scan_only = end_only || ((tagged & 4) && first_iter);
        const bool tg = tg_trace && !scan_only;
        int blk[2];
        for (int L = 0; L < 2; ++L) blk[L] = (ctl[L].phase != 2 && ctl[L].next_blk >= 0) ? ctl[L].next_blk : 0;
        bool scan[2][FG];
        for (int L = 0; L < 2; ++L)
            for (int g = 0; g < FG; ++g) scan[L][g] = (ctl_scanmask(ctl[L]) >> g) & 1u;
        // load per-lane state
        for (int g = 0; g < FG; ++g) {
            ThreadState<R> s0, s1;
            init_state(s0); init_state(s1);
            auto load = [&](ThreadState<R> &s, int b) {
                if (b == 0) return;
                const uint32_t *p = &ck[((size_t)(b - 1) * FG + g) * CW];
                for (int r = 0; r < R; ++r) { s.H[r] = p[r]; s.E[r] = p[R + r]; }
                s.hu_prev = p[2 * R]; s.fout = p[2 * R + 1];
            };
            load(s0, blk[0]); load(s1, blk[1]);
            auto mix = [&](uint32_t a, uint32_t b) {
                const uint32_t w = (a & 0xffffu) | (b & 0xffff0000u);
                return tg ? to_tagged(w) : w;
            };
            for (int r = 0; r < R; ++r) { st[g].H[r] = mix(s0.H[r], s1.H[r]); st[g].E[r] = mix(s0.E[r], s1.E[r]); }
            st[g].hu_prev = mix(s0.hu_prev, s1.hu_prev);
            st[g].fout = mix(s0.fout, s1.fout);
        }
        const uint32_t f_top = tg ? k.neg_o16 : k.neg_o;
        const int mul = tg ? 16 : 1;
        bool found[2][FG];
        for (int L = 0; L < 2; ++L) for (int g = 0; g < FG; ++g) found[L][g] = false;
        for (int u = 0; u < FBLK; ++u) {
            const int t0 = blk[0] * FBLK + u, t1 = blk[1] * FBLK + u;
            uint32_t hu[FG], fin[FG];
            for (int g = 0; g < FG; ++g) {
                hu[g] = g == 0 ? 0u : st[g - 1].H[R - 1];
                fin[g] = g == 0 ? f_top : st[g - 1].fout;
            }
            for (int g = 0; g < FG; ++g) {
                const uint32_t ts = (tw[t0 - g + FG] & 0x00ffu) | (tw[t1 - g + FG] & 0xff00u);
                uint32_t cmax = 0;
                uint32_t trw[RW];
                if (scan_only) {
                    if (step == 2) score_step<R, 2>(st[g].H, st[g].E, st[g].qp, cmax, ts, st[g].hu_prev, fin[g], st[g].fout, k);
                    else if (step == 1) score_step<R, 1>(st[g].H, st[g].E, st[g].qf, cmax, ts, st[g].hu_prev, fin[g], st[g].fout, k);
                    else score_step<R, 0>(st[g].H, st[g].E, st[g].qs, cmax, ts, st[g].hu_prev, fin[g], st[g].fout, k);
                } else {
                    if (tg) trace_step_tagged<R>(st[g].H, st[g].E, st[g].qs, ts, st[g].hu_prev, fin[g], st[g].fout, k, trw, cmax);
                    else trace_step_plain<R>(st[g].H, st[g].E, st[g].qs, ts, st[g].hu_prev, fin[g], st[g].fout, k, trw, cmax);
                    for (int w = 0; w < RW; ++w) tr[(size_t)tile_index<R>(u, g, w)] = trw[w];
                }
                st[g].hu_prev = hu[g];
                for (int L = 0; L < 2; ++L) {
                    if (!scan[L][g] || found[L][g]) continue;
                    const int cm = L == 0 ? lane_lo(cmax) : lane_hi(cmax);
                    if (cm != ctl[L].S * mul) continue;
                    for (int r = 0; r < R; ++r) {
                        const int hv = L == 0 ? lane_lo(st[g].H[r]) : lane_hi(st[g].H[r]);
                        if (hv == ctl[L].S * mul) {
                            found[L][g] = true;
                            ctl[L].fj[g] = (L == 0 ? t0 : t1) - g;
                            ctl[L].fr[g] = r;
                            break;
                        }
                    }
                }
            }
        }
        for (int L = 0; L < 2; ++L)
            for (int g = 0; g < FG; ++g)
                if (scan[L][g] && !found[L][g]) return -3;  // a candidate must find its cell
        for (int L = 0; L < 2; ++L) scans[L] += ctl[L].phase == 0;
        const uint32_t *tile = scan_only ? nullptr : tr.data();
        ctl_advance<R>(ctl[0], tile, 0, StagedAcc{ tw.data(), qc.data(), 0 }, k, sp0, ops_cap, end_only);
        ctl_advance<R>(ctl[1], tile, 1, StagedAcc{ tw.data(), qc.data(), 1 }, k, sp1, ops_cap, end_only);
        first_iter = false;
    }
    if (scan_info)
        for (int L = 0; L < 2; ++L) { scan_info[2 * L] = scans[L]; scan_info[2 * L + 1] = first_blk[L]; }
    if (end_only) {
        finalize_end(ctl[0], *out_a, 0);
        finalize_end(ctl[1], *out_b, 1);
        return 0;
    }
    finalize_result(ctl[0], *out_a, 0, clipl_a, clipr_a, min_length);
    finalize_result(ctl[1], *out_b, 1, clipl_b, clipr_b, min_length);
    if (ops_cap > 0) {
        const LaneCtl *cl[2] = { &ctl[0], &ctl[1] };
        uint32_t *dst[2] = { ops_a, ops_b };
        for (int L = 0; L < 2; ++L) {
            const LaneCtl &c = *cl[L];
            if (c.S <= 0 || c.nrev == 0) { for (int w = 0; w < ops_cap; ++w) dst[L][w] = 0; continue; }
            forward_ops(spill[L].data(), ops_cap, c.nrev, c.i + 1, c.qlen - 1 - c.end_i, dst[L]);
        }
    }
    return 0;
}

}  // namespace

extern "C" int fadeemu_align_pair(int R, const uint8_t *qa, int qlen_a, const uint8_t *ta, int tlen_a,
                                  const uint8_t *qb, int qlen_b, const uint8_t *tb, int tlen_b,
                                  int open, int extend, int match, int mismatch, int extra_blocks,
                                  int tagged, int min_length, const uint32_t *clips /*[4]: la ra lb rb*/,
                                  AlnOut *out_a, AlnOut *out_b)
{
    SwConsts k = make_consts(open, extend, match, mismatch);
    k.shortcut = (tagged & 2) ? 0 : 1;   // bit 1 of `tagged`: disable the ungapped-diagonal shortcut
                                         // bit 3: integer score-only step even where the fp16 one is exact
                                         // bit 4: fill_step_f16 even where fill_step_f16x2 is exact
#define CASE(RR)                                                                                   \
    case RR:                                                                                       \
        return align_pair<RR>(qa, qlen_a, ta, tlen_a, qb, qlen_b, tb, tlen_b, k, extra_blocks,    \
                              tagged, min_length, clips[0], clips[1], clips[2], clips[3], out_a, out_b);
    switch (R) {
        CASE(1) CASE(2) CASE(3) CASE(5) CASE(13) CASE(19) CASE(25) CASE(32) CASE(38)
    default: return -10;
    }
#undef CASE
}

// The same with the full-CIGAR spill of fadegpu_align_pairs: ops_a / ops_b receive the first ops_cap forward ops.
extern "C" int fadeemu_align_pair_ops(int R, const uint8_t *qa, int qlen_a, const uint8_t *ta, int tlen_a,
                                      const uint8_t *qb, int qlen_b, const uint8_t *tb, int tlen_b,
                                      int open, int extend, int match, int mismatch, int tagged, int ops_cap,
                                      AlnOut *out_a, AlnOut *out_b, uint32_t *ops_a, uint32_t *ops_b)
{
    if (ops_cap <= 0) return -11;
    SwConsts k = make_consts(open, extend, match, mismatch);
    k.shortcut = (tagged & 2) ? 0 : 1;
#define CASE(RR)                                                                                   \
    case RR:                                                                                       \
        return align_pair<RR>(qa, qlen_a, ta, tlen_a, qb, qlen_b, tb, tlen_b, k, 0, tagged, 0, 0, 0, 0, 0, \
                              out_a, out_b, ops_cap, ops_a, ops_b);
    switch (R) {
        CASE(1) CASE(2) CASE(3) CASE(5) CASE(13) CASE(19) CASE(25) CASE(32) CASE(38)
    default: return -10;
    }
#undef CASE
}

// The score-only calls (fadegpu_score_pairs / _regions): scan-only replays with the score-only step, walkers that stop
// at the end cell, finalize_end records.  scan_info[4]: per lane, the number of scan replays and the first candidate
// block (-1: no scan).  `tagged` bits 1, 3 and 4 as above.
extern "C" int fadeemu_score_pair(int R, const uint8_t *qa, int qlen_a, const uint8_t *ta, int tlen_a,
                                  const uint8_t *qb, int qlen_b, const uint8_t *tb, int tlen_b,
                                  int open, int extend, int match, int mismatch, int extra_blocks, int tagged,
                                  AlnOut *out_a, AlnOut *out_b, int32_t *scan_info)
{
    SwConsts k = make_consts(open, extend, match, mismatch);
    k.shortcut = (tagged & 2) ? 0 : 1;
#define CASE(RR)                                                                                   \
    case RR:                                                                                       \
        return align_pair<RR>(qa, qlen_a, ta, tlen_a, qb, qlen_b, tb, tlen_b, k, extra_blocks,    \
                              tagged | 32, 0, 0, 0, 0, 0, out_a, out_b, 0, nullptr, nullptr, scan_info);
    switch (R) {
        CASE(1) CASE(2) CASE(3) CASE(5) CASE(13) CASE(19) CASE(25) CASE(32) CASE(38)
    default: return -10;
    }
#undef CASE
}

// helpers exposed for unit tests of the decoding primitives
extern "C" int fadeemu_comp_code_of_nt16(int nib) { return comp_code_of_nt16(nib); }
extern "C" uint32_t fadeemu_prmt(uint32_t a, uint32_t b, uint32_t s) { return prmt_sx(a, b, s); }
extern "C" int fadeemu_sizeof_alnout(void) { return (int)sizeof(AlnOut); }
extern "C" int fadeemu_f16_ok(int open, int extend, int match, int mismatch) { return make_consts(open, extend, match, mismatch).f16_ok; }
extern "C" int fadeemu_tagged_ok(int open, int extend, int match, int mismatch) { return make_consts(open, extend, match, mismatch).tagged_ok; }
// make_consts' choice for fill_step_f16x2: out = { f16_pair_ok, high byte of match, of mismatch, IMAD addend c }
extern "C" void fadeemu_f16_pair(int open, int extend, int match, int mismatch, uint32_t *out)
{
    const SwConsts k = make_consts(open, extend, match, mismatch);
    out[0] = (uint32_t)k.f16_pair_ok; out[1] = k.plut0 & 0xffu; out[2] = (k.plut0 >> 8) & 0xffu; out[3] = k.pair_c;
}
// f16_step_exact(pair = true) for the given high bytes and addend
extern "C" int fadeemu_f16_pair_exact(int open, int extend, int match, int mismatch, uint32_t pm, uint32_t px, uint32_t c)
{
    SwConsts k = make_consts(open, extend, match, mismatch);
    k.plut0 = pm | (px << 8) | (px << 16) | (px << 24);
    k.plut1 = px * 0x01010101u;
    k.pair_c = c;
    return f16_step_exact(k, true) ? 1 : 0;
}
extern "C" void fadeemu_fma_f16x2(const uint32_t *a, const uint32_t *b, const uint32_t *c, uint32_t *out, int64_t n)
{
    for (int64_t i = 0; i < n; ++i) out[i] = fma_f16x2(a[i], b[i], c[i]);
}
