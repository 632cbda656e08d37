// sw_core.cuh -- arithmetic core of the realignment kernels, shared by the sm_100a kernels
// (kernels.cu) and by the host-side lock-step emulation used in CPU tests (emu/emu.cu).
//
// What it replaces in the reference: parasail_sw_trace_striped_16 + parasail_result_get_cigar as
// reached through dparasail's Parasail.sw_striped at source/analysis.d:67,69 (rules P1-P5 of
// SURVEY.md 8a), plus the accept predicates of source/analysis.d:69-80,98-104.
//
// Layout of the dynamic program (one "group" of FG=8 threads per PAIR of alignments):
//   * the two alignments of a pair live in the two int16 lanes of every 32-bit word (s16x2);
//   * thread g of the group owns query rows [g*R, g*R+R) in registers (H, E, query codes);
//   * at step t thread g computes target column j = t - g (a skewed wavefront); the bottom-row H
//     and the running F are handed to thread g+1 with one shuffle each per step;
//   * every FBLK=32 steps the complete wavefront state is written to a checkpoint (coalesced),
//     so that the traceback can re-run any 32-step block with trace recording (no full trace
//     matrix is ever stored);
//   * scores are computed with DPX packed int16 instructions (VIADDMNMX / VIMNMX.S16x2).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define FD __host__ __device__ __forceinline__
#else
#define FD inline
#endif

namespace fade {

constexpr int FG = 8;     // threads per group
constexpr int FBLK = 32;  // steps per checkpoint block
constexpr int OPS_CAP = 10;  // == FADEGPU_MAX_OPS: fade rejects CIGARs of more than 10 ops (analysis.d:69)

// symbol codes (P1: parasail_matrix_create("ACTGN",...) order), plus padding codes
enum : int { C_A = 0, C_C = 1, C_T = 2, C_G = 3, C_N = 4, C_WILD = 5, C_TPAD = 6, C_QPAD = 7 };

// BAM CIGAR op codes
enum : uint32_t { OP_I = 1, OP_D = 2, OP_S = 4, OP_EQ = 7, OP_X = 8 };

struct SwConsts {
    uint32_t lut0, lut1;  // PRMT byte LUT indexed by (qcode ^ tcode): [0] = match, [1..7] = mismatch
    uint32_t neg_o, neg_e;  // packed (-open,-open), (-extend,-extend)
    int32_t open, extend, match, mismatch;
    // "tagged" x16 domain of the trace replay (value = 16*score + tag, see trace_step)
    uint32_t tlut0, tlut1;      // byte LUT of 16*s + 8 (the DIAG tag)
    uint32_t neg_o16;           // packed -16*open
    uint32_t neg_e16_e;         // packed -16*extend + 1 (E extension tag)
    uint32_t neg_e16_f;         // packed -16*extend + 2 (F extension tag)
    int32_t tagged_ok;          // scoring fits the tagged encoding
    int32_t shortcut;           // traceback may use the ungapped-diagonal proof instead of a replay
    uint32_t flut0, flut1;      // byte LUT of the fp16 score words of fill_step_f16
    int32_t f16_ok;             // fill_step_f16 is exact for this scoring (checked in make_consts)
    uint32_t plut0, plut1;      // byte LUT of the row-pair score words of fill_step_f16x2
    uint32_t pair_c;            // IMAD addend that forms the second row's word of a pair (see fill_step_f16x2)
    int32_t f16_pair_ok;        // fill_step_f16x2 is exact for this scoring (checked in make_consts)
};

// ---- packed helpers -------------------------------------------------------------------------
FD int lane_lo(uint32_t w) { return (int)(int16_t)(w & 0xffffu); }
FD int lane_hi(uint32_t w) { return (int)(int16_t)(w >> 16); }
FD uint32_t pack2(int lo, int hi) { return ((uint32_t)lo & 0xffffu) | ((uint32_t)hi << 16); }

// prmt.b32 in its default mode: selector nibble bit 3 replicates the sign of the selected byte.
FD uint32_t prmt_sx(uint32_t a, uint32_t b, uint32_t sel)
{
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
#else
    const uint64_t v = ((uint64_t)b << 32) | a;
    uint32_t d = 0;
    for (int i = 0; i < 4; ++i) {
        const uint32_t c = (sel >> (4 * i)) & 0xf;
        uint32_t byte = (uint32_t)(v >> (8 * (c & 7))) & 0xff;
        if (c & 8) byte = (byte & 0x80) ? 0xff : 0x00;
        d |= byte << (8 * i);
    }
    return d;
#endif
}

// selector-form code words: sel = q_sel ^ t_sel has nibbles (xa, xa|8, xb, xb|8)
FD uint32_t q_sel(int ca, int cb) { return (uint32_t)(ca * 0x11) | ((uint32_t)(cb * 0x11) << 8); }
FD uint32_t t_sel(int ca, int cb) { return (uint32_t)(ca * 0x11 | 0x80) | ((uint32_t)(cb * 0x11 | 0x80) << 8); }
FD uint32_t score_word(uint32_t qs, uint32_t ts, const SwConsts &k) { return prmt_sx(k.lut0, k.lut1, qs ^ ts); }

// ---- fp16x2 arithmetic on score words ----------------------------------------------------------
// A non-negative score n <= 2047 has the same bit pattern as int16 and as the fp16 number n * 2^-24
// (subnormals and the first normal binade both have ulp 2^-24), so HFMA2 and the DPX int16
// instructions can work on the same registers.  A negative fp16 result is sign-magnitude (0x8000 | m),
// i.e. negative as an int16, and a .RELU DPX instruction that consumes it clamps it to 0, as it clamps a
// two's-complement negative.  fp16 never carries from one lane into the other (an int16x2 IMAD does,
// which is why the integer step cannot use the FMA pipe this way; DESIGN.md 4.1).
//
// Host branch: exact emulation of one lane of fma.rn.f16 on finite operands: exact product and sum, one
// round-to-nearest-even to fp16, overflow to infinity, IEEE signs of zero results.
FD uint32_t f16_fma_lane(uint32_t a, uint32_t b, uint32_t c)
{
    struct Dec { int neg, m, e; };   // |value| = m * 2^(e - 24)
    auto dec = [](uint32_t x) {
        const int ex = (int)((x >> 10) & 31), fr = (int)(x & 1023);
        return Dec{ (int)((x >> 15) & 1), ex ? (fr | 1024) : fr, ex ? ex - 1 : 0 };
    };
    const Dec da = dec(a), db = dec(b), dc = dec(c);
    // exact values in units of 2^-48: |product| < 2^80, |c| < 2^64
    const __int128 p = (__int128)((int64_t)da.m * db.m) << (da.e + db.e);
    const __int128 q = (__int128)dc.m << (dc.e + 24);
    const __int128 v = ((da.neg ^ db.neg) ? -p : p) + (dc.neg ? -q : q);
    if (v == 0) return (p == 0 && q == 0 && (da.neg ^ db.neg) && dc.neg) ? 0x8000u : 0u;
    const uint32_t sign = v < 0 ? 0x8000u : 0u;
    const __int128 av = v < 0 ? -v : v;
    int e = 0;
    while (e < 30 && (av >> (24 + e)) >= 2048) ++e;
    const int sh = 24 + e;
    __int128 m = av >> sh;
    const __int128 rem = av - (m << sh), half = (__int128)1 << (sh - 1);
    if (rem > half || (rem == half && (m & 1))) ++m;
    if (m == 2048) { m = 1024; ++e; }
    if (e > 29) return sign | 0x7c00u;
    if (m < 1024) return sign | (uint32_t)m;                          // subnormal (e == 0)
    return sign | ((uint32_t)(e + 1) << 10) | (uint32_t)(m - 1024);
}

// fma.rn.f16x2 without .ftz: the subnormals are the scores, they must not flush
FD uint32_t fma_f16x2(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    uint32_t d;
    asm("fma.rn.f16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
#else
    return f16_fma_lane(a & 0xffffu, b & 0xffffu, c & 0xffffu) | (f16_fma_lane(a >> 16, b >> 16, c >> 16) << 16);
#endif
}

// packed fp16 2^-24: fma_f16x2(s, F16_UNIT, h) adds the fp16 number s to h in units of the score grid
constexpr uint32_t F16_UNIT = 0x00010001u;

// Query words of the fp16 step: against the same t_sel target words, sel = q_self ^ t_sel has nibbles
// (xa|8, xa, xb|8, xb), so each lane is (LUT byte in the high half, its sign replicated in the low half).
FD uint32_t q_self(int ca, int cb) { return (uint32_t)(ca * 0x11 | 0x88) | ((uint32_t)(cb * 0x11 | 0x88) << 8); }
FD uint32_t score_word_f16(uint32_t qs, uint32_t ts, const SwConsts &k) { return prmt_sx(k.flut0, k.flut1, qs ^ ts); }

// Query word of a row pair for fill_step_f16x2: against the same t_sel target words, sel = q_pair ^ t_sel has nibbles
// (xa1, xa0, xb1, xb0) (x = q ^ t of lane a / b in the pair's first row 0 and second row 1), so one PRMT yields
// [sa1, sa0, sb1, sb0]: the first row's fp16 word in both lanes, with the second row's bytes as its low bytes.
FD uint32_t q_pair(int ca0, int cb0, int ca1, int cb1)
{
    return (uint32_t)(ca1 | (ca0 | 8) << 4) | ((uint32_t)(cb1 | (cb0 | 8) << 4) << 8);
}

// fp16 word w (16 bits) in units of 2^-25
FD int64_t f16_word_x2(uint32_t w)
{
    const int ex = (int)((w >> 10) & 31), fr = (int)(w & 1023);
    const int64_t mag = ex ? (int64_t)(fr | 1024) << ex : (int64_t)fr * 2;
    return (w & 0x8000u) ? -mag : mag;
}

// fp16 word (b:00 for b < 0x80, b:FF otherwise -- what score_word_f16 produces from LUT byte b) in units of 2^-25
FD int64_t f16_byte_word_x2(uint32_t b) { return f16_word_x2(b < 0x80 ? (b << 8) : ((b << 8) | 0xffu)); }

// How far inside half a unit of the score v the finite fp16 word hb:lb lies, in units of 2^-25 (> 0: it rounds to v
// when added to an integer; make_consts still checks the choice with f16_step_exact)
FD int64_t f16_pair_margin(uint32_t hb, uint32_t lb, int v)
{
    if ((hb & 0x7c) == 0x7c) return -1;   // infinity / NaN
    const int64_t d = f16_word_x2((hb << 8) | lb) - ((int64_t)v << 25);
    return ((int64_t)1 << 24) - (d < 0 ? -d : d);
}

// LUT byte for score v: the one whose word is nearest to v (+2 -> 0x40 = 2.0, -3 -> 0xC1 = -2.998).  Adding a
// word within half a unit of v to an integer n rounds to exactly n + v; make_consts checks it (f16_step_exact).
FD uint32_t f16_score_byte(int v)
{
    uint32_t best = 0;
    int64_t bd = -1;
    for (uint32_t b = 0; b < 256; ++b) {
        if ((b & 0x7c) == 0x7c) continue;   // infinity / NaN
        const int64_t d = f16_byte_word_x2(b) - ((int64_t)v << 25);
        const int64_t ad = d < 0 ? -d : d;
        if (bd < 0 || ad < bd) { bd = ad; best = b; }
    }
    return best;
}

// Is fill_step_f16 (pair == false) or fill_step_f16x2 (pair == true) exact for this scoring?  On the packed kernels
// (at most FG * 38 = 304 query rows) H stays within [0, max(match, mismatch) * 304].  For every H in that range and
// every score word the step can form, the fp16 diagonal add must give H + s where H + s > 0, and a word that is not
// positive as an int16 where H + s <= 0 (the .RELU max clamps it to 0).  fill_step_f16's words are a flut byte with
// its sign replicated below it; fill_step_f16x2's are a plut byte with any of the low bytes {fm, fx, pair_c} below it.
FD bool f16_step_exact(const SwConsts &k, bool pair = false)
{
    const int top = (k.match > k.mismatch ? k.match : k.mismatch) * FG * 38;
    if (top > 2047) return false;
    const int sc[2] = { k.match, k.mismatch };
    const uint32_t sel[2] = { q_self(0, 0) ^ t_sel(0, 0), q_self(0, 0) ^ t_sel(1, 1) };   // codes equal / different
    const uint32_t low[3] = { k.plut0 & 0xffu, (k.plut0 >> 8) & 0xffu, k.pair_c & 0xffu };
    for (int i = 0; i < 2; ++i) {
        for (int l = 0; l < (pair ? 3 : 1); ++l) {
            const uint32_t s = pair ? ((low[i] << 8) | low[l]) * 0x10001u : prmt_sx(k.flut0, k.flut1, sel[i]);
            for (int n = 0; n <= top; ++n) {
                const int want = n + sc[i];
                const uint32_t d = fma_f16x2(s, F16_UNIT, (uint32_t)n * 0x10001u);
                if (want > 0 ? d != (uint32_t)want * 0x10001u : (lane_lo(d) > 0 || lane_hi(d) > 0)) return false;
            }
        }
    }
    return true;
}

FD SwConsts make_consts(int open, int extend, int match, int mismatch)
{
    SwConsts k;
    const uint32_t m = (uint32_t)(match & 0xff), x = (uint32_t)(mismatch & 0xff);
    k.lut0 = m | (x << 8) | (x << 16) | (x << 24);
    k.lut1 = x | (x << 8) | (x << 16) | (x << 24);
    const uint32_t no = (uint32_t)((-open) & 0xffff), ne = (uint32_t)((-extend) & 0xffff);
    k.neg_o = no | (no << 16);
    k.neg_e = ne | (ne << 16);
    k.open = open; k.extend = extend; k.match = match; k.mismatch = mismatch;
    // The tagged recorder needs its DIAG candidates 16*s + 8 as signed LUT bytes, 16*(-open - extend) + 2 in an int16
    // lane, and 16*H + 15 in an int16 lane for every H of the tallest packed query (FG * 38 rows): H <= match * 304 <=
    // 2047.  Past that bound (match >= 7) 16*H wraps on queries of 2048 / match rows or more, so the plain recorder
    // (MODE 1) takes the scoring.
    const int tm = 16 * match + 8, tx = 16 * mismatch + 8;
    k.tagged_ok = (tm <= 127 && tx >= -128 && open <= 1000 && match * FG * 38 <= 2047) ? 1 : 0;
    const uint32_t bm = (uint32_t)(tm & 0xff), bx = (uint32_t)(tx & 0xff);
    k.tlut0 = bm | (bx << 8) | (bx << 16) | (bx << 24);
    k.tlut1 = bx | (bx << 8) | (bx << 16) | (bx << 24);
    const uint32_t o16 = (uint32_t)((-16 * open) & 0xffff);
    const uint32_t ee = (uint32_t)((-16 * extend + 1) & 0xffff), ef = (uint32_t)((-16 * extend + 2) & 0xffff);
    k.neg_o16 = o16 | (o16 << 16);
    k.neg_e16_e = ee | (ee << 16);
    k.neg_e16_f = ef | (ef << 16);
    k.shortcut = 1;
    const uint32_t fm = f16_score_byte(match), fx = f16_score_byte(mismatch);
    k.flut0 = fm | (fx << 8) | (fx << 16) | (fx << 24);
    k.flut1 = fx | (fx << 8) | (fx << 16) | (fx << 24);
    k.f16_ok = f16_step_exact(k) ? 1 : 0;
    // fill_step_f16x2: the high bytes pm / px and the addend c with the largest smallest margin over the words hb:lb,
    // hb in {pm, px}, lb in {pm, px, c} (default scoring: 0x3F = 1.75 + lb / 1024, 0xC1 = -2.5 - lb / 512, c = 0x3F;
    // 0xC1 with c = 0 would form -2.5, a tie).  The choice is then checked exactly.
    uint32_t pm = 0, px = 0, pc = 0;
    int64_t best = 0;
    for (uint32_t bm = 0; bm < 256; ++bm) {
        const int64_t m0 = f16_pair_margin(bm, bm, match);
        if (m0 <= best) continue;
        for (uint32_t bx = 0; bx < 256; ++bx) {
            int64_t m1 = m0;
            const int64_t mm[3] = { f16_pair_margin(bm, bx, match), f16_pair_margin(bx, bm, mismatch),
                                    f16_pair_margin(bx, bx, mismatch) };
            for (int i = 0; i < 3; ++i) m1 = mm[i] < m1 ? mm[i] : m1;
            if (m1 <= best) continue;
            for (uint32_t c = 0; c < 256; ++c) {
                const int64_t a = f16_pair_margin(bm, c, match), b = f16_pair_margin(bx, c, mismatch);
                const int64_t m2 = a < b ? (a < m1 ? a : m1) : (b < m1 ? b : m1);
                if (m2 > best) { best = m2; pm = bm; px = bx; pc = c; }
            }
        }
    }
    k.plut0 = pm | (px << 8) | (px << 16) | (px << 24);
    k.plut1 = px | (px << 8) | (px << 16) | (px << 24);
    k.pair_c = pc;
    k.f16_pair_ok = (best > 0 && f16_step_exact(k, true)) ? 1 : 0;
    return k;
}

// ---- reference / read decoding ----------------------------------------------------------------
// Device-resident reference: 2-bit plane (16 bases / word, code order A C T G), N plane and
// wildcard plane (1 bit / base).  Replaces fai.fetchSequence(...).toUpper, source/analysis.d:63.
struct RefPlanes {
    const uint32_t *two;  // 2 bits per base
    const uint32_t *nmask;
    const uint32_t *xmask;
};

FD int ref_code(const RefPlanes &rp, int64_t p)
{
    const uint32_t w = rp.two[p >> 4];
    int c = (int)((w >> (2 * (int)(p & 15))) & 3u);
    if ((rp.nmask[p >> 5] >> (int)(p & 31)) & 1u) c = C_N;
    if ((rp.xmask[p >> 5] >> (int)(p & 31)) & 1u) c = C_WILD;
    return c;
}

// BAM nt16 nibble of base i (source/util.d:31)
FD int nt16_at(const uint8_t *seq4, int i) { return (seq4[i >> 1] >> ((~i & 1) << 2)) & 0xf; }

// code of the COMPLEMENT of an nt16 nibble (source/util.d:18-21 seq_comp_table then P1 mapper):
// A(1)->T, C(2)->G, G(4)->C, T(8)->A, N(15)->N, everything else -> wildcard
FD int comp_code_of_nt16(int nib)
{
    // nibble-indexed LUT: idx 1->C_T(2), 2->C_G(3), 4->C_C(1), 8->C_A(0), 15->C_N(4), else 5
    const uint64_t lut = 0x4555555055515325ull;
    return (int)((lut >> (4 * nib)) & 0xf);
}

// row i of the reverse-complemented read (source/util.d:23-34, source/analysis.d:40)
FD int rc_query_code(const uint8_t *seq4, int qlen, int i)
{
    return comp_code_of_nt16(nt16_at(seq4, qlen - 1 - i));
}

// ---- DP steps -----------------------------------------------------------------------------------
FD uint32_t FADE_VADD(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vadd2(a, b);
#else
    return pack2(lane_lo(a) + lane_lo(b), lane_hi(a) + lane_hi(b));
#endif
}
FD uint32_t FADE_VMAX(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vmaxs2(a, b);
#else
    const int l = lane_lo(a) > lane_lo(b) ? lane_lo(a) : lane_lo(b);
    const int h = lane_hi(a) > lane_hi(b) ? lane_hi(a) : lane_hi(b);
    return pack2(l, h);
#endif
}
FD uint32_t FADE_VMAX3(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __vimax3_s16x2(a, b, c);
#else
    return FADE_VMAX(FADE_VMAX(a, b), c);
#endif
}
FD uint32_t FADE_VIADDMAX(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __viaddmax_s16x2(a, b, c);
#else
    return FADE_VMAX(FADE_VADD(a, b), c);
#endif
}
FD uint32_t FADE_VIADDMAX_RELU(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __viaddmax_s16x2_relu(a, b, c);
#else
    return FADE_VMAX(FADE_VIADDMAX(a, b, c), 0u);
#endif
}

// One wavefront step of the score-only pass for one thread: column j of rows [0,R) of this thread.
//   hdiag = H[first_row-1][j-1], f_in = F[first_row][j]; returns f_out = F[first_row+R][j].
// P2: E[i][j+1] = max(H[i][j]-o, E[i][j]-e); F[i+1][j] = max(H[i][j]-o, F[i][j]-e);
//     H = max(0, Hdiag + s, E, F).
// Per packed cell pair: LOP3 + PRMT (score), VIADDMNMX.RELU, VIMNMX, VIADD (H-open), 2x VIADDMNMX and
// half a VIMNMX3 (running maximum over two rows) = 7.5 ALU-pipe instructions, all of them issued at
// 64 threads / clk / SM (profiles/r01_ubench_b200.txt).  The score-only pass uses it for scorings that
// fill_step_f16 below cannot take exactly (SwConsts::f16_ok == 0).  Moving H-open to the FMA pipe as a
// 32-bit IMAD needs a biased domain (a negative low lane borrows from the high lane), in which the .RELU
// zero floor no longer works; fp16x2 has neither problem (DESIGN.md 4.1).
template <int R>
FD void fill_step(uint32_t (&H)[R], uint32_t (&E)[R], const uint32_t (&qs)[R], uint32_t &M,
                  uint32_t ts, uint32_t hdiag, uint32_t f_in, uint32_t &f_out, const SwConsts &k)
{
    uint32_t f = f_in;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t s = score_word(qs[r], ts, k);
        const uint32_t t1 = FADE_VIADDMAX_RELU(hdiag, s, E[r]);
        const uint32_t h = FADE_VMAX(t1, f);
        hdiag = H[r];
        H[r] = h;
        const uint32_t ho = FADE_VADD(h, k.neg_o);
        E[r] = FADE_VIADDMAX(E[r], k.neg_e, ho);
        f = FADE_VIADDMAX(f, k.neg_e, ho);
        M = FADE_VMAX(M, h);
    }
    f_out = f;
}

FD uint32_t FADE_VMAX3_RELU(uint32_t a, uint32_t b, uint32_t c)
{
#if defined(__CUDA_ARCH__)
    return __vimax3_s16x2_relu(a, b, c);
#else
    return FADE_VMAX(FADE_VMAX3(a, b, c), 0u);
#endif
}

// fill_step with the diagonal add on the FMA pipe, for scorings with k.f16_ok (query words from q_self): Hdiag + s
// is one HFMA2 on the fp16 score word (exact, see the fp16 section above; a negative sum reads as a negative int16),
// and max(0, Hdiag + s, E, F) one VIMNMX3.RELU, which replaces VIADDMNMX.RELU + VIMNMX.  H, E and F, and so the
// checkpoints, are bit-identical to fill_step's.  Moving H - open to the FMA pipe as well (HADD2, with E' and F'
// clamped at 0) was measured no faster: VIADD.16x2 already co-issues with the DPX max instructions
// (profiles/r03_ubench_b200.txt).
template <int R>
FD void fill_step_f16(uint32_t (&H)[R], uint32_t (&E)[R], const uint32_t (&qs)[R], uint32_t &M,
                      uint32_t ts, uint32_t hdiag, uint32_t f_in, uint32_t &f_out, const SwConsts &k)
{
    uint32_t f = f_in;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t d = fma_f16x2(score_word_f16(qs[r], ts, k), F16_UNIT, hdiag);
        const uint32_t h = FADE_VMAX3_RELU(d, E[r], f);
        hdiag = H[r];
        H[r] = h;
        const uint32_t ho = FADE_VADD(h, k.neg_o);
        E[r] = FADE_VIADDMAX(E[r], k.neg_e, ho);
        f = FADE_VIADDMAX(f, k.neg_e, ho);
        M = FADE_VMAX(M, h);
    }
    f_out = f;
}

// fill_step_f16 with one substitution lookup for every two rows, for scorings with k.f16_pair_ok (query words from
// q_pair, ceil(R/2) of them).  One LOP3 + PRMT gives w = [sa1, sa0, sb1, sb0], which is the first row's score word in
// both lanes (its low bytes sa1 / sb1 are don't-cares); one IMAD gives w * 256 + c = [c, sa1, sa0, sb1], the second
// row's word (low bytes c and sa0).  make_consts picks the LUT bytes and c so that every such low byte leaves the
// word within half a unit of its score.  The IMAD runs on the FMA pipe beside the DPX maxima (c is not a compile-time
// constant, so the multiply-add stays an IMAD rather than a shift on the ALU pipe).  An odd R pairs its last row with
// a padding code.  H, E and F are bit-identical to fill_step's (DESIGN.md 4.1).
template <int R>
FD void fill_step_f16x2(uint32_t (&H)[R], uint32_t (&E)[R], const uint32_t (&qp)[(R + 1) / 2], uint32_t &M,
                        uint32_t ts, uint32_t hdiag, uint32_t f_in, uint32_t &f_out, const SwConsts &k)
{
    uint32_t f = f_in, w = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        uint32_t s;
        if ((r & 1) == 0) s = w = prmt_sx(k.plut0, k.plut1, qp[r >> 1] ^ ts);
        else s = w * 256u + k.pair_c;
        const uint32_t d = fma_f16x2(s, F16_UNIT, hdiag);
        const uint32_t h = FADE_VMAX3_RELU(d, E[r], f);
        hdiag = H[r];
        H[r] = h;
        const uint32_t ho = FADE_VADD(h, k.neg_o);
        E[r] = FADE_VIADDMAX(E[r], k.neg_e, ho);
        f = FADE_VIADDMAX(f, k.neg_e, ho);
        M = FADE_VMAX(M, h);
    }
    f_out = f;
}

// The score-only steps: STEP 0 fill_step, 1 fill_step_f16, 2 fill_step_f16x2 (make_consts decides which is exact:
// score_step_for).  Their query words: one per row (q_sel / q_self) or one per row pair (q_pair).
FD int score_step_for(const SwConsts &k) { return k.f16_pair_ok ? 2 : (k.f16_ok ? 1 : 0); }
template <int R, int STEP> FD constexpr int query_words() { return STEP == 2 ? (R + 1) / 2 : R; }

// Set the query word(s) of row r (rows in order: the first row of a pair also writes the padding code of a second row)
template <int STEP, int N>
FD void set_query(uint32_t (&qs)[N], int r, int ca, int cb)
{
    if (STEP == 0) qs[r] = q_sel(ca, cb);
    else if (STEP == 1) qs[r] = q_self(ca, cb);
    else if ((r & 1) == 0) qs[r >> 1] = q_pair(ca, cb, C_QPAD, C_QPAD);
    else qs[r >> 1] = (qs[r >> 1] & 0xf0f0u) | (uint32_t)ca | ((uint32_t)cb << 8);
}

template <int R, int STEP>
FD void score_step(uint32_t (&H)[R], uint32_t (&E)[R], const uint32_t (&qs)[query_words<R, STEP>()], uint32_t &M,
                   uint32_t ts, uint32_t hdiag, uint32_t f_in, uint32_t &f_out, const SwConsts &k)
{
    if constexpr (STEP == 2) fill_step_f16x2<R>(H, E, qs, M, ts, hdiag, f_in, f_out, k);
    else if constexpr (STEP == 1) fill_step_f16<R>(H, E, qs, M, ts, hdiag, f_in, f_out, k);
    else fill_step<R>(H, E, qs, M, ts, hdiag, f_in, f_out, k);
}

// Trace nibble of cell (i,j) (one per int16 lane):
//   bit 0   = E[i][j+1] was obtained by EXTENSION (0: opened from H[i][j]; open iff H-o > E-e)
//   bit 1   = F[i+1][j] was obtained by EXTENSION
//   bits 2-3 = source of H[i][j]: 2 = DIAG, 1 = F, 0 = E   (P4 priority DIAG > F > E)
// A cell with H == 0 always stops the traceback (ZERO); the walker knows H along the path, so
// ZERO needs no code of its own.
// Storage: one 32-bit word per (step, thread, row quad): rows 4w..4w+3 of lane a in bits 0-15,
// of lane b in bits 16-31.
template <int R> FD constexpr int trace_words() { return (R + 3) / 4; }

FD uint32_t trace_nibble_plain(int d0, int ev, int fv, int h, int o, int e)
{
    uint32_t nib = (h == d0) ? 8u : ((h == fv) ? 4u : 0u);
    if (!(h - o > ev - e)) nib |= 1u;
    if (!(h - o > fv - e)) nib |= 2u;
    return nib;
}

// Wavefront step with trace recording, plain score domain, any scoring (unpacked compares).
// trw receives trace_words<R>() words; cmax accumulates the packed maximum of H over the rows.
template <int R>
FD void trace_step_plain(uint32_t (&H)[R], uint32_t (&E)[R], const uint32_t (&qs)[R],
                         uint32_t ts, uint32_t hdiag, uint32_t f_in, uint32_t &f_out, const SwConsts &k,
                         uint32_t *trw, uint32_t &cmax)
{
    uint32_t f = f_in, acc = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t s = score_word(qs[r], ts, k);
        const uint32_t d0 = FADE_VIADDMAX_RELU(hdiag, s, 0u);
        const uint32_t ev = E[r];
        const uint32_t h = FADE_VMAX(FADE_VMAX(d0, ev), f);
        const uint32_t nl = trace_nibble_plain(lane_lo(d0), lane_lo(ev), lane_lo(f), lane_lo(h), k.open, k.extend);
        const uint32_t nh = trace_nibble_plain(lane_hi(d0), lane_hi(ev), lane_hi(f), lane_hi(h), k.open, k.extend);
        acc |= (nl | (nh << 16)) << (4 * (r & 3));
        if ((r & 3) == 3 || r == R - 1) { trw[r >> 2] = acc; acc = 0; }
        hdiag = H[r];
        H[r] = h;
        cmax = FADE_VMAX(cmax, h);
        const uint32_t ho = FADE_VADD(h, k.neg_o);
        E[r] = FADE_VIADDMAX(ev, k.neg_e, ho);
        f = FADE_VIADDMAX(f, k.neg_e, ho);
    }
    f_out = f;
}

// Same step in the TAGGED domain: every value is 16*score + tag, and the tag of the winner of
// each packed max IS the trace decision, so no compare / select instructions are needed:
//   DIAG candidate  16*(Hdiag+s) + 8        F candidate  16*F + 4 (+2 if F was extended)
//   E candidate     16*E (+1 if E was extended)
//   E' = max(16*(H-o) [tag 0 = opened], 16*(E-e) + 1 [extended wins ties])   likewise F' with +2.
// H[] holds CLEAN values (tag stripped); E[] and f carry their extension tag.
template <int R>
FD void trace_step_tagged(uint32_t (&H)[R], uint32_t (&E)[R], const uint32_t (&qs)[R],
                          uint32_t ts, uint32_t hdiag, uint32_t f_in, uint32_t &f_out, const SwConsts &k,
                          uint32_t *trw, uint32_t &cmax)
{
    uint32_t f = f_in, acc = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t s16 = prmt_sx(k.tlut0, k.tlut1, qs[r] ^ ts);
        const uint32_t t1 = FADE_VIADDMAX_RELU(hdiag, s16, E[r]);
        const uint32_t hv = FADE_VIADDMAX(f, 0x00040004u, t1);
        const uint32_t hc = hv & 0xfff0fff0u;
        hdiag = H[r];
        H[r] = hc;
        cmax = FADE_VMAX(cmax, hc);
        const uint32_t ho = FADE_VADD(hc, k.neg_o16);
        const uint32_t en = FADE_VIADDMAX(E[r] & 0xfff0fff0u, k.neg_e16_e, ho);
        const uint32_t fn = FADE_VIADDMAX(f & 0xfff0fff0u, k.neg_e16_f, ho);
        E[r] = en;
        f = fn;
        const uint32_t nib = (hv & 0x000c000cu) | ((en | fn) & 0x00030003u);
        acc += nib << (4 * (r & 3));
        if ((r & 3) == 3 || r == R - 1) { trw[r >> 2] = acc; acc = 0; }
    }
    f_out = f;
}

// plain -> tagged domain
FD uint32_t to_tagged(uint32_t w) { return (w << 4) & 0xfff0fff0u; }


enum : int { T_ZERO = 0, T_DIAG = 1, T_F = 2, T_E = 3, T_EOPEN = 4, T_FOPEN = 8 };  // generic kernel

// ---- geometry -----------------------------------------------------------------------------------
// cell (i,j) is computed by thread g = i / R at step t = j + g; block = t / FBLK, u = t % FBLK.
template <int R>
FD void locate(int i, int j, int &blk, int &u)
{
    const int g = i / R;
    const int t = j + g;
    blk = t / FBLK;
    u = t % FBLK;
}

// number of 32-step blocks needed for a target of tmax columns
FD constexpr int num_blocks(int tmax) { return (tmax + FG - 1 + FBLK - 1) / FBLK; }
// checkpoint words per thread: H[R], E[R], hu_prev, f_out
template <int R> FD constexpr int ck_words() { return 2 * R + 2; }

// ---- per-lane traceback control (lives in shared memory on the device) ---------------------------
struct LaneCtl {
    // filled from the score-only pass
    int32_t best[FG];   // per-thread running maximum
    int32_t blk[FG];    // block in which that maximum was first reached
    // scan results
    int32_t fj[FG];     // first column with H == S for candidate thread g (scan)
    int32_t fr[FG];     // ... and first row inside the thread
    uint32_t scanned;   // bit g: candidate g already scanned
    int32_t S;
    int32_t phase;      // 0 scan, 1 walk, 2 done
    int32_t next_blk;   // block to (re)play next, -1 = none
    int32_t cur_blk;    // block whose trace currently sits in shared memory (-1 none)
    // walker
    int32_t i, j, mode; // mode 0 = H, 1 = arrived in F, 2 = arrived in E
    int32_t hval, gval; // H of the current cell (mode 0) / value of the gap state we came from
    int32_t end_i, end_j;
    int32_t nrev;       // completed reversed RLE ops pushed so far
    uint32_t cur;       // op being accumulated (len<<4|op), 0 = none
    uint32_t ring[OPS_CAP];
    int32_t qlen, tlen;
};

FD void ctl_init(LaneCtl &c, int qlen, int tlen)
{
    c.qlen = qlen; c.tlen = tlen;
    int S = 0;
    for (int g = 0; g < FG; ++g) if (c.best[g] > S) S = c.best[g];
    c.S = S;
    c.scanned = 0;
    c.cur_blk = -1;
    c.nrev = 0; c.cur = 0;
    c.i = c.j = c.mode = 0;
    c.hval = c.gval = 0;
    c.end_i = c.end_j = 0;
    if (S <= 0 || qlen <= 0 || tlen <= 0) { c.phase = 2; c.next_blk = -1; return; }
    c.phase = 0;
    int nb = 0x7fffffff;
    for (int g = 0; g < FG; ++g) if (c.best[g] == S && c.blk[g] < nb) nb = c.blk[g];
    c.next_blk = nb;
}

// Does thread g have to look for its first H == S cell during the replay of c.next_blk?
FD bool ctl_scan_me(const LaneCtl &c, int g)
{
    return c.phase == 0 && c.best[g] == c.S && c.blk[g] == c.next_blk && !((c.scanned >> g) & 1u);
}

FD void walk_push(LaneCtl &c, uint32_t op)
{
    if (c.cur != 0 && (c.cur & 0xf) == op) { c.cur += 16; return; }
    if (c.cur != 0) { c.ring[c.nrev % OPS_CAP] = c.cur; ++c.nrev; }
    c.cur = (1u << 4) | op;
}

// Trace tile of one replayed block: word (u, w, g) = step u, row quad w, thread g.  The layout
// [u][w][g] makes the 8 threads of a group write 8 consecutive words (one 32 B sector) per store.
template <int R> FD constexpr int tile_words() { return FBLK * trace_words<R>() * FG; }
template <int R> FD int tile_index(int u, int g, int w) { return (u * trace_words<R>() + w) * FG + g; }

// bit g set: thread g must look for its first H == S cell during the replay of c.next_blk
FD uint32_t ctl_scanmask(const LaneCtl &c)
{
    uint32_t m = 0;
    if (c.phase != 0) return 0;
    for (int g = 0; g < FG; ++g)
        if (c.best[g] == c.S && c.blk[g] == c.next_blk && !((c.scanned >> g) & 1u)) m |= 1u << g;
    return m;
}

// After a replay of block c.next_blk (its trace tile is `tile`): advance the per-lane state
// machine.  lane = 0/1 (int16 half of the tile words); acc.qcode(i) / acc.tcode(j) give the symbol
// codes of query row i / target column j.  P3 (end cell) and P4 (traceback) of SURVEY 8a.
// Phase 0 bookkeeping after a scan replay (P3): mark the scanned candidates; either request the
// next candidate block (returns false) or select the end cell and switch to the walk (true).
template <int R>
FD bool ctl_select_end(LaneCtl &c)
{
    for (int g = 0; g < FG; ++g)
        if (c.best[g] == c.S && c.blk[g] == c.cur_blk) c.scanned |= 1u << g;
    int nb = 0x7fffffff;
    for (int g = 0; g < FG; ++g)
        if (c.best[g] == c.S && !((c.scanned >> g) & 1u) && c.blk[g] < nb) nb = c.blk[g];
    if (nb != 0x7fffffff) { c.next_blk = nb; return false; }
    // P3: smallest column holding S, then smallest row
    int bg = -1;
    for (int g = 0; g < FG; ++g)
        if (c.best[g] == c.S && (bg < 0 || c.fj[g] < c.fj[bg])) bg = g;
    c.end_j = c.fj[bg];
    c.end_i = bg * R + c.fr[bg];
    c.i = c.end_i; c.j = c.end_j; c.mode = 0;
    c.hval = c.S;
    c.phase = 1;
    return true;
}

// spill (optional): a second ring of `spill_cap` words in global storage that receives every op the walker completes,
// at ring[nrev % spill_cap], so that CIGARs longer than OPS_CAP can be assembled in full (fadegpu_align_pairs).
// c.ring is written as before either way.
// end_only (fadegpu_score_pairs / _regions): the alignment is done once its end cell is selected; no walk (finalize_end).
template <int R, class Acc>
FD void ctl_advance(LaneCtl &c, const uint32_t *tile, int lane, const Acc &acc, const SwConsts &k,
                    uint32_t *spill = nullptr, int spill_cap = 0, bool end_only = false)
{
    if (c.phase == 2) return;
    c.cur_blk = c.next_blk;
    if (c.phase == 0 && !ctl_select_end<R>(c)) return;
    if (end_only) { c.phase = 2; c.next_blk = -1; return; }
    // P4: walk while the current cell lies in the replayed block (hot fields in registers)
    int i = c.i, j = c.j, mode = c.mode, hval = c.hval, gval = c.gval, nrev = c.nrev;
    uint32_t cur = c.cur;
    const int cur_blk = c.cur_blk;
    bool done = false;
    int need = -1;
    auto push = [&](uint32_t op) {
        if (cur != 0 && (cur & 0xf) == op) { cur += 16; return; }
        if (cur != 0) { c.ring[nrev % OPS_CAP] = cur; if (spill) spill[nrev % spill_cap] = cur; ++nrev; }
        cur = (1u << 4) | op;
    };
    for (;;) {
        if (i < 0 || j < 0) { done = true; break; }
        if (mode == 0 && hval <= 0) { done = true; break; }   // ZERO
        const int g = i / R, r = i - g * R;
        const int t = j + g;
        const int blk = t / FBLK, u = t % FBLK;
        if (blk != cur_blk || tile == nullptr) {   // tile == nullptr: the block was only scanned, not traced
            // Ungapped-diagonal proof (no replay needed): we are in state H at a cell whose exact value
            // hval is known.  Any ungapped alignment of k steps ending here scores at most hval, so the
            // remainder R_k = hval - sum of the k step scores is never negative; if it reaches exactly 0,
            // H == Hdiag + s holds at every cell on the way (induction over H >= Hdiag + s and
            // H >= R), DIAG has priority in the traceback (P4), and the cell after the last step holds
            // 0 (ZERO).  So the remaining path IS this diagonal.  If the diagonal leaves the matrix
            // first, nothing is proven and the block is replayed.
            if (mode == 0 && k.shortcut) {
                int rem = hval, steps = 0;
                bool proven = false;
                for (int ii = i, jj = j; ii >= 0 && jj >= 0; --ii, --jj) {
                    rem -= acc.qcode(ii) == acc.tcode(jj) ? k.match : k.mismatch;
                    ++steps;
                    if (rem <= 0) { proven = rem == 0; break; }
                }
                if (proven) {
                    for (int m = 0; m < steps; ++m) push(acc.qcode(i - m) == acc.tcode(j - m) ? OP_EQ : OP_X);
                    i -= steps; j -= steps; hval = 0;
                    continue;
                }
            }
            need = blk;
            break;
        }
        const uint32_t nib = (tile[tile_index<R>(u, g, r >> 2)] >> (16 * lane + 4 * (r & 3))) & 0xfu;
        if (mode == 0) {
            const uint32_t src = nib >> 2;
            if (src == 2u) {
                const bool eq = acc.qcode(i) == acc.tcode(j);
                push(eq ? OP_EQ : OP_X);
                hval -= eq ? k.match : k.mismatch;
                --i; --j;
            } else if (src == 1u) { push(OP_I); --i; mode = 1; gval = hval; }
            else { push(OP_D); --j; mode = 2; gval = hval; }
        } else if (mode == 1) {
            if (!(nib & 2u)) { hval = gval + k.open; mode = 0; }
            else { push(OP_I); --i; gval += k.extend; }
        } else {
            if (!(nib & 1u)) { hval = gval + k.open; mode = 0; }
            else { push(OP_D); --j; gval += k.extend; }
        }
    }
    c.i = i; c.j = j; c.mode = mode; c.hval = hval; c.gval = gval;
    if (done && cur != 0) {   // flush the last op
        c.ring[nrev % OPS_CAP] = cur;
        if (spill) spill[nrev % spill_cap] = cur;
        ++nrev; cur = 0;
    }
    c.cur = cur; c.nrev = nrev;
    if (!done) { c.next_blk = need; return; }
    c.phase = 2;
    c.next_blk = -1;
}

// accessor over staged arrays (emulation and unit tests)
struct StagedAcc {
    const uint16_t *tw;   // target selector words, column j at index j + FG
    const uint8_t *qc;    // query codes, lane a low nibble, lane b high nibble
    int lane;
    FD int qcode(int i) const { return (qc[i] >> (4 * lane)) & 0x7; }
    FD int tcode(int j) const { return (tw[j + FG] >> (8 * lane)) & 0x7; }
};

// ---- result record (device -> host, one per alignment) ---------------------------------------
struct AlnOut {
    int32_t score, end_query, end_ref, beg_query, beg_ref, n_ops;
    uint32_t flags;  // FADEGPU_R_*
    int32_t read;    // index of the read inside the batch
    uint32_t ops[OPS_CAP];
};

constexpr uint32_t R_ALIGNED = 1u, R_ART_LEFT = 2u, R_ART_RIGHT = 4u, R_OPS_TRUNC = 8u, R_GENERIC = 16u, R_SCORE_ONLY = 64u;

// accept predicate for one side, source/analysis.d:69-80 (left) / :98-104 (right)
FD bool accept_side(bool left, int score, int n_ops, uint32_t first_op, uint32_t last_op,
                    int lead_s, int trail_s, uint32_t clip_len, int32_t min_length)
{
    if (clip_len == 0 || clip_len <= (uint32_t)min_length) return false;  // analysis.d:34 (uint <= int)
    if (n_ops == 0 || n_ops > 10) return false;                          // analysis.d:69-70
    const uint32_t edge = left ? last_op : first_op;
    if ((edge & 0xf) != OP_EQ) return false;                             // analysis.d:74 / :98
    const float cutoff = (float)((double)clip_len * 0.9 * 2);            // analysis.d:43
    if (!((float)score > cutoff)) return false;                          // analysis.d:76 / :100
    if (left) return !(trail_s != 0 || lead_s == 0);                     // analysis.d:78-80
    return !(lead_s != 0 || trail_s == 0);                               // analysis.d:102-104
}

// Can an alignment of this score be accepted on either side at all?  The score test of accept_side (analysis.d:43,
// 76 / 100, same float arithmetic) is the only predicate that needs nothing but the fill's result; when it fails for
// both clips no traceback can change the read's tags (FADEGPU_F_TAGS_ONLY).
FD bool score_may_accept(int score, uint32_t clip_left, uint32_t clip_right, int32_t min_length)
{
    for (int side = 0; side < 2; ++side) {
        const uint32_t clip_len = side == 0 ? clip_left : clip_right;
        if (clip_len == 0 || clip_len <= (uint32_t)min_length) continue;
        const float cutoff = (float)((double)clip_len * 0.9 * 2);
        if ((float)score > cutoff) return true;
    }
    return false;
}

// P5 (dparasail wrapper): forward CIGAR = [S lead] + reversed ring + [S trail].  `ring` holds the last `cap` of the
// nrev reversed ops the walker pushed (entry nrev % cap), i.e. the first ones of the forward CIGAR; dst receives the
// first min(n_ops, cap) forward ops, zero-padded to cap.  finalize_result and sw_generic_kernel do the same for their
// 10-entry rings.
FD void forward_ops(const uint32_t *ring, int cap, int nrev, int lead, int trail, uint32_t *dst)
{
    const int n = (lead > 0) + nrev + (trail > 0);
    int w = 0;
    if (lead > 0) dst[w++] = ((uint32_t)lead << 4) | OP_S;
    for (int k = nrev - 1; k >= 0 && w < cap; --k) {
        if (nrev - k > cap) break;  // older entries were overwritten in the ring
        dst[w++] = ring[k % cap];
    }
    if (trail > 0 && w < cap && w == n - 1) dst[w++] = ((uint32_t)trail << 4) | OP_S;
    for (int k = w; k < cap; ++k) dst[k] = 0;
}

// P5 (dparasail wrapper): forward CIGAR = [S lead] + reversed ring + [S trail]; then predicates.
FD void finalize_result(const LaneCtl &c, AlnOut &o, int read, uint32_t clip_left, uint32_t clip_right,
                        int32_t min_length)
{
    o.read = read;
    o.score = c.S;
    if (c.S <= 0 || c.nrev == 0) {
        o.end_query = o.end_ref = o.beg_query = o.beg_ref = 0;
        o.n_ops = 0;
        o.flags = R_ALIGNED;
        for (int k = 0; k < OPS_CAP; ++k) o.ops[k] = 0;
        return;
    }
    o.end_query = c.end_i;
    o.end_ref = c.end_j;
    o.beg_query = c.i + 1;
    o.beg_ref = c.j + 1;
    const int lead = o.beg_query, trail = c.qlen - 1 - c.end_i;
    const int n = (lead > 0) + c.nrev + (trail > 0);
    o.n_ops = n;
    int w = 0;   // (forward_ops with cap OPS_CAP, written out so that the annotate kernels compile as they always have)
    if (lead > 0) o.ops[w++] = ((uint32_t)lead << 4) | OP_S;
    for (int k = c.nrev - 1; k >= 0 && w < OPS_CAP; --k) {
        if (c.nrev - k > OPS_CAP) break;  // older entries were overwritten in the ring
        o.ops[w++] = c.ring[k % OPS_CAP];
    }
    if (trail > 0 && w < OPS_CAP && w == n - 1) o.ops[w++] = ((uint32_t)trail << 4) | OP_S;
    for (int k = w; k < OPS_CAP; ++k) o.ops[k] = 0;
    uint32_t flags = R_ALIGNED;
    if (n > OPS_CAP) flags |= R_OPS_TRUNC;
    // first / last op of the forward CIGAR (valid whenever n <= 10, the only case that matters)
    const uint32_t first_op = lead > 0 ? (uint32_t)OP_S : (c.ring[(c.nrev - 1) % OPS_CAP] & 0xf);
    const uint32_t last_op = trail > 0 ? (uint32_t)OP_S : (c.ring[0] & 0xf);
    if (accept_side(true, c.S, n, first_op, last_op, lead, trail, clip_left, min_length)) flags |= R_ART_LEFT;
    if (accept_side(false, c.S, n, first_op, last_op, lead, trail, clip_right, min_length)) flags |= R_ART_RIGHT;
    o.flags = flags;
}

// Score-only record (fadegpu_score_pairs / _regions): the score and the end cell P3 selected, no begin cell and no
// CIGAR.  Equal, field for field, to what finalize_result writes for score and end cell.
FD void finalize_end(const LaneCtl &c, AlnOut &o, int read)
{
    o.read = read;
    o.score = c.S;
    o.end_query = c.S > 0 ? c.end_i : 0;
    o.end_ref = c.S > 0 ? c.end_j : 0;
    o.beg_query = o.beg_ref = 0;
    o.n_ops = 0;
    o.flags = R_ALIGNED;
    for (int k = 0; k < OPS_CAP; ++k) o.ops[k] = 0;
}

}  // namespace fade
