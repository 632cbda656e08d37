// ubench.cu -- instruction-throughput microbenchmarks for the INT16x2 DP instruction mix on B200.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o ubench ubench.cu ; run on the GPU box.
// Prints thread-instructions / clk / SM for each kernel (8 independent chains per thread unless noted), then the
// score-only DP step of the fill kernel (sw_core.cuh) in cells / clk / SM.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
#include "../fade_b200/csrc/sw_core.cuh"

__device__ __forceinline__ uint32_t add_f16x2(uint32_t a, uint32_t b)
{
    uint32_t d;
    asm("add.rn.f16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
    return d;
}

// fade::fill_step_f16 with H - open as HADD2 on the FMA pipe too: its negative results are sign-magnitude, so E' and
// F' take the .RELU max (clamped at 0; H and the trace decisions would not change).  Measured here, not used.
template <int R>
__device__ __forceinline__ void fill_step_f16_ho(uint32_t (&H)[R], uint32_t (&E)[R], const uint32_t (&qs)[R], uint32_t &M,
                                                 uint32_t ts, uint32_t hdiag, uint32_t f_in, uint32_t &f_out,
                                                 const fade::SwConsts &k, uint32_t neg_o_f16)
{
    uint32_t f = f_in;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const uint32_t d = fade::fma_f16x2(fade::score_word_f16(qs[r], ts, k), fade::F16_UNIT, hdiag);
        const uint32_t h = __vimax3_s16x2_relu(d, E[r], f);
        hdiag = H[r];
        H[r] = h;
        const uint32_t ho = add_f16x2(h, neg_o_f16);
        E[r] = __viaddmax_s16x2_relu(E[r], k.neg_e, ho);
        f = __viaddmax_s16x2_relu(f, k.neg_e, ho);
        M = __vmaxs2(M, h);
    }
    f_out = f;
}

#define CHK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)

template <int KIND>
__global__ void __launch_bounds__(256) k(uint32_t *out, int iters, uint32_t c1, uint32_t c2, uint32_t one)
{
    uint32_t x[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) x[i] = threadIdx.x * 3 + i;
    uint32_t y[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) y[i] = threadIdx.x * 5 + i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (KIND == 0) x[i] = __viaddmax_s16x2(x[i], c1, c2);
                if (KIND == 1) x[i] = __vimax3_s16x2(x[i], c1, c2);
                // max / logic chains with loop-invariant operands collapse at compile time (max is idempotent, two LOP3 of the
                // same three inputs fuse into one): the second operand changes every iteration instead
                if (KIND == 2) { x[i] = __vmaxs2(x[i], y[i]); y[i] = __vadd2(y[i], c1); }            // VIMNMX + VIADD
                if (KIND == 3) x[i] = __vadd2(x[i], c1);
                if (KIND == 4) x[i] = __byte_perm(x[i], c1, c2);
                if (KIND == 5) { x[i] = (x[i] ^ y[i]) & c1; y[i] = (y[i] | x[i]) ^ c2; }             // 2 LOP3 of four inputs
                if (KIND == 6) x[i] = x[i] * one + c1;                       // IMAD
                if (KIND == 7) { x[i] = __viaddmax_s16x2(x[i], c1, c2); y[i] = y[i] * one + c1; }   // ALU + FMA pipes
                if (KIND == 8) { x[i] = __viaddmax_s16x2(x[i], c1, c2); y[i] = __vmaxs2(y[i], c1); } // 2 ALU
                if (KIND == 9) x[i] = __viaddmax_s16x2_relu(x[i], c1, c2);
                if (KIND == 10) { x[i] = __viaddmax_s16x2(x[i], c1, y[i]); y[i] = (y[i] ^ x[i]) & c2; }
                if (KIND == 11) { x[i] = __viaddmax_s16x2(x[i], c1, y[i]); y[i] = __viaddmax_s16x2(y[i], c2, x[i]); } // 3 register operands
                if (KIND == 12) { x[i] = __vmaxs2(x[i], y[i]); y[i] = y[i] * one + c1; }
                if (KIND == 13) x[i] = __vimax3_s16x2_relu(x[i], c1, c2);
                // fp16x2 on integer score words (sw_core.cuh): c1 / c2 are small subnormals
                if (KIND == 14) x[i] = fade::fma_f16x2(x[i], c1, c2);                                // HFMA2
                if (KIND == 15) x[i] = add_f16x2(x[i], c1);                                    // HADD2
                if (KIND == 16) { x[i] = __viaddmax_s16x2(x[i], c1, c2); y[i] = fade::fma_f16x2(y[i], c1, c2); }
                if (KIND == 17) { x[i] = __vimax3_s16x2_relu(x[i], c1, c2); y[i] = fade::fma_f16x2(y[i], c1, c2); }
                // co-issue with independent chains (the r02 LOP3 row, KIND 10, is a dependent pair and latency-bound)
                if (KIND == 18) { x[i] = __viaddmax_s16x2(x[i], c1, c2); y[i] = __byte_perm(y[i], x[i], c2); }
                if (KIND == 19) { x[i] = __viaddmax_s16x2(x[i], c1, c2); y[i] = (y[i] ^ x[i]) & c1; }
                if (KIND == 20) { x[i] = fade::fma_f16x2(x[i], c1, c2); y[i] = y[i] * one + c1; }
            }
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) r ^= x[i] ^ y[i];
    if (r == 0x12345678u) out[0] = r;
}

template <int KIND>
int run(const char *name, int per_iter, int sms, double mhz)
{
    uint32_t *d;
    CHK(cudaMalloc(&d, 64));
    const int blocks = sms * 8, threads = 256, iters = 2048;
    cudaEvent_t e0, e1;
    CHK(cudaEventCreate(&e0)); CHK(cudaEventCreate(&e1));
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        CHK(cudaEventRecord(e0));
        k<KIND><<<blocks, threads>>>(d, iters, 0x00010003u, 0xfffefffdu, 1u);
        CHK(cudaEventRecord(e1));
        CHK(cudaEventSynchronize(e1));
        float ms; CHK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep && ms < best) best = ms;
    }
    const double ops = (double)blocks * threads * iters * 64.0 * per_iter;
    const double per_clk_sm = ops / (best * 1e-3) / (mhz * 1e6) / sms;
    printf("%-34s %8.3f ms  %7.1f thread-instr/clk/SM  (%.2e /s)\n", name, best, per_clk_sm, ops / (best * 1e-3));
    cudaFree(d);
    return 0;
}

// The score-only step of sw_fill_kernel<19> on register data: 19 rows x 2 lanes per thread and step, the target
// word from 8 registers, the diagonal H from the thread's own bottom row (no shuffle, no memory traffic).  The target
// codes change with the iteration (rot), so the substitution lookups cannot be hoisted out of the loop.
// V = 0: fill_step, 1: fill_step_f16 (diagonal add on the FMA pipe), 2: fill_step_f16 with H - open there too,
// 3: fill_step_f16x2 (one lookup per row pair).
template <int V>
__global__ void __launch_bounds__(128, 5) step_k(uint32_t *out, int iters, fade::SwConsts k)
{
    constexpr int R = 19;
    constexpr int STEP = V == 3 ? 2 : (V ? 1 : 0);
    uint32_t H[R], E[R], qs[fade::query_words<R, STEP>()], ts[8];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        // codes the compiler cannot prove equal, so it cannot share lookups between rows
        const int ca = (int)((threadIdx.x * 2654435761u) >> (r + 3)) & 3, cb = (int)((threadIdx.x * 2246822519u) >> (r + 5)) & 3;
        fade::set_query<STEP>(qs, r, ca, cb);
        H[r] = 0u; E[r] = k.neg_o;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)
        ts[i] = fade::t_sel((int)((threadIdx.x * 3266489917u) >> (i + 7)) & 3, (int)((threadIdx.x * 668265263u) >> (i + 9)) & 3);
    uint32_t M = 0u, f = k.neg_o, hu_prev = 0u;
    for (int it = 0; it < iters; ++it) {
        const uint32_t rot = (uint32_t)(it & 3) * 0x1111u;   // target codes c ^ (it & 3), still in 0..3
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const uint32_t hu = H[R - 1];
            if constexpr (V == 0) fade::fill_step<R>(H, E, qs, M, ts[u] ^ rot, hu_prev, f, f, k);
            else if constexpr (V == 1) fade::fill_step_f16<R>(H, E, qs, M, ts[u] ^ rot, hu_prev, f, f, k);
            else if constexpr (V == 2) fill_step_f16_ho<R>(H, E, qs, M, ts[u] ^ rot, hu_prev, f, f, k, 0x800a800au);   // fp16 -10 (open)
            else fade::fill_step_f16x2<R>(H, E, qs, M, ts[u] ^ rot, hu_prev, f, f, k);
            hu_prev = hu;
        }
    }
    uint32_t r = M ^ f;
#pragma unroll
    for (int i = 0; i < R; ++i) r ^= H[i] ^ E[i];
    if (r == 0x12345678u) out[0] = r;
}

// returns the best time in ms (the first row is the baseline of the speed-up column), < 0 on an error
template <int V>
float run_step(const char *name, int sms, double mhz, double base_ms)
{
    uint32_t *d;
    if (cudaMalloc(&d, 64) != cudaSuccess) return -1.f;
    const fade::SwConsts kc = fade::make_consts(10, 2, 2, -3);
    const int blocks = sms * 5 * 4, threads = 128, iters = 512;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(e0);
        step_k<V><<<blocks, threads>>>(d, iters, kc);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) return -1.f;
        float ms; cudaEventElapsedTime(&ms, e0, e1);
        if (rep && ms < best) best = ms;
    }
    const double cells = (double)blocks * threads * iters * 8.0 * 2 * 19;
    printf("%-44s %8.3f ms  %6.2f cells/clk/SM  %5.3fx\n", name, best, cells / (best * 1e-3) / (mhz * 1e6) / sms,
           base_ms > 0 ? base_ms / best : 1.0);
    cudaFree(d);
    return best;
}

int main()
{
    cudaDeviceProp p; CHK(cudaGetDeviceProperties(&p, 0));
    int khz = 0; cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, 0);
    const double mhz = khz / 1000.0;
    printf("%s, %d SMs, max clock %.0f MHz (rates assume max clock)\n", p.name, p.multiProcessorCount, mhz);
    const int s = p.multiProcessorCount;
    run<0>("VIADDMNMX.S16x2", 1, s, mhz);
    run<9>("VIADDMNMX.S16x2.RELU", 1, s, mhz);
    run<1>("VIMNMX3.S16x2", 1, s, mhz);
    run<13>("VIMNMX3.S16x2.RELU", 1, s, mhz);
    run<2>("VIMNMX.S16x2 + VIADD.16x2 (2 per iter)", 2, s, mhz);
    run<3>("VIADD.16x2", 1, s, mhz);
    run<4>("PRMT", 1, s, mhz);
    run<5>("LOP3 (2 per iter)", 2, s, mhz);
    run<6>("IMAD", 1, s, mhz);
    run<7>("VIADDMNMX + IMAD (2 per iter)", 2, s, mhz);
    run<8>("VIADDMNMX + VIMNMX (2 per iter)", 2, s, mhz);
    run<10>("VIADDMNMX + LOP3 (2 per iter)", 2, s, mhz);
    run<11>("VIADDMNMX 3-reg x2 (2 per iter)", 2, s, mhz);
    run<12>("VIMNMX + IMAD (2 per iter)", 2, s, mhz);
    run<14>("HFMA2", 1, s, mhz);
    run<15>("HADD2", 1, s, mhz);
    run<16>("VIADDMNMX + HFMA2 (2 per iter)", 2, s, mhz);
    run<17>("VIMNMX3.RELU + HFMA2 (2 per iter)", 2, s, mhz);
    run<18>("VIADDMNMX + PRMT (2 per iter)", 2, s, mhz);
    run<19>("VIADDMNMX + LOP3 indep. (2 per iter)", 2, s, mhz);
    run<20>("HFMA2 + IMAD (2 per iter)", 2, s, mhz);
    const float base = run_step<0>("fill_step<19> (integer)", s, mhz, 0.0);
    run_step<1>("fill_step_f16<19> diagonal add on FMA (A)", s, mhz, base);
    run_step<2>("fill_step_f16<19> + H-open on FMA (A+B)", s, mhz, base);
    run_step<3>("fill_step_f16x2<19> one lookup per row pair", s, mhz, base);
    return 0;
}
