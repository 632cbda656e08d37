// Device side of tests/test_f16_step.py: runs fade::fma_f16x2 (sw_core.cuh) elementwise on the GPU,
// so that the test can compare the hardware with the host emulation the CPU tests rely on.
#include <cuda_runtime.h>
#include "../../fade_b200/csrc/sw_core.cuh"

__global__ void f16x2_kernel(const uint32_t *a, const uint32_t *b, const uint32_t *c, uint32_t *out, int64_t n)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        out[i] = fade::fma_f16x2(a[i], b[i], c[i]);
}

// out = fma_f16x2(a, b, c) over host arrays of n words; returns a cudaError_t
extern "C" int f16x2_device(const uint32_t *a, const uint32_t *b, const uint32_t *c, uint32_t *out, int64_t n)
{
    const size_t bytes = (size_t)n * 4;
    uint32_t *d[4] = { nullptr, nullptr, nullptr, nullptr };
    cudaError_t e = cudaSuccess;
    for (int i = 0; i < 4 && e == cudaSuccess; ++i) e = cudaMalloc(&d[i], bytes);
    if (e == cudaSuccess) e = cudaMemcpy(d[0], a, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d[1], b, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(d[2], c, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        f16x2_kernel<<<1024, 256>>>(d[0], d[1], d[2], d[3], n);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpy(out, d[3], bytes, cudaMemcpyDeviceToHost);
    for (int i = 0; i < 4; ++i) cudaFree(d[i]);
    return (int)e;
}
