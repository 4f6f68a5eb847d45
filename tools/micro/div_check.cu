// div_check.cu -- how often does the residual-corrected quotient of csrc/ldpc.cuh's check-node update differ from IEEE div.rn?
//   nvcc -arch=sm_100a -O3 -o div_check tools/micro/div_check.cu && ./div_check
// Operands are drawn from the ranges the LDPC check-node update divides in (decoders.py:146-149): P / t with |t| in
// (1e-6, 1], |P| <= |t|, and e / ((e - 1.18)(1.18 + e)) with e in [-1, 1].  Prints one JSON line.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>
__device__ __forceinline__ float div_rn_fast(float a, float b) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b));
    const float q = __fmul_rn(a, r);
    return __fmaf_rn(__fmaf_rn(-q, b, a), r, q);
}
__device__ __forceinline__ uint32_t rng(uint64_t& s) { s = s * 6364136223846793005ull + 1442695040888963407ull; return (uint32_t)(s >> 32); }
__device__ __forceinline__ float u01(uint64_t& s) { return (rng(s) >> 8) * (1.0f / 16777216.0f); }
__global__ void k(unsigned long long* out, int iters) {
    uint64_t s = 0x9e3779b97f4a7c15ull * (blockIdx.x * blockDim.x + threadIdx.x + 1);
    unsigned long long bad1 = 0, bad2 = 0, worse = 0;
    for (int i = 0; i < iters; ++i) {
        const float t = (u01(s) < 0.5f ? -1.f : 1.f) * exp2f(-20.0f * u01(s) * u01(s));        // |t| in (1e-6, 1], dense near 1
        const float P = t * (2.0f * u01(s) - 1.0f);
        const float e0 = __fdiv_rn(P, t), e1 = div_rn_fast(P, t);
        if (__float_as_uint(e0) != __float_as_uint(e1)) { ++bad1; if (fabsf(e0 - e1) > 1.5f * fabsf(e0) * 1.2e-7f) ++worse; }
        const float c = __fmul_rn(__fadd_rn(e0, -1.18f), __fadd_rn(1.18f, e0));
        const float n0 = __fdiv_rn(e0, c), n1 = div_rn_fast(e0, c);
        if (__float_as_uint(n0) != __float_as_uint(n1)) { ++bad2; if (fabsf(n0 - n1) > 1.5f * fabsf(n0) * 1.2e-7f) ++worse; }
    }
    atomicAdd(&out[0], bad1); atomicAdd(&out[1], bad2); atomicAdd(&out[2], worse);
}
int main() {
    unsigned long long* d; cudaMalloc(&d, 24); cudaMemset(d, 0, 24);
    const int blocks = 148 * 8, threads = 256, iters = 4096;
    k<<<blocks, threads>>>(d, iters);
    unsigned long long h[3]; cudaMemcpy(h, d, 24, cudaMemcpyDeviceToHost);
    const double n = (double)blocks * threads * iters;
    printf("{\"quotients_each\": %.0f, \"first_quotient_differs\": %llu, \"second_quotient_differs\": %llu, \"more_than_one_ulp\": %llu, "
           "\"rate\": %.3g, \"err\": %d}\n", n, h[0], h[1], h[2], (h[0] + h[1]) / (2 * n), (int)cudaGetLastError());
    return 0;
}
