// spectrogram.cuh -- S1: waterfall rows for a batch of cycles.
//
// Restates AudioIn.get_hop_spectrum (receiver.py:288-293) driven once per 480-sample hop
// (receiver.py:295-306) for an isolated cycle (SURVEY.md A1, H5):
//     grid[h, k] = 20*log10(|rfft(x[480h-3840 : 480h] * hanning(3840))[k]| + 1e-12),  k < 976, 1 <= h <= 375
// with x = 0 before the cycle start and grid[0, :] = 1.0 (the reference's initial fill).
//
// One CTA of 128 threads per row (measured best on B200: 5.4 vs 6.1 ms / 2048 cycles with 4 rows per CTA).  The 3840-point
// real transform is a 1920-point complex Stockham FFT of z[n] = x[2n] + i*x[2n+1] in shared memory (passes 15,8,16);
// the first pass reads the windowed audio straight from global memory (int16 -> fp32 fused), the
// epilogue untangles only the 976 bins that are kept and writes dB.  Consecutive CTAs take adjacent rows,
// so their 7/8-overlapping windows hit L1/L2: HBM sees the audio once and the grid once.
//
// Round-2 experiments that REDUCED the shared-memory / L1 wavefronts per row and still lost (profiles/r02_experiments.md):
// two adjacent rows per 128-thread group sharing the window and twiddle loads with the untangle fused into the last pass
// (-22 % wavefronts, 96 registers, 5 CTAs/SM: 12.5 ms vs 7.7), and the fused untangle alone (-10 % wavefronts, z[16] live
// across two barriers: 9.7 ms).  The kernel is not on a single roof (data pipe 68 %, issue 60 %, FMA 45 % in ncu r02i): it
// needs its 32 resident warps of short, independent phases more than it needs fewer wavefronts.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "fft.cuh"

namespace ft8 {

constexpr int SP_NT = 128;          // threads per row
constexpr int SP_BUF_LEN = 1936;    // one in-place buffer (ping-pong buffers measured slower): 1920 + one pad element per 120
constexpr int SP_T8_OFF = 14 * 128;  // per-pass twiddle tables of the 1920-point transform: [(15,1): 14 x 128 | (8,15): 7 x 16]
constexpr int GRID_ROWS = 376, GRID_COLS = 976, CYCLE_SAMPLES = 180000, NFFT_S = 3840, HOP = 480;

// two consecutive samples starting at an even index (one 32-bit / 64-bit load)
__device__ __forceinline__ float2 load_sample_pair(const int16_t* a, int i) {
    const short2 v = __ldg(reinterpret_cast<const short2*>(a + i));
    return make_float2((float)v.x, (float)v.y);
}
__device__ __forceinline__ float2 load_sample_pair(const float* a, int i) { return __ldg(reinterpret_cast<const float2*>(a + i)); }

// RING = false: isolated cycles (the batch path; compiled exactly as before the live mode existed -- the extra branch in the
// 15-operand load loop cost 27 % when it was a run-time test).  RING = true: live mode, see prev_tail / out_wrap.
// Launch bounds: 64 registers -> 8 CTAs (32 warps) per SM; measured best on B200.
template <typename T, bool RING = false>
__global__ void __launch_bounds__(SP_NT, 8)
k_spectrogram(const T* __restrict__ audio, float* __restrict__ grid, const float* __restrict__ hann,
              const float2* __restrict__ TS, const float2* __restrict__ W3840, int row_lo, int row_hi, int out_rows,
              int out_row0, int fill_row0, const float* __restrict__ prev_tail = nullptr, int out_wrap = 0) {
    extern __shared__ float2 sp_smem[];
    const int cyc = blockIdx.y;
    const int lt = threadIdx.x;
    const int h = row_lo + blockIdx.x;                    // grid row = window ending at sample 480*h
    const bool live = h <= row_hi;
    float2* buf = sp_smem;
    const T* x = audio + (size_t)cyc * CYCLE_SAMPLES;
    // live ring (receiver.py:295-306): the windows of the first hops of a cycle reach back into the previous cycle's audio;
    // prev_tail holds its last 3840 samples per stream as float32, whatever T is (zeros for a stream without a previous
    // cycle; nullptr: isolated cycle, samples before the start read as 0)
    const float* xp = (RING && prev_tail) ? prev_tail + (size_t)cyc * NFFT_S : nullptr;
    float* out = grid + (size_t)cyc * out_rows * GRID_COLS;
    if (blockIdx.x == 0 && fill_row0) {
        for (int k = threadIdx.x; k < GRID_COLS; k += blockDim.x) out[k] = 1.0f;
    }
    const int s0 = HOP * h - NFFT_S;      // first sample of the window (may be negative)

    // pass (R=15, S=1, M=128) with operands gathered from global memory: butterfly p = lt reads z[p + 128 j], j < 15 --
    // exactly one butterfly per thread, radix 15 = 3 x 5 in registers
    {
        float2 a[15];
#pragma unroll
        for (int j = 0; j < 15; ++j) {
            const int n = lt + 128 * j;
            const int si = s0 + 2 * n;
            float2 z = make_float2(0.f, 0.f);
            if (live && si >= 0) {                      // si is even: the pair never straddles the cycle start
                const float2 w = __ldg(reinterpret_cast<const float2*>(hann + 2 * n));
                const float2 v = load_sample_pair(x, si);
                z = cmul_elem(v, w);
            } else if (RING && live && xp) {            // si in [-3840, 0): previous cycle's tail
                const float2 w = __ldg(reinterpret_cast<const float2*>(hann + 2 * n));
                const float2 v = load_sample_pair(xp, NFFT_S + si);
                z = cmul_elem(v, w);
            }
            a[j] = z;
        }
        Pass<1920, 15, 1>::template compute_store<false, true>(buf, lt, a, TS);
        __syncthreads();
    }
    // pass (R=8, S=15, M=16), p-major: butterflies t = lt and lt + 128 share p = lt % 16, so the 7 twiddles are loaded once
    // (16 consecutive entries per warp request); loads have stride 15 elements (odd: no bank conflict); the output goes to
    // the padded layout i + i/120 (element q + 120 p + 15 k -> q + 121 p + 15 k, stride 121 across lanes: no conflict --
    // unpadded, 25 % of this kernel's shared-store wavefronts were conflict replays).
    {
        const int p = lt & 15, q0 = lt >> 4;                       // q = q0 and q0 + 8 (second butterfly exists for q0 < 7)
        float2 w[7];
#pragma unroll
        for (int k = 1; k < 8; ++k) w[k - 1] = __ldg(&TS[SP_T8_OFF + (k - 1) * 16 + p]);
        float2 a[2][8];
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int q = q0 + 8 * i;
            if (q < 15) {
#pragma unroll
                for (int j = 0; j < 8; ++j) a[i][j] = buf[q + 15 * (p + 16 * j)];
            }
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int q = q0 + 8 * i;
            if (q < 15) {
                Dft<8, false>::run(a[i]);
                float2* d = buf + q + 121 * p;
                d[0] = a[i][0];
#pragma unroll
                for (int k = 1; k < 8; ++k) d[15 * k] = cmul(a[i][k], w[k - 1]);
            }
        }
        __syncthreads();
    }
    // last pass (R=16, S=120, M=1) on the padded layout, in place: each thread rewrites the 16 positions it read
    if (lt < 120) {
        float2 a[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) a[j] = buf[lt + 121 * j];
        Dft<16, false>::run(a);
#pragma unroll
        for (int k = 0; k < 16; ++k) buf[lt + 121 * k] = a[k];
    }
    __syncthreads();

    // untangle the real transform for bins 0..975 and write dB
    if (live) {
        int ri = h - out_row0;
        if (RING && out_wrap) ri %= out_rows;                   // 750-row ring: row 375 of the odd cycle is ring row 0
        float* row = out + (size_t)ri * GRID_COLS;
        for (int k = lt; k < GRID_COLS; k += SP_NT) {
            const int km = (k == 0) ? 0 : 1920 - k;
            const float2 zk = buf[k + k / 120];                     // padded layout
            const float2 zm = buf[km + km / 120];
            // e = (zk + conj(zm))/2,  o = -i/2 * (zk - conj(zm)) = (0.5 (zk.y + zm.y), -0.5 (zk.x - zm.x))
            const float2 e = cscale(0.5f, cfma_elem(zm, 1.0f, -1.0f, zk));
            const float2 dz = cfma_elem(zm, -1.0f, 1.0f, zk);
            const float2 o = make_float2(0.5f * dz.y, -0.5f * dz.x);
            const float2 w = __ldg(&W3840[k]);
            const float2 X = cadd(e, cmul(o, w));
            // 20*log10(|X| + 1e-12): for |X|^2 > 1e-8 the 1e-12 is below half an ulp of |X| and 20*log10|X| = 10*log10(|X|^2),
            // evaluated as (10*log10(2)) * log2 with the 2-ulp hardware log2; the exact form is kept for (near-)silent bins
            const float pw = fmaf(X.x, X.x, X.y * X.y);
            row[k] = (pw > 1e-8f) ? 3.01029995663981195f * __log2f(pw) : 20.0f * log10f(sqrtf(pw) + 1e-12f);
        }
    }
}

}  // namespace ft8
