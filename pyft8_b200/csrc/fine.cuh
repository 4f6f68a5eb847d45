// fine.cuh -- F1 (cycle spectrum) and F2/F3 (per-candidate fine time/frequency sync).
//
// F1 restates AudioIn.get_cycle_spectrum (receiver.py:280-286): rfft of the 180000-sample cycle
// zero-padded to 192000 (0.0625 Hz bins).  The real transform is a 96000-point complex transform
// of z[n] = x[2n] + i x[2n+1], done four-step as 375 x 256:
//   A (k_cs_cols): for 16 columns n2 at a time, 375-point FFTs over n1 (n = 256 n1 + n2) in shared
//                  memory, times w_96000^(n2 k1), to scratch Y[k1][n2];
//   B (k_cs_rows): 256-point FFTs of rows k1 and of their mirror rows 375-k1, then the real-FFT
//                  untangle for bins k = k1 + 375 k2 and 96000-k in the same CTA.
// Only bins [1418, 48832) are ever read by the fine stage (SURVEY.md 8a F1); the pipeline keeps bins
// < FINE_SPEC_STRIDE, the stand-alone op writes all 96001.
//
// F2/F3 restate Candidate._get_llr_fine / _get_signal_grid_fine (receiver.py:140-206; SURVEY A4/A5, H3):
// one CTA per candidate; 1000 bins around fb -> taper (upper edge taper is inverted in the reference and
// is reproduced as is) -> 3200-point inverse FFT in shared memory (passes 5,5,8,16; the first pass gathers the band
// straight from global memory, 2200 of its 3200 inputs are structurally zero) -> 32-sample symbol DFTs, four per warp.
// The 8 time tweaks share one inverse FFT; the 9 frequency tweaks need one each (the ftweak = 0 one is the time-scan
// transform).  Only the MIDDLE Costas block is scored, so for scoring the last FFT pass is evaluated on just the
// 224-238 samples that block covers; the winner's operands are kept in a third shared buffer and get the full last
// pass for the final 79x8 grid.  Scoring of transform e shares a barrier phase with the first pass of transform e+1.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "fft.cuh"
#include "sync.cuh"

namespace ft8 {

constexpr int CS_N = 96000, CS_N1 = 375, CS_N2 = 256, CS_COLS = 16, CS_NT = 256;
constexpr int FINE_SPEC_STRIDE = 49152;
constexpr int FINE_N = 3200, FINE_NT = 256;
#define FINE_BUFS 3        // best-so-far + baseband being built + FFT scratch (2-buffer variants measured 11 % slower)
// Last-pass operand buffers (po, pb) are stored with one pad element per 200 (index q + 201 j instead of q + 200 j): the
// stores of pass (8,25) then walk the banks continuously across the run boundaries of a warp (ncu: 22 % of this kernel's
// shared-store wavefronts were bank-conflict replays without it), the loads of the last pass stay consecutive in q.
constexpr int FINE_NP = FINE_N + FINE_N / 200;

template <typename T> __device__ __forceinline__ float2 load_pair(const T* x, int n);
template <> __device__ __forceinline__ float2 load_pair<int16_t>(const int16_t* x, int n) {
    const short2 v = *reinterpret_cast<const short2*>(x + 2 * n);
    return make_float2((float)v.x, (float)v.y);
}
template <> __device__ __forceinline__ float2 load_pair<float>(const float* x, int n) {
    return *reinterpret_cast<const float2*>(x + 2 * n);
}

// grid (16, B).  Y: [B][375][256] float2.
template <typename T>
__global__ void __launch_bounds__(CS_NT)
k_cs_cols(const T* __restrict__ audio, float2* __restrict__ Y, const float2* __restrict__ TC,
          const float2* __restrict__ W96000T) {
    extern __shared__ float2 cs_smem[];          // [16][375]
    const int cyc = blockIdx.y, n2_0 = blockIdx.x * CS_COLS;
    const T* x = audio + (size_t)cyc * CYCLE_SAMPLES;
    // 6000 sample pairs per CTA: batches of 8 independent loads per thread keep the memory pipe busy
    constexpr int LD_ITERS = (CS_COLS * CS_N1 + CS_NT - 1) / CS_NT;      // 24
#pragma unroll
    for (int b0 = 0; b0 < LD_ITERS; b0 += 8) {
        float2 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = threadIdx.x + (b0 + u) * CS_NT;
            const int n1 = i / CS_COLS, c = i - n1 * CS_COLS;
            const int n = CS_N2 * n1 + n2_0 + c;
            v[u] = (i < CS_COLS * CS_N1 && n < CYCLE_SAMPLES / 2) ? load_pair<T>(x, n) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = threadIdx.x + (b0 + u) * CS_NT;
            const int n1 = i / CS_COLS, c = i - n1 * CS_COLS;
            if (i < CS_COLS * CS_N1) cs_smem[c * CS_N1 + n1] = v[u];
        }
    }
    __syncthreads();
    // per-pass twiddle tables [k-1][p]: (3,1) 2 x 125 | (5,3) 4 x 25 | (5,15) 4 x 5; the last pass has none
    pass_inplace_batched<375, 3, 1, CS_COLS, CS_NT, false, true>(cs_smem, threadIdx.x, TC);
    pass_inplace_batched<375, 5, 3, CS_COLS, CS_NT, false, true, true>(cs_smem, threadIdx.x, TC + 250);   // p-major: strides 3 / 15
    pass_inplace_batched<375, 5, 15, CS_COLS, CS_NT, false, true>(cs_smem, threadIdx.x, TC + 350);
    pass_inplace_batched<375, 5, 75, CS_COLS, CS_NT, false>(cs_smem, threadIdx.x, TC);
    float2* y = Y + (size_t)cyc * CS_N;
    for (int i = threadIdx.x; i < CS_COLS * CS_N1; i += CS_NT) {
        const int k1 = i / CS_COLS, c = i - k1 * CS_COLS;
        const int n2 = n2_0 + c;
        const float2 w = __ldg(&W96000T[k1 * CS_N2 + n2]);       // = w_96000^(n2 k1), stored [k1][n2] so the load is coalesced
        y[k1 * CS_N2 + n2] = cmul(cs_smem[c * CS_N1 + k1], w);
    }
}

constexpr int CSR_G = 8;      // k1 values per CTA (plus their mirrors)
constexpr int CSR_STRIDE = CS_N2 + CS_N2 / 16 + 4;   // 276: row stride = 4 (mod 16) 8-byte banks, so the untangle's 8-row gathers are conflict-free
// grid (24, B): k1 in {0} u [1,187] in groups of 8.  spec: [B][spec_stride] float2, bins <= kmax written.
__global__ void __launch_bounds__(CS_NT)
k_cs_rows(const float2* __restrict__ Y, float2* __restrict__ spec, int spec_stride, int kmax,
          const float2* __restrict__ T256, const float2* __restrict__ W192000) {
    // [0..7] rows k1, [8..15] mirror rows 375-k1; row stride 272: the intermediate of the two radix-16 passes is stored
    // with one pad per 16 elements (Pad16Map), otherwise the first pass's stride-16 stores all hit one bank
    __shared__ float2 rows[2 * CSR_G][CSR_STRIDE];
    const int cyc = blockIdx.y, g0 = blockIdx.x * CSR_G;
    const float2* y = Y + (size_t)cyc * CS_N;
    {
        float2 v[2 * CSR_G];                         // thread = column; 16 independent row loads in flight
#pragma unroll
        for (int r = 0; r < 2 * CSR_G; ++r) {
            const int k1 = g0 + (r & (CSR_G - 1));
            const int row = (r < CSR_G) ? k1 : (CS_N1 - k1) % CS_N1;
            v[r] = (k1 <= 187) ? y[row * CS_N2 + threadIdx.x] : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int r = 0; r < 2 * CSR_G; ++r) rows[r][threadIdx.x] = v[r];
    }
    __syncthreads();
    pass_inplace_batched<256, 16, 1, 2 * CSR_G, CS_NT, false, true, false, IdMap, Pad16Map, CSR_STRIDE>(&rows[0][0], threadIdx.x, T256);    // [15][16]
    pass_inplace_batched<256, 16, 16, 2 * CSR_G, CS_NT, false, false, false, Pad16Map, IdMap, CSR_STRIDE>(&rows[0][0], threadIdx.x, T256);
    float2* out = spec + (size_t)cyc * spec_stride;
    for (int i = threadIdx.x; i < CSR_G * CS_N2; i += CS_NT) {
        const int k2 = i / CSR_G, r = i - k2 * CSR_G;
        const int k1 = g0 + r;
        if (k1 > 187) continue;
        const int k = k1 + CS_N1 * k2;                      // bin of the complex transform
        // partner Z[96000-k] sits in the mirror row at column 255-k2 (k1 > 0) or (256-k2)%256 (k1 == 0)
        const int k2m = (k1 == 0) ? ((CS_N2 - k2) & (CS_N2 - 1)) : (CS_N2 - 1 - k2);
        const float2 zk = rows[r][k2];
        const float2 zm = rows[CSR_G + r][k2m];
        const float2 e = cscale(0.5f, cfma_elem(zm, 1.0f, -1.0f, zk));                       // (zk + conj(zm))/2
        const float2 dz = cfma_elem(zm, -1.0f, 1.0f, zk);
            const float2 o = make_float2(0.5f * dz.y, -0.5f * dz.x);       // -i/2 (zk - conj(zm))
        const float2 wo = cmul(o, __ldg(&W192000[k]));
        if (k <= kmax) out[k] = cadd(e, wo);
        const int km = CS_N - k;                            // mirrored output bin, conj(E - W O)
        if (km <= kmax && !(k1 == 0 && k2 > 128)) out[km] = make_float2(e.x - wo.x, -(e.y - wo.y));
    }
}

// ---------------------------------------------------------------------------------------------- F2/F3
struct FineTables {
    float taper[100];          // 0.5*(1+cos(linspace(-pi,0,100))): rises 0 -> 1
    float2 w32[32];            // exp(-2 pi i m / 32)
};
__constant__ FineTables c_fine;

struct FineOut {               // per candidate
    int32_t tt, ff, nsync;
    float sd;
    int32_t snr;
};

// Inverse 3200-point FFT of the tapered band around fb (receiver.py:180-186).
// Band layout after the reference's roll(-150): a[i] = spec[fb + i] for i < 850 (taper on [750,850)),
// spec[fb + i - 3200] for i >= 3050 (taper on [3050,3150)), zero elsewhere.  First pass (R=5, S=1, M=640) reads the
// operands a[p + 640 j] straight from the spectrum: j = 2, 3 are always zero, j = 1 is non-zero only for p < 210 and
// j = 4 only for p >= 490, so the radix-5 butterfly degenerates to b_k = a0 + a1 w^k + a4 conj(w^k), w = e^{+2 pi i/5}.
// Per-pass twiddle tables in TF ([k-1][p] layout): first pass 4 x 640 | (5,5) 4 x 128 | (8,25) 7 x 16.
constexpr int FINE_T5_OFF = 4 * 640, FINE_T8_OFF = FINE_T5_OFF + 4 * 128, FINE_TF_LEN = FINE_T8_OFF + 7 * 16;

// Passes (5,1) and (5,5) fused, one thread per p2 < 128 (four warps): the thread builds the five sparse first-pass
// butterflies p = p2 + 128 j in registers (25 values, same arithmetic as fine_pass1), then runs the five second-pass
// butterflies (p2, q) on them and stores the second-pass output y[q + 25 p2 + 5 k] (stride 25 across lanes: no bank
// conflict).  Against the two separate passes this drops the 3200-element store + reload of the intermediate and 16 of the
// 20 second-pass twiddle loads per p2 -- about 30 % of the kernel's traffic on the shared-memory / L1 pipe, which is what
// bounds it -- and needs no shared-memory input, so the other four warps can score the previous transform meanwhile.
// The spectrum reads of a fused transform come from L2 (several hundred cycles): they are issued one barrier phase early
// (fine_pass12_load, before pass (8,25) of the transform in flight) and consumed after it (fine_pass12_finish).
struct FineIn { float2 a0[5]; float2 ax[4]; };    // ax: the second non-zero operand of butterflies j = 0, 1 (a1) and 3, 4 (a4)

__device__ __forceinline__ void fine_pass12_load(FineIn& in, const float2* __restrict__ spec, int fb, int p2) {
#pragma unroll
    for (int j = 0; j < 5; ++j) in.a0[j] = __ldg(&spec[fb + p2 + 128 * j]);
    in.ax[0] = __ldg(&spec[fb + p2 + 640]);                                  // j = 0: p = p2 < 210 always
    in.ax[1] = (p2 + 128 < 210) ? __ldg(&spec[fb + p2 + 128 + 640]) : make_float2(0.f, 0.f);
    in.ax[2] = (p2 + 384 >= 490) ? __ldg(&spec[fb + p2 + 384 - 640]) : make_float2(0.f, 0.f);
    in.ax[3] = __ldg(&spec[fb + p2 + 512 - 640]);                            // j = 4: p >= 512 always
}

// First-pass output q of sparse butterfly with second operand a1 (at j = 1) / a4 (at j = 4): b_q = a0 + a1 w^q, a0 + a4 conj(w^q)
template <int Q, bool A4> __device__ __forceinline__ float2 fine_b(float2 a0, float2 ax) {
    const float2 w1 = make_float2(0.30901699437494742410f, 0.95105651629515357212f);
    const float2 w2 = make_float2(-0.80901699437494742410f, 0.58778525229247312917f);
    if (Q == 0) return cadd(a0, ax);
    const float2 w = (Q == 1 || Q == 4) ? w1 : w2;
    const bool conj = (Q >= 3) != A4;                     // a1 form: conj for q = 3, 4; a4 form: conj for q = 1, 2
    return cadd(a0, conj ? cmulc(ax, w) : cmul(ax, w));
}

// One column q at a time (the five first-pass outputs q, then second-pass butterfly (p2, q)): same arithmetic as building
// all 25 first-pass outputs first, but ~40 live registers instead of ~90, which is what lets three CTAs share an SM.
template <int Q>
__device__ __forceinline__ void fine_pass12_col(const FineIn& in, const float2 (&ax)[4], float2* dst, int p2,
                                                const float2* __restrict__ TF, const float2 (&w)[8]) {
    float2 a[5];
    a[0] = fine_b<Q, false>(in.a0[0], ax[0]);
    a[1] = (p2 < 82) ? fine_b<Q, false>(in.a0[1], ax[1]) : in.a0[1];
    a[2] = in.a0[2];
    a[3] = (p2 >= 106) ? fine_b<Q, true>(in.a0[3], ax[2]) : in.a0[3];
    a[4] = fine_b<Q, true>(in.a0[4], ax[3]);
    if (Q > 0) {
#pragma unroll
        for (int j = 0; j < 5; ++j) a[j] = cmulc(a[j], __ldg(&TF[(Q - 1) * 640 + p2 + 128 * j]));
    }
    Dft<5, true>::run(a);
    dst[Q + 25 * p2] = a[0];
#pragma unroll
    for (int k = 1; k < 5; ++k) dst[Q + 25 * p2 + 5 * k] = cmulc(a[k], w[k - 1]);
}

// w5[0..3]: the thread's second-pass twiddles w^(5 p2 k), k = 1..4 (held in registers by the producer warps)
__device__ __forceinline__ void fine_pass12_finish(const FineIn& in, float2* dst, int p2, const float2* __restrict__ TF,
                                                   const float* taper, const float2 (&w)[8]) {
    // tapered edge operands (receiver.py:182-183): a1 of p = p2 (>= 110) and p2 + 128; a4 of p2 + 384 and p2 + 512 (< 590)
    float2 ax[4] = {in.ax[0], in.ax[1], in.ax[2], in.ax[3]};
    if (p2 >= 110) ax[0] = cscale(taper[p2 - 110], ax[0]);
    if (p2 < 82) ax[1] = cscale(taper[p2 + 18], ax[1]);
    if (p2 >= 106) ax[2] = cscale(taper[p2 - 106], ax[2]);
    if (p2 < 78) ax[3] = cscale(taper[p2 + 22], ax[3]);
    fine_pass12_col<0>(in, ax, dst, p2, TF, w);
    fine_pass12_col<1>(in, ax, dst, p2, TF, w);
    fine_pass12_col<2>(in, ax, dst, p2, TF, w);
    fine_pass12_col<3>(in, ax, dst, p2, TF, w);
    fine_pass12_col<4>(in, ax, dst, p2, TF, w);
}

__device__ __forceinline__ void fine_pass12(float2* dst, const float2* __restrict__ spec, int fb, int p2,
                                            const float2* __restrict__ TF, const float* taper, const float2 (&w)[8]) {
    FineIn in;
    fine_pass12_load(in, spec, fb, p2);
    fine_pass12_finish(in, dst, p2, TF, taper, w);
}

// Pass (8,25) px -> po by NT threads (a multiple of 16), p-major: thread tid owns p = tid % 16 in every butterfly it runs
// (q = tid / 16, tid / 16 + NT / 16, ...), so its 7 twiddles w^(25 p k) live in registers for the whole kernel (tw8, loaded
// once) -- no twiddle loads in this pass at all.  Loads have stride 25 elements across lanes, stores go to the padded
// operand layout q + 201 p + 25 k (stride 201): both conflict-free.  One barrier at the end.
template <int NT>
__device__ __forceinline__ void fine_pass3(const float2* src, float2* dst, int tid, const float2 (&tw8)[7]) {
    const int p = tid & 15;
#pragma unroll
    for (int r = 0; r < (25 * 16 + NT - 1) / NT; ++r) {
        const int q = (tid >> 4) + (NT / 16) * r;
        if (q < 25) {
            float2 a[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) a[j] = src[q + 25 * p + 400 * j];
            Dft<8, true>::run(a);
            float2* d = dst + q + 201 * p;
            d[0] = a[0];
#pragma unroll
            for (int k = 1; k < 8; ++k) d[25 * k] = cmulc(a[k], tw8[k - 1]);
        }
    }
    __syncthreads();
}

// Full last pass (16,200) of the winner by NT threads: padded operands pb -> natural-order samples in dst.  One barrier at
// the end.
template <int NT>
__device__ __forceinline__ void fine_last_full(const float2* src, float2* dst, int tid) {
#pragma unroll
    for (int t0 = 0; t0 < 200; t0 += NT) {
        const int t = t0 + tid;
        if (t < 200) {
            float2 a[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) a[j] = src[t + 201 * j];
            Dft<16, true>::run(a);
#pragma unroll
            for (int k = 0; k < 16; ++k) dst[t + 200 * k] = a[k];
        }
    }
    __syncthreads();
}

// Last pass (16,200) restricted to the `len` <= 256 consecutive output samples n0 .. n0+len-1 that the Costas scoring
// reads (7 symbols x 32 samples, + 14 for the time scan): z[n] = sum_j x[n%200 + 200 j] * w^(j k), k = n/200, w = e^{+2 pi i/16}.
// A full pass would produce 3200 samples of which the score uses 7 %; only the winning transform gets the full pass.
// One output per thread, evaluated radix-4 style: j = 4a + b, w^(4 a k) = i^(a k), so with r = k mod 4
//   y_b = x_b0 + i^r x_b1 + i^2r x_b2 + i^3r x_b3 = (x_b0 +- x_b2) + i^r (x_b1 +- x_b3)      (signs: - for odd r)
//   z   = y_0 + w^k y_1 + w^2k y_2 + w^3k y_3
// i.e. 16 loads, multiplications by 0/+-1 only inside y_b (exact), and 3 twiddle multiplies instead of 15.
// Executed by the 128 threads of warps 0-3 (two outputs each); no barrier inside.
__device__ __forceinline__ void fine_pass4_window(const float2* x, float2* zwin, int n0, int len, int tid, const float2* w16) {
#pragma unroll
    for (int o = tid; o < 256; o += 128) if (o < len) {
        const int n = n0 + o;
        const int kk = n / 200, q = n - 200 * kk;
        const int r = kk & 3;
        const float sg = (r & 1) ? -1.0f : 1.0f;                                    // x_b0 + sg x_b2,  x_b1 + sg x_b3
        const float2 ir = make_float2(r == 0 ? 1.0f : (r == 2 ? -1.0f : 0.0f), r == 1 ? 1.0f : (r == 3 ? -1.0f : 0.0f));   // i^r
        float2 y[4];
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const float2 x0 = x[q + 201 * b], x1 = x[q + 201 * (4 + b)], x2 = x[q + 201 * (8 + b)], x3 = x[q + 201 * (12 + b)];   // padded operand layout
            const float2 s = caxpy(sg, x2, x0), t = caxpy(sg, x3, x1);
            y[b] = cmac(s, t, ir);
        }
        float2 acc = y[0];
#pragma unroll
        for (int b = 1; b < 4; ++b) acc = cmac(acc, y[b], w16[(b * kk) & 15]);
        zwin[o] = acc;
    }
}

// 32-sample symbol DFTs (receiver.py:195), FOUR windows per warp: lane = 8*g + m serves window g (0..3) and holds its
// samples m, m+8, m+16, m+24.  Since w32^(8t) = (-i)^t, summing those four samples with the bin-t kernel is a 4-point DFT
// (bin t mod 4) times this lane's twiddle tw[t] = exp(-2 pi i t m/32); the 8 partial bins are then summed over the 8 lanes
// of the window with a halving exchange (offsets 4, 2, 1: 14 shuffles), after which lane m holds bin m.
// Returns |bin (lane & 7)| / 3200 of window (lane >> 3)  (numpy's ifft carries the 1/N).
__device__ __forceinline__ float2 shfl_xor2(float2 v, int o) {
    return make_float2(__shfl_xor_sync(0xffffffffu, v.x, o), __shfl_xor_sync(0xffffffffu, v.y, o));
}

__device__ __forceinline__ float dft32x4_mag(const float2* z, int i0, int lane, const float2 (&tw)[8]) {
    const int m = lane & 7;
    float2 v[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) v[a] = z[i0 + m + 8 * a];
    Dft<4, false>::run(v);
    float2 c[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) c[t] = cmul(v[t & 3], tw[t]);
    const bool h4 = lane & 4, h2 = lane & 2, h1 = lane & 1;
    float2 d4[4], d2[2];
#pragma unroll
    for (int j = 0; j < 4; ++j) {                       // lanes with bit 2 clear keep bins 0..3, the others 4..7
        const float2 send = h4 ? c[j] : c[j + 4], keep = h4 ? c[j + 4] : c[j];
        d4[j] = cadd(keep, shfl_xor2(send, 4));
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const float2 send = h2 ? d4[j] : d4[j + 2], keep = h2 ? d4[j + 2] : d4[j];
        d2[j] = cadd(keep, shfl_xor2(send, 2));
    }
    const float2 send = h1 ? d2[0] : d2[1], keep = h1 ? d2[1] : d2[0];
    const float2 s = cadd(keep, shfl_xor2(send, 1));
    return sqrtf(fmaf(s.x, s.x, s.y * s.y)) * (1.0f / 3200.0f);
}

__device__ __forceinline__ int clip_start(int i) { return max(0, min(FINE_N - 32, i)); }

// Weighted middle-Costas sum (receiver.py:198-203) over symbol rows k0 .. k0+3 (rows >= 7 contribute nothing) for a window
// start tb: sum over tones 0..6 of |bin| * (+1 on the Costas tone, -1/6 elsewhere).  Every lane gets the 4-row total.
// `z0` = index in z of the first sample of Costas symbol 0 of the block.
__device__ __forceinline__ float costas_rows4(const float2* z, int z0, int k0, int lane, const float2 (&tw)[8]) {
    const int k = k0 + (lane >> 3), bin = lane & 7;
    const float g = dft32x4_mag(z, z0 + 32 * min(k, 6), lane, tw);
    float c = 0.0f;
    if (k < 7 && bin < 7) c = (bin == ((0x2560413 >> (4 * k)) & 7)) ? g : g * (-1.0f / 6.0f);   // Costas 3,1,4,0,6,5,2 as nibbles (a lane-indexed __constant__ read would serialise)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    return c;
}

constexpr int FINE_SMEM_BYTES = (FINE_N + 2 * FINE_NP) * (int)sizeof(float2) + (79 * 8 + 16 + 100) * (int)sizeof(float) + (32 + 16 + 256) * (int)sizeof(float2);

// Optional phase timing (-DFINE_PROFILE, tools/fine_phase_profile.py): clock64 sums per barrier phase of the frequency scan.
#ifdef FINE_PROFILE
__device__ unsigned long long g_fine_prof[16];
#define FP_T(v) const long long v = clock64()
#define FP_ADD(i, d) do { if (lane == 0) atomicAdd(&g_fine_prof[i], (unsigned long long)(d)); } while (0)
#else
#define FP_T(v)
#define FP_ADD(i, d)
#endif
// One CTA per work item (grid-stride over list[0..*count)).  cand arrays are indexed by the global slot id.
// spec: [B][spec_stride] float2.  Outputs per slot: fo[slot], llr_fine[slot][174], optional sig_grid[slot][79][8].
__global__ void __launch_bounds__(FINE_NT, 2)
k_fine(const float2* __restrict__ spec, int spec_stride, const int32_t* __restrict__ list, const int32_t* __restrict__ count,
       int n_direct, const int32_t* __restrict__ cycle_of, const int16_t* __restrict__ cand_f0,
       const int16_t* __restrict__ cand_h0, const float2* __restrict__ TF, FineOut* __restrict__ fo,
       float* __restrict__ llr_fine, float* __restrict__ sig_grid) {
    extern __shared__ float2 fine_smem[];
    float* G = reinterpret_cast<float*>(fine_smem + FINE_N + 2 * FINE_NP);      // [79][8]
    float* score = G + 79 * 8;                                        // [16]
    float* taper = score + 16;                                        // [100]
    float2* w32 = reinterpret_cast<float2*>(taper + 100);             // [32]  exp(-2 pi i m/32)
    float2* w16 = w32 + 32;                                           // [16]  exp(+2 pi i m/16)
    float2* zwin = w16 + 16;                                          // [256] scoring window of the current transform
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 32) w32[tid] = c_fine.w32[tid];
    if (tid < 16) { const float2 w = c_fine.w32[2 * tid]; w16[tid] = make_float2(w.x, -w.y); }
    if (tid < 100) taper[tid] = c_fine.taper[tid];
    __syncthreads();
    float2 tw[8];                                                     // this lane's DFT32 twiddles, fixed for the kernel
#pragma unroll
    for (int t = 0; t < 8; ++t) tw[t] = w32[(t * (lane & 7)) & 31];
    // the producer warps never run symbol DFTs: their tw[0..3] hold the second-pass twiddles of p2 = tid - 128 instead
    if (warp >= 4) {
#pragma unroll
        for (int k = 1; k < 5; ++k) tw[k - 1] = __ldg(&TF[FINE_T5_OFF + (k - 1) * 128 + (tid - 128)]);
    }
    float2 tw8[7];                                                    // this thread's pass-(8,25) twiddles (p = tid % 16), fixed too
#pragma unroll
    for (int k = 1; k < 8; ++k) tw8[k - 1] = __ldg(&TF[FINE_T8_OFF + (k - 1) * 16 + (tid & 15)]);
    const int n_items = list ? *count : n_direct;
    // the first transform of the CTA's first item; every later item's first transform is built by the producer warps
    // during the final stage of the item before it
    if (warp >= 4 && (int)blockIdx.x < n_items) {
        const int slot = list ? list[blockIdx.x] : (int)blockIdx.x;
        fine_pass12(fine_smem, spec + (size_t)cycle_of[slot] * spec_stride, 50 * cand_f0[slot], tid - 128, TF, taper, tw);
    }
    __syncthreads();
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int slot = list ? list[item] : item;
        const int cyc = cycle_of[slot];
        const int f0 = cand_f0[slot], h0 = cand_h0[slot];
        const float2* sp = spec + (size_t)cyc * spec_stride;
        const int fb0 = 50 * f0;                                   // int(0.5 + 16*fHz), fHz = 3.125*f0
        const int tb0 = (h0 >= 0) ? 8 * h0 : 8 * h0 + 1;           // int(0.5 + 200*tsec) truncates toward zero
        // Three 3200-sample buffers: px = second-pass output of the transform being built, po = last-pass operands of the
        // transform being scored, pb = last-pass operands of the best transform so far.  Per transform there are two
        // barrier phases: (A) all warps run pass (8,25) px -> po; (B) warps 0-3 produce the samples the Costas score reads
        // (windowed last pass) and score them, while warps 4-7 build the NEXT transform's fused passes (5,1)(5,5) from
        // global memory into px.
        float2 *px = fine_smem, *po = fine_smem + FINE_N, *pb = fine_smem + FINE_N + FINE_NP;
        // ---- time scan at ftweak = 0 (receiver.py:147-152): 8 window starts share one inverse FFT.
        //      Middle-Costas windows start at tb0 + tt + 32*(36+k) in [849, 2082] for every reachable h0: never clipped.
        //      px already holds the fused first passes of this item's ftweak = 0 transform.
        FineIn fin;
        FP_T(ts0);
        if (warp >= 4) fine_pass12_load(fin, sp, fb0 - 32, tid - 128);       // operands of the next transform: in flight during pass (8,25)
        fine_pass3<FINE_NT>(px, po, tid, tw8);
        FP_T(ts1);
        if (warp < 4) {
            fine_pass4_window(po, zwin, tb0 - 8 + 1152, 238, tid, w16);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            // warp w scores window starts 2w and 2w+1 (tt = -8 + 2*start)
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int st = 2 * warp + u;
                const float sc = costas_rows4(zwin, 2 * st, 0, lane, tw) + costas_rows4(zwin, 2 * st, 4, lane, tw);
                if (lane == 0) score[st] = sc;
            }
            FP_T(ts2);
            if (warp == 0) { FP_ADD(8, ts1 - ts0); FP_ADD(9, ts2 - ts1); FP_ADD(11, 1); }
        } else {
            fine_pass12_finish(fin, px, tid - 128, TF, taper, tw);        // first frequency tweak, built during the time scan
            FP_T(ts2);
            if (warp == 4) FP_ADD(10, ts2 - ts1);
        }
        __syncthreads();
        int tt = -8;
        float bestf = score[0];
        for (int ti = 1; ti < 8; ++ti) if (score[ti] > bestf) { bestf = score[ti]; tt = -8 + 2 * ti; }   // first maximum
        // ---- frequency scan at the chosen time tweak (receiver.py:154-159).  The ftweak = 0 evaluation is the time-scan
        // score at tt (same baseband, same window starts).  "First maximum in ascending ftweak order" = larger score, or
        // equal score and smaller index.  Warps 0 and 1 score Costas symbols 0..3 and 4..6.
        { float2* t = pb; pb = po; po = t; }                          // best = ftweak 0
        int best_fi = 4;
        for (int e = 0; e < 8; ++e) {
            const int fi = e < 4 ? e : e + 1;
            if (warp >= 4 && e < 7) fine_pass12_load(fin, sp, fb0 + (-32 + 8 * (e + 1 < 4 ? e + 1 : e + 2)), tid - 128);
            FP_T(t0);
            fine_pass3<FINE_NT>(px, po, tid, tw8);
            FP_T(t1);
            if (warp < 4) {
                fine_pass4_window(po, zwin, tb0 + tt + 1152, 224, tid, w16);
                FP_T(tw0);
                asm volatile("bar.sync 1, 128;" ::: "memory");
                if (warp < 2) {
                    const float r = costas_rows4(zwin, 0, 4 * warp, lane, tw);
                    if (lane == 0) score[8 + warp] = r;
                }
                FP_T(t2);
                if (warp == 0) { FP_ADD(0, t1 - t0); FP_ADD(1, t2 - t1); FP_ADD(4, tw0 - t1); FP_ADD(6, 1); }
                if (warp == 3) { FP_ADD(5, t2 - t1); }
            } else if (e < 7) {
                fine_pass12_finish(fin, px, tid - 128, TF, taper, tw);
                FP_T(t2);
                if (warp == 4) { FP_ADD(2, t2 - t1); FP_ADD(7, 1); }
            }
            __syncthreads();
            FP_T(t3);
            if (warp == 0) FP_ADD(3, t3 - t1);
            const float sc = score[8] + score[9];
            if (sc > bestf || (sc == bestf && fi < best_fi)) { bestf = sc; best_fi = fi; float2* t = pb; pb = po; po = t; }
        }
        const int ff = -32 + 8 * best_fi;
        // ---- full last pass of the winner, then the final grid (receiver.py:161) by the consumer warps (four symbol rows
        //      per warp and call) and the Costas count + LLRs by warp 0, while the producer warps already build the first
        //      transform of this CTA's next item into px (unused during this stage)
        FP_T(tf0);
        fine_last_full<FINE_NT>(pb, po, tid);
        FP_T(tf1);
        if (warp < 4) {
            const float2* z = po;
            for (int j0 = 4 * warp; j0 < 79; j0 += 16) {
                const int j = j0 + (lane >> 3);
                const float g = dft32x4_mag(z, clip_start(tb0 + tt + 32 * min(j, 78)), lane, tw);
                if (j < 79) G[j * 8 + (lane & 7)] = g;
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (sig_grid) for (int i = tid; i < 79 * 8; i += 128) sig_grid[(size_t)slot * 632 + i] = G[i];
            if (tid < 32) {
                int hit = 0;
                if (lane < 21) {
                    const int blk = lane / 7, k = lane - 7 * blk;
                    const int row = (blk == 0) ? k : (blk == 1 ? 36 + k : 72 + k);
                    int am = 0;
                    float mv = G[row * 8];
                    for (int t = 1; t < 8; ++t) if (G[row * 8 + t] > mv) { mv = G[row * 8 + t]; am = t; }
                    hit = (am == ((0x2560413 >> (4 * k)) & 7)) ? 1 : 0;
                }
                const int nsync = __reduce_add_sync(0xffffffffu, hit);
                float p[2][8];
                if (lane < 29) {
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const int sym = lane + (q ? 43 : 7);                  // PAYLOAD_SYMB_IDXS = 7..35, 43..71
#pragma unroll
                        for (int t = 0; t < 8; ++t) p[q][t] = 20.0f * log10f(G[sym * 8 + t]);
                    }
                }
                float sd; int snr;
                llr_from_payload_warp(p, lane, llr_fine + (size_t)slot * 174, sd, snr);
                if (lane == 0) {
                    FineOut o; o.tt = tt; o.ff = ff; o.nsync = nsync; o.sd = sd; o.snr = snr;
                    fo[slot] = o;
                }
            }
        } else {
            const int nitem = item + gridDim.x;
            if (nitem < n_items) {
                const int nslot = list ? list[nitem] : nitem;
                fine_pass12(px, spec + (size_t)cycle_of[nslot] * spec_stride, 50 * cand_f0[nslot], tid - 128, TF, taper, tw);
            }
            FP_T(tf2);
            if (warp == 4) FP_ADD(14, tf2 - tf1);
        }
        FP_T(tf3);
        if (warp == 0) { FP_ADD(12, tf1 - tf0); FP_ADD(13, tf3 - tf1); }
        if (warp == 3) { FP_ADD(15, tf3 - tf1); }
        __syncthreads();
    }
}

}  // namespace ft8
