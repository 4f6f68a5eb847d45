// fft.cuh -- shared-memory Stockham FFT building blocks (radix 2/3/4/5/8/15/16), fp32 complex, packed f32x2 arithmetic.
//
// Every transform on the FT8 receive path has a length with factors 2, 3 and 5 only
// (3840 = 2*1920 real, 192000 = 2*(375*256) real, 3200, 32; SURVEY.md H9), so the library
// carries its own mixed-radix kernels instead of calling cuFFT: the transforms are fused with
// windowing / untangling / log-magnitude (S1), band extraction + taper (F3) and the per-symbol
// DFTs that follow them, which a library call cannot do.
//
// Formulation: decimation-in-frequency Stockham autosort.  A transform of length N runs as a
// sequence of passes (R, S) with S = product of the radices already done; pass (R,S) maps
//     y[q + S*(R*p + k)] = w_{N/S}^{p*k} * sum_j x[q + S*(p + M*j)] * w_R^{j*k},   M = N/(S*R)
// for p < M, q < S.  Natural order in, natural order out, no bit reversal.  Twiddles come from a
// table W[j] = exp(-2*pi*i*j/N) computed in double on the host (w_{N/S}^{p*k} = W[p*k*S]).
#pragma once
#include <cuda_runtime.h>

namespace ft8 {

// ---- complex helpers on Blackwell packed fp32x2 (FFMA2 / FADD2 / FMUL2, one instruction per complex number; ptxas folds
// operand swaps, scalar broadcasts and per-half sign changes into modifiers such as R.F32x2.LO_HI.NP / R.F32, so a
// complex multiply is 2 instructions and a multiply by +-i inside an add is free).  Each half rounds like the scalar
// instruction (products rounded once, fma exactly where the formulas below have fmaf).
// Why packed, measured on B200 (tools/micro/ffma2_bench.cu, tools/variant_bench.py): FFMA2 sustains the FFMA flop rate
// with half the issue slots (72 Tflop/s either way); against plain FFMA / FADD / FMUL the packed build is 2 % faster on
// the whole step (k_spectrogram 8.15 -> 7.91 ms, k_fine 54.0 -> 52.0 ms), records bit-identical.
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk(float lo, float hi) { u64 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ u64 P(float2 a) { return pk(a.x, a.y); }
__device__ __forceinline__ float2 U(u64 v) { float2 r; asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v)); return r; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 bc(float s) { return pk(s, s); }                      // scalar broadcast
__device__ __forceinline__ u64 sw(float2 a) { return pk(a.y, a.x); }                // swapped halves
// (fmaf(a.x, b.x, -a.y*b.y), fmaf(a.x, b.y, a.y*b.x))
__device__ __forceinline__ float2 cmul(float2 a, float2 b) { return U(fma2(bc(a.x), P(b), mul2(pk(b.y, -b.x), bc(-a.y)))); }
// a * conj(b) = (fmaf(a.x, b.x, a.y*b.y), fmaf(a.y, b.x, -a.x*b.y))
__device__ __forceinline__ float2 cmulc(float2 a, float2 b) { return U(fma2(P(a), bc(b.x), mul2(pk(a.y, -a.x), bc(b.y)))); }
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return U(add2(P(a), P(b))); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return U(sub2(P(a), P(b))); }
// s*a + c per component, s*a, a*b per component, a*(sx,sy) + c per component
__device__ __forceinline__ float2 caxpy(float s, float2 a, float2 c) { return U(fma2(bc(s), P(a), P(c))); }
__device__ __forceinline__ float2 cscale(float s, float2 a) { return U(mul2(bc(s), P(a))); }
__device__ __forceinline__ float2 cmul_elem(float2 a, float2 b) { return U(mul2(P(a), P(b))); }
__device__ __forceinline__ float2 cfma_elem(float2 a, float sx, float sy, float2 c) { return U(fma2(P(a), pk(sx, sy), P(c))); }
// d + s*rot90<INV>(x) and d - s*rot90<INV>(x)   (rot90 = times +i for INV, -i otherwise; s = 1: a plain add/sub)
template <bool INV> __device__ __forceinline__ float2 addrot(float2 d, float2 x, float s = 1.0f) {
    return U(fma2(sw(x), INV ? pk(-s, s) : pk(s, -s), P(d)));
}
template <bool INV> __device__ __forceinline__ float2 subrot(float2 d, float2 x, float s = 1.0f) {
    return U(fma2(sw(x), INV ? pk(s, -s) : pk(-s, s), P(d)));
}
// acc + v*w with acc.x = fmaf(v.x, w.x, fmaf(-v.y, w.y, acc.x)), acc.y = fmaf(v.x, w.y, fmaf(v.y, w.x, acc.y))
__device__ __forceinline__ float2 cmac(float2 acc, float2 v, float2 w) {
    return U(fma2(bc(v.x), P(w), fma2(pk(w.y, -w.x), bc(-v.y), P(acc))));
}
// multiply by -i (forward) or +i (inverse)
template <bool INV> __device__ __forceinline__ float2 rot90(float2 a) {
    return INV ? make_float2(-a.y, a.x) : make_float2(a.y, -a.x);
}

template <int R, bool INV, bool ROT2 = false> struct Dft;

template <bool INV> struct Dft<2, INV, false> {
    static __device__ __forceinline__ void run(float2* a) {
        float2 t = a[0];
        a[0] = cadd(t, a[1]);
        a[1] = csub(t, a[1]);
    }
};

template <bool INV> struct Dft<3, INV, false> {
    static __device__ __forceinline__ void run(float2* a) {
        const float s = 0.86602540378443864676f;
        const float2 t = cadd(a[1], a[2]);
        const float2 u = csub(a[1], a[2]);               // a1, a2 = m +- s*rot90(u)
        const float2 m = caxpy(-0.5f, t, a[0]);
        a[0] = cadd(a[0], t);
        a[1] = addrot<INV>(m, u, s);
        a[2] = subrot<INV>(m, u, s);
    }
};

// ROT2: a[2] is still to be multiplied by -/+ i (folded into the first add/sub)
template <bool INV, bool ROT2> struct Dft<4, INV, ROT2> {
    static __device__ __forceinline__ void run(float2* a) {
        const float2 s02 = ROT2 ? addrot<INV>(a[0], a[2]) : cadd(a[0], a[2]);
        const float2 d02 = ROT2 ? subrot<INV>(a[0], a[2]) : csub(a[0], a[2]);
        const float2 s13 = cadd(a[1], a[3]), u = csub(a[1], a[3]);
        a[0] = cadd(s02, s13);
        a[2] = csub(s02, s13);
        a[1] = addrot<INV>(d02, u);
        a[3] = subrot<INV>(d02, u);
    }
};

template <bool INV> struct Dft<5, INV, false> {
    static __device__ __forceinline__ void run(float2* a) {
        const float c1 = 0.30901699437494742410f, c2 = -0.80901699437494742410f;
        const float s1 = 0.95105651629515357212f, s2 = 0.58778525229247312917f;
        const float2 t1 = cadd(a[1], a[4]), t2 = cadd(a[2], a[3]);
        const float2 t3 = csub(a[1], a[4]), t4 = csub(a[2], a[3]);
        const float2 m1 = caxpy(c1, t1, caxpy(c2, t2, a[0]));
        const float2 m2 = caxpy(c2, t1, caxpy(c1, t2, a[0]));
        const float2 u1 = caxpy(s1, t3, cscale(s2, t4));            // n1 = rot90(u1), n2 = rot90(u2)
        const float2 u2 = caxpy(s2, t3, cscale(-s1, t4));
        a[0] = cadd(a[0], cadd(t1, t2));
        a[1] = addrot<INV>(m1, u1);
        a[4] = subrot<INV>(m1, u1);
        a[2] = addrot<INV>(m2, u2);
        a[3] = subrot<INV>(m2, u2);
    }
};

// 8 = 2 x 4 in registers: j = 4*j1 + j2, k = k1 + 2*k2
template <bool INV> struct Dft<8, INV, false> {
    static __device__ __forceinline__ void run(float2* a) {
        const float h = 0.70710678118654752440f;
        float2 c[2][4];
#pragma unroll
        for (int j2 = 0; j2 < 4; ++j2) {
            c[0][j2] = cadd(a[j2], a[4 + j2]);
            c[1][j2] = csub(a[j2], a[4 + j2]);
        }
        // twiddle w8^(j2*k1) on the k1 = 1 row; c[1][2] (times -/+ i) is rotated inside the radix-4 step
        {
            float2 v = c[1][1];   // * w8^1 = (1 -/+ i)/sqrt2 :  INV (h(vx-vy), h(vx+vy)),  fwd (h(vx+vy), h(vy-vx))
            c[1][1] = cscale(h, addrot<INV>(v, v));
            v = c[1][3];          // * w8^3 = (-1 -/+ i)/sqrt2 : INV (-h(vx+vy), h(vx-vy)), fwd (h(vy-vx), -h(vx+vy))
            c[1][3] = cscale(-h, subrot<INV>(v, v));
        }
        Dft<4, INV, false>::run(c[0]);
        Dft<4, INV, true>::run(c[1]);
#pragma unroll
        for (int k2 = 0; k2 < 4; ++k2) {
            a[2 * k2] = c[0][k2];
            a[2 * k2 + 1] = c[1][k2];
        }
    }
};

// 16 = 4 x 4 in registers: j = 4*j1 + j2, k = k1 + 4*k2
template <bool INV> struct Dft<16, INV, false> {
    static __device__ __forceinline__ void run(float2* a) {
        const float c1 = 0.92387953251128675613f, s1 = 0.38268343236508977173f, h = 0.70710678118654752440f;
        float2 c[4][4];   // c[k1][j2]
#pragma unroll
        for (int j2 = 0; j2 < 4; ++j2) {
            float2 t[4] = {a[j2], a[4 + j2], a[8 + j2], a[12 + j2]};
            Dft<4, INV, false>::run(t);
#pragma unroll
            for (int k1 = 0; k1 < 4; ++k1) c[k1][j2] = t[k1];
        }
        // twiddles w16^(j2*k1), k1,j2 in 1..3 : exponents 1,2,3 / 2,4,6 / 3,6,9  (w16^4 = -/+ i is folded into the radix-4 step)
        const float2 w1 = make_float2(c1, -s1), w2 = make_float2(h, -h), w3 = make_float2(s1, -c1);
        const float2 w6 = make_float2(-h, -h), w9 = make_float2(-c1, s1);
#define FT8_TW(v, w) v = INV ? cmulc(v, w) : cmul(v, w)
        FT8_TW(c[1][1], w1); FT8_TW(c[1][2], w2); FT8_TW(c[1][3], w3);
        FT8_TW(c[2][1], w2); FT8_TW(c[2][3], w6);
        FT8_TW(c[3][1], w3); FT8_TW(c[3][2], w6); FT8_TW(c[3][3], w9);
#undef FT8_TW
        Dft<4, INV, false>::run(c[0]);
        Dft<4, INV, false>::run(c[1]);
        Dft<4, INV, true>::run(c[2]);
        Dft<4, INV, false>::run(c[3]);
#pragma unroll
        for (int k1 = 0; k1 < 4; ++k1) {
#pragma unroll
            for (int k2 = 0; k2 < 4; ++k2) a[k1 + 4 * k2] = c[k1][k2];
        }
    }
};

// 15 = 3 x 5 in registers: j = 5*j1 + j2, k = k1 + 3*k2;  w15^(jk) = w3^(j1 k1) * w15^(j2 k1) * w5^(j2 k2)
template <bool INV> struct Dft<15, INV, false> {
    static __device__ __forceinline__ void run(float2* a) {
        float2 c[3][5];   // c[k1][j2]
#pragma unroll
        for (int j2 = 0; j2 < 5; ++j2) {
            float2 t[3] = {a[j2], a[5 + j2], a[10 + j2]};
            Dft<3, INV>::run(t);
#pragma unroll
            for (int k1 = 0; k1 < 3; ++k1) c[k1][j2] = t[k1];
        }
#define FT8_TW15(v, wr, wi) v = INV ? cmulc(v, make_float2(wr, wi)) : cmul(v, make_float2(wr, wi))
        FT8_TW15(c[1][1], 0.91354545764260087f, -0.40673664307580015f);
        FT8_TW15(c[1][2], 0.66913060635885824f, -0.74314482547739413f);
        FT8_TW15(c[1][3], 0.30901699437494745f, -0.95105651629515353f);
        FT8_TW15(c[1][4], -0.10452846326765333f, -0.9945218953682734f);
        FT8_TW15(c[2][1], 0.66913060635885824f, -0.74314482547739413f);
        FT8_TW15(c[2][2], -0.10452846326765333f, -0.9945218953682734f);
        FT8_TW15(c[2][3], -0.80901699437494734f, -0.58778525229247325f);
        FT8_TW15(c[2][4], -0.97814760073380569f, 0.20791169081775907f);
#undef FT8_TW15
#pragma unroll
        for (int k1 = 0; k1 < 3; ++k1) {
            Dft<5, INV>::run(c[k1]);
#pragma unroll
            for (int k2 = 0; k2 < 5; ++k2) a[k1 + 3 * k2] = c[k1][k2];
        }
    }
};

// Index maps for shared-memory buffers: identity, or one padding element after every 16 (turns the stride-16 stores of a
// radix-16 first pass, which would all hit one 8-byte bank, into stride 17).
struct IdMap { static __device__ __forceinline__ int at(int i) { return i; } };
struct Pad16Map { static __device__ __forceinline__ int at(int i) { return i + (i >> 4); } };

// One Stockham pass for butterfly t (0 <= t < N/R).  x, y may be any addressable memory.
// PM selects how t maps to (p, q): false -> p = t / S, q = t % S (consecutive threads read consecutive elements);
// true -> q = t / M, p = t % M: consecutive threads take consecutive p, so loads have stride S and stores stride R*S
// elements -- conflict-free in shared memory when both are odd -- and the [k-1][p] twiddle reads are fully coalesced.
template <int N, int R, int S, bool PM = false> struct Pass {
    static constexpr int M = N / (S * R);
    static __device__ __forceinline__ void decode(int t, int& p, int& q) {
        if (PM) { q = t / M; p = t - q * M; } else { p = t / S; q = t - p * S; }
    }
    template <class MapIn = IdMap>
    static __device__ __forceinline__ void load(const float2* x, int t, float2* a) {
        int p, q;
        decode(t, p, q);
#pragma unroll
        for (int j = 0; j < R; ++j) a[j] = x[MapIn::at(q + S * (p + M * j))];
    }
    // TT = false: W is the plain length-N table, twiddle w_{N/S}^{pk} = W[p*k*S] (a gather whose stride grows with k: up
    // to one 32-byte sector per lane).  TT = true: W is this pass's own table laid out [k-1][p] (pass_table() on the host,
    // same values), so the lanes of a warp read consecutive entries -- the twiddle loads of a pass then cost 2-8 sectors
    // per request instead of up to 32 on the L1/shared-memory data path that bounds the FFT kernels.
    template <bool INV, bool TT = false, class MapOut = IdMap>
    static __device__ __forceinline__ void compute_store(float2* y, int t, float2* a, const float2* __restrict__ W) {
        int p, q;
        decode(t, p, q);
        Dft<R, INV>::run(a);
        y[MapOut::at(q + S * (R * p))] = a[0];
#pragma unroll
        for (int k = 1; k < R; ++k) {
            float2 v = a[k];
            if (M > 1) {
                float2 w = __ldg(TT ? &W[(k - 1) * M + p] : &W[p * k * S]);
                v = INV ? cmulc(v, w) : cmul(v, w);
            }
            y[MapOut::at(q + S * (R * p + k))] = v;
        }
    }
};

// In-place pass over a shared-memory buffer by a group of NT threads (lt = thread index in the group):
// all operands are read into registers, the group synchronises (sync functor), then results are written.
template <int N, int R, int S, int NT, bool INV, class Sync, bool TT = false>
__device__ __forceinline__ void pass_inplace(float2* buf, int lt, const float2* __restrict__ W, Sync sync) {
    constexpr int NBF = N / R;
    constexpr int PER = (NBF + NT - 1) / NT;
    float2 a[PER][R];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        int t = lt + i * NT;
        if (t < NBF) Pass<N, R, S>::load(buf, t, a[i]);
    }
    sync();
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        int t = lt + i * NT;
        if (t < NBF) Pass<N, R, S>::template compute_store<INV, TT>(buf, t, a[i], W);
    }
    sync();
}

struct CtaSync {
    __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

// Complete in-place transforms for the sizes on the path (NT threads cooperate, CTA-wide barriers).
template <int NT, bool INV> __device__ __forceinline__ void fft1920(float2* buf, int lt, const float2* __restrict__ W) {
    pass_inplace<1920, 15, 1, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<1920, 8, 15, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<1920, 16, 120, NT, INV>(buf, lt, W, CtaSync());
}
template <int NT, bool INV> __device__ __forceinline__ void fft3200(float2* buf, int lt, const float2* __restrict__ W) {
    pass_inplace<3200, 5, 1, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<3200, 5, 5, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<3200, 8, 25, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<3200, 16, 200, NT, INV>(buf, lt, W, CtaSync());
}
template <int NT, bool INV> __device__ __forceinline__ void fft375(float2* buf, int lt, const float2* __restrict__ W) {
    pass_inplace<375, 3, 1, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<375, 5, 3, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<375, 5, 15, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<375, 5, 75, NT, INV>(buf, lt, W, CtaSync());
}
template <int NT, bool INV> __device__ __forceinline__ void fft256(float2* buf, int lt, const float2* __restrict__ W) {
    pass_inplace<256, 16, 1, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<256, 16, 16, NT, INV>(buf, lt, W, CtaSync());
}
template <int NT, bool INV> __device__ __forceinline__ void fft32(float2* buf, int lt, const float2* __restrict__ W) {
    pass_inplace<32, 8, 1, NT, INV>(buf, lt, W, CtaSync());
    pass_inplace<32, 4, 8, NT, INV>(buf, lt, W, CtaSync());
}

// Batched variant: NB independent transforms of length N stored back to back in `buf`.
template <int N, int R, int S, int NB, int NT, bool INV, bool TT = false, bool PM = false, class MapIn = IdMap, class MapOut = IdMap,
          int STRIDE = N>
__device__ __forceinline__ void pass_inplace_batched(float2* buf, int tid, const float2* __restrict__ W) {
    constexpr int NBF = N / R;
    constexpr int ITEMS = NBF * NB;
    constexpr int PER = (ITEMS + NT - 1) / NT;
    float2 a[PER][R];
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int it = tid + i * NT;
        if (it < ITEMS) {
            const int b = it / NBF, t = it - b * NBF;
            Pass<N, R, S, PM>::template load<MapIn>(buf + b * STRIDE, t, a[i]);
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int it = tid + i * NT;
        if (it < ITEMS) {
            const int b = it / NBF, t = it - b * NBF;
            Pass<N, R, S, PM>::template compute_store<INV, TT, MapOut>(buf + b * STRIDE, t, a[i], W);
        }
    }
    __syncthreads();
}

}  // namespace ft8
