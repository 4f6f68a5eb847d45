// osd.cuh -- ordered-statistics decoding (order 0 + single/double flips), one warp per codeword.
//
// Restates osd_012 (decoders.py:223-272; SURVEY.md A7).  The reference runs Gauss-Jordan on a 91x174 uint8 matrix
// G0 = [I | A^T] with row/column permutation lists and then multiplies trial vectors by G[:, :91].  Everything it
// produces is a function of the most-reliable basis (the first 91 linearly independent columns in reliability order) and
// of the order in which its members were found -- not of which row each pivot used -- so the elimination here is free to
// pick rows, and it only ever stores the 83 PARITY columns (round 2; the first version carried all 174):
//   * columns are bit-packed over the 91 rows (3 x u32); parity column j lives in lane j%32, register slot j/32;
//   * columns are visited in reliability order (|llr| descending, ties by ascending index, NaN last -- numpy's
//     argsort(-|llr|) made stable, SURVEY H6);
//   * a systematic column c whose row c is still free is a unit vector: it joins the basis on row c and nothing has to be
//     eliminated (no matrix work at all);
//   * a parity column with a 1 in a free row p joins the basis on row p: every other stored column with a 1 in row p gets
//     the pivot column (row p cleared) XORed in.  The pivot column itself would become the unit vector e_p and carries no
//     information any more, so its slot is left untouched and from then on holds M[:, p], the image of the systematic
//     column p under the accumulated row operations (the in-place inversion trick); `own` maps row p -> that slot;
//   * a systematic column c whose row is taken is that stored image: if it has a 1 in a free row p' it joins the basis on
//     p' (same update) and its slot becomes the image of column p', else it is dependent;
//   * when a parity pivot can choose its row it prefers rows whose systematic column sits late in the reliability order
//     (position >= 96, where the search has usually ended): that column is then never visited as a stored image, which
//     cuts the eliminations per call from ~60 to ~43 (noise-like llr; tools/osd_model.py is the Python model of this scheme, checked
//     against the oracle trial word by trial word).
// At the end every basis slot holds the image of one NON-basis systematic column c'; the order-0 word is
//   bit c  = hard decision of c                      for basis systematic columns,
//   bit c' = parity(image(c') & u), u[row of pivot k] = hard decision of pivot k's column,
// and flipping pivot k adds bit (row of k) of every image, plus the unit bit of k's own column when it is systematic.
// CRC-14 is linear, so each of the 1+S vectors carries its 14-bit syndrome and a trial's CRC test is an XOR; the 91-bit
// word of a trial is only assembled when that XOR is zero.
// The work splits by what it depends on.  osd_basis (the order, the basis, the images and the flip syndromes) reads only
// |llr|; osd_eval (u, the order-0 word and its syndrome, the trials) is the only part that reads the hard decisions.  Calls
// whose inputs differ only in signs share one osd_basis (the AP attempts RR73, 73 and RRR, passes.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "codec.cuh"

namespace ft8 {

struct OsdTables {
    uint32_t col[174][3];      // column c of G0 over the 91 rows, LSB-first
};
__constant__ OsdTables c_osd;

constexpr int OSD_MAX_FLIPS = 91;

struct OsdWarpScratch {
    uint32_t order[176];             // sorted position -> entry (32-bit: no sub-word extraction in the visit loop)
    uint8_t piv_row[96];             // pivot k -> row
    uint8_t piv_col[96];             // pivot k -> original column (>= 91: a parity column)
    uint8_t pcol[96];                // parity rank (position among the parity columns in reliability order) -> column
    uint16_t syn[OSD_MAX_FLIPS];     // CRC syndrome of the vector that flip i adds
    uint16_t ssyn[96];               // CRC syndrome of the systematic column whose image slot j holds (0: not a basis slot)
    uint32_t colw[3 * 97];           // the stored columns word-major [3][OSD_W_PITCH] (odd pitch: the three words of a slot
                                     // sit in different banks)
};
constexpr int OSD_W_PITCH = 97;

// CTA-shared copies of the constant tables the lanes index differently (a lane-indexed read of __constant__ memory is
// replayed once per distinct address): generator columns word-major [3][176], CRC syndrome of each codeword bit.
constexpr int OSD_COL_PITCH = 176;
struct OsdCtaTables { uint32_t col[3 * OSD_COL_PITCH]; uint16_t syn[96]; };
__device__ __forceinline__ void load_osd_tables(OsdCtaTables& t) {
    for (int i = threadIdx.x; i < 174; i += blockDim.x) {
        t.col[i] = c_osd.col[i][0]; t.col[OSD_COL_PITCH + i] = c_osd.col[i][1]; t.col[2 * OSD_COL_PITCH + i] = c_osd.col[i][2];
    }
    for (int i = threadIdx.x; i < 96; i += blockDim.x) t.syn[i] = (i < 91) ? c_codec.crc_syn[i] : (uint16_t)0;
}

// a[w] for a warp-uniform w in 0..2 without branches (the ternary form compiles to a BSSY / BRA / BSYNC diamond)
__device__ __forceinline__ uint32_t sel3(int w, uint32_t a0, uint32_t a1, uint32_t a2) {
    uint32_t r;
    asm("{\n .reg .pred p0, p1;\n setp.eq.s32 p0, %1, 0;\n setp.eq.s32 p1, %1, 1;\n selp.b32 %0, %3, %4, p1;\n selp.b32 %0, %2, %0, p0;\n}"
        : "=&r"(r) : "r"(w), "r"(a0), "r"(a1), "r"(a2));
    return r;
}
// One elimination step on a lane's three stored columns: slot k gets (x0, x1, x2) XORed in when its word `T` has the pivot
// bit and it is not the pivot's own slot (j == 32 k + lane); the own slot records the pivot row instead.  Written in PTX so
// that the XORs stay predicated (the C form becomes nine SELs and nine LOP3s).
#define OSD_ELIM(T0, T1, T2)                                                                                              \
    asm("{\n .reg .pred q0, q1, q2, n0, n1, n2;\n .reg .b32 t0, t1, t2, l1, l2;\n"                                      \
        " add.s32 l1, %16, 32;\n add.s32 l2, %16, 64;\n"                                                                  \
        " setp.eq.s32 n0, %15, %16;\n setp.eq.s32 n1, %15, l1;\n setp.eq.s32 n2, %15, l2;\n"                              \
        " and.b32 t0, %18, %12;\n and.b32 t1, %19, %12;\n and.b32 t2, %20, %12;\n"                                        \
        " setp.ne.and.b32 q0, t0, 0, !n0;\n setp.ne.and.b32 q1, t1, 0, !n1;\n setp.ne.and.b32 q2, t2, 0, !n2;\n"          \
        " @q0 xor.b32 %0, %0, %13;\n @q0 xor.b32 %1, %1, %14;\n @q0 xor.b32 %2, %2, %21;\n"                               \
        " @q1 xor.b32 %3, %3, %13;\n @q1 xor.b32 %4, %4, %14;\n @q1 xor.b32 %5, %5, %21;\n"                               \
        " @q2 xor.b32 %6, %6, %13;\n @q2 xor.b32 %7, %7, %14;\n @q2 xor.b32 %8, %8, %21;\n"                               \
        " @n0 mov.b32 %9, %17;\n @n1 mov.b32 %10, %17;\n @n2 mov.b32 %11, %17;\n}"                                        \
        : "+r"(c0[0]), "+r"(c1[0]), "+r"(c2[0]), "+r"(c0[1]), "+r"(c1[1]), "+r"(c2[1]), "+r"(c0[2]), "+r"(c1[2]), "+r"(c2[2]), \
          "+r"(ownrow[0]), "+r"(ownrow[1]), "+r"(ownrow[2])                                                               \
        : "r"(pb), "r"(x0), "r"(x1), "r"(j), "r"(lane), "r"(p), "r"(T0), "r"(T1), "r"(T2), "r"(x2))


// The same step when the pivot's slot is known at compile time (a parity column of rank j lives in slot j/32, and parity
// columns are visited in rank order, so the visit loop runs through the three slots one after the other): only the own
// slot A needs the "not my own lane" test, and no slot has to be selected at run time.
#define OSD_ELIM_S(A, B, D, TA, TB, TD)                                                                                   \
    asm("{\n .reg .pred q0, q1, q2, n0;\n .reg .b32 t0, t1, t2;\n"                                                        \
        " setp.eq.s32 n0, %14, %15;\n"                                                                                     \
        " and.b32 t0, %17, %10;\n and.b32 t1, %18, %10;\n and.b32 t2, %19, %10;\n"                                        \
        " setp.ne.and.b32 q0, t0, 0, !n0;\n setp.ne.b32 q1, t1, 0;\n setp.ne.b32 q2, t2, 0;\n"                            \
        " @q0 xor.b32 %0, %0, %11;\n @q0 xor.b32 %1, %1, %12;\n @q0 xor.b32 %2, %2, %13;\n"                               \
        " @q1 xor.b32 %3, %3, %11;\n @q1 xor.b32 %4, %4, %12;\n @q1 xor.b32 %5, %5, %13;\n"                               \
        " @q2 xor.b32 %6, %6, %11;\n @q2 xor.b32 %7, %7, %12;\n @q2 xor.b32 %8, %8, %13;\n"                               \
        " @n0 mov.b32 %9, %16;\n}"                                                                                         \
        : "+r"(c0[A]), "+r"(c1[A]), "+r"(c2[A]), "+r"(c0[B]), "+r"(c1[B]), "+r"(c2[B]), "+r"(c0[D]), "+r"(c1[D]), "+r"(c2[D]), \
          "+r"(ownrow[A])                                                                                                 \
        : "r"(pb), "r"(x0), "r"(x1), "r"(x2), "r"(jl), "r"(lane), "r"(p), "r"(TA), "r"(TB), "r"(TD))

// What osd_basis leaves in registers for osd_eval: the lane's three stored columns and the row whose image each slot holds.
struct OsdBasis {
    uint32_t c0[3], c1[3], c2[3];
    uint32_t ownrow[3];               // row (= systematic column) whose image the slot holds, 255: not a basis slot
};

// Steps 1-4 without the hard decisions: reliability order, basis, images, and the syndromes of the S flip vectors
// (s.piv_row, s.piv_col, s.syn, s.ssyn, s.colw; ob).  llr: 174 floats in shared or global memory; only |llr| is read.
__device__ __forceinline__ void osd_basis(OsdWarpScratch& s, const OsdCtaTables& g, const float* llr, int lane, int S, OsdBasis& ob) {
    constexpr uint32_t FULL = 0xffffffffu;
    // ---- 1. reliability order.  Fast path: bitonic sort of 256 32-bit keys (8 per lane, slot e = 32*r + lane), descending,
    //      key = code(|llr|) << 8 | (255 - index) with a monotone 24-bit code (zero, or 5 exponent bits for [2^-26, 2^5)
    //      and the top 19 mantissa bits); padding slots are 0.  The order by (code, index) IS the order by (|llr|, index)
    //      unless two different |llr| share a code, which shows up as an adjacent pair with equal codes and different
    //      values; then, and for values outside the code's range (NaN, inf, >= 32, tiny), the exact order is found by
    //      counting (compact, ~4x slower, a few % of the calls).  One compare-exchange is a SHFL and a min/max.
    uint32_t key[8];
    bool bad = false;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int i = 32 * r + lane;
        uint32_t k = 0u;
        if (i < 174) {
            const uint32_t u = __float_as_uint(llr[i]) & 0x7FFFFFFFu;
            const uint32_t e = u >> 23;
            uint32_t code = 0u;
            if (u != 0u) {
                if (e < 101u || e > 131u) bad = true;
                code = ((e - 100u) << 19) | ((u >> 4) & 0x7FFFFu);
            }
            k = (code << 8) | (uint32_t)(255 - i);
        }
        key[r] = k;
    }
    bad = __any_sync(FULL, bad);
    if (!bad) {
#pragma unroll
        for (int k = 2; k <= 256; k <<= 1) {
#pragma unroll
            for (int j = k >> 1; j > 0; j >>= 1) {
                if (j >= 32) {                                   // partner slot lives in the same lane
                    const int jr = j >> 5;
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        if ((r & jr) == 0) {
                            const bool desc = ((32 * r) & k) == 0;   // lane bits do not matter for k >= 64
                            const uint32_t x = key[r], y = key[r | jr];
                            key[r] = desc ? max(x, y) : min(x, y);
                            key[r | jr] = desc ? min(x, y) : max(x, y);
                        }
                    }
                } else {                                         // partner slot is in lane ^ j, same register
                    const bool lower = (lane & j) == 0;
#pragma unroll
                    for (int r = 0; r < 8; ++r) {
                        const bool desc = ((32 * r + lane) & k) == 0;
                        const uint32_t x = key[r];
                        const uint32_t y = __shfl_xor_sync(FULL, x, j);
                        key[r] = (lower == desc) ? max(x, y) : min(x, y);
                    }
                }
            }
        }
        // adjacent sorted slots with equal codes must hold equal values
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            uint32_t nb = __shfl_sync(FULL, key[r], (lane + 1) & 31);
            const uint32_t nx = __shfl_sync(FULL, key[r + 1], 0);
            if (lane == 31) nb = nx;
            if (nb != 0u && ((key[r] ^ nb) >> 8) == 0u) {
                const uint32_t ua = __float_as_uint(llr[255 - (key[r] & 0xFFu)]) & 0x7FFFFFFFu;
                const uint32_t ub = __float_as_uint(llr[255 - (nb & 0xFFu)]) & 0x7FFFFFFFu;
                if (ua != ub) bad = true;
            }
        }
        bad = __any_sync(FULL, bad);
    }
    // ---- 2. publish the order: entry = column for a systematic column, 128 + parity rank for a parity
    //      column (its rank among the parity columns in reliability order = the slot it will live in); rows whose
    //      systematic column comes late (position >= 96)
    uint32_t L0 = 0, L1 = 0, L2 = 0;
    if (!bad) {
        int pbase = 0;
#pragma unroll
        for (int r = 0; r < 6; ++r) {
            const int sp = lane + 32 * r;
            const int c = 255 - (int)(key[r] & 0xFFu);
            const bool isp = sp < 174 && c >= 91;
            const uint32_t bal = __ballot_sync(FULL, isp);
            const int prank = pbase + __popc(bal & ((1u << lane) - 1u));
            pbase += __popc(bal);
            if (sp < 174) {
                if (isp) s.pcol[prank] = (uint8_t)c;
                s.order[sp] = (uint32_t)(isp ? 128 + prank : c);
                if (r >= 3 && c < 91) {
                    const uint32_t b = 1u << (c & 31);
                    if (c < 32) L0 |= b; else if (c < 64) L1 |= b; else L2 |= b;
                }
            }
        }
    } else {
        // exact order by counting: position of column i = number of columns that precede it
        // (larger |llr|, or equal |llr| and smaller index; NaN after every number); parity rank = the parity columns among them
        for (int i = lane; i < 174; i += 32) {
            const float a = fabsf(llr[i]);
            const uint32_t ui = (a != a) ? 0u : (__float_as_uint(a) + 1u);
            int rank = 0, prank = 0;
            for (int q = 0; q < 174; ++q) {
                const float aq = fabsf(llr[q]);
                const uint32_t uq = (aq != aq) ? 0u : (__float_as_uint(aq) + 1u);
                const int before = (uq > ui || (uq == ui && q < i)) ? 1 : 0;
                rank += before;
                prank += (q >= 91) ? before : 0;
            }
            if (i >= 91) s.pcol[prank] = (uint8_t)i;
            s.order[rank] = (uint32_t)(i >= 91 ? 128 + prank : i);
            if (rank >= 96 && i < 91) {
                const uint32_t b = 1u << (i & 31);
                if (i < 32) L0 |= b; else if (i < 64) L1 |= b; else L2 |= b;
            }
        }
    }
    L0 = __reduce_or_sync(FULL, L0); L1 = __reduce_or_sync(FULL, L1); L2 = __reduce_or_sync(FULL, L2);
    // ---- 3. the 83 parity columns (slot r of lane l: the parity column of rank 32 r + l), eliminated in place
    __syncwarp();
    uint32_t (&c0)[3] = ob.c0, (&c1)[3] = ob.c1, (&c2)[3] = ob.c2, (&ownrow)[3] = ob.ownrow;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int j = 32 * r + lane;
        ownrow[r] = 255;
        if (j < 83) { const int col = s.pcol[j]; c0[r] = g.col[col]; c1[r] = g.col[OSD_COL_PITCH + col]; c2[r] = g.col[2 * OSD_COL_PITCH + col]; }
        else c0[r] = c1[r] = c2[r] = 0u;
    }
    uint32_t own0 = 0, own1 = 0, own2 = 0;        // slot holding the image of row lane / 32 + lane / 64 + lane
    uint32_t used0 = 0, used1 = 0, used2 = 0;     // rows already holding a pivot
    int npiv = 0;
    // One visit of a stored column (slot j, fetched as v0..v2): dependent -> false; else pick the pivot row, do the
    // bookkeeping and eliminate.  JR = 0..2: the slot index is static (parity column in rank order); JR = 3: dynamic (the
    // stored image of a systematic column).  col = the column being visited.
    auto visit = [&](auto JRc, uint32_t v0, uint32_t v1, uint32_t v2, int j, int jl, int col) -> bool {
        constexpr int JR = decltype(JRc)::value;
        const uint32_t f0 = v0 & ~used0, f1 = v1 & ~used1, f2 = v2 & ~used2;
        if ((f0 | f1 | f2) == 0) return false;    // dependent column
        uint32_t g0 = f0 & L0, g1 = f1 & L1, g2 = f2 & L2;
        if ((g0 | g1 | g2) == 0) { g0 = f0; g1 = f1; g2 = f2; }
        const int pw = g0 ? 0 : (g1 ? 1 : 2);
        const uint32_t gw = g0 ? g0 : (g1 ? g1 : g2);
        const uint32_t pb = gw & (0u - gw);
        const int pl = 31 - __clz(pb);
        const int p = 32 * pw + pl;
        if (lane == 0) { s.piv_row[npiv] = (uint8_t)p; s.piv_col[npiv] = (uint8_t)col; }
        // pw is warp-uniform: three copies of the update, each testing a fixed word
        uint32_t x0 = v0, x1 = v1, x2 = v2;       // the pivot column with the pivot row cleared
        constexpr int A = JR < 3 ? JR : 0, B = (A + 1) % 3, D = (A + 2) % 3;
        if (pw == 0) {
            used0 |= pb;
            if (lane == pl) own0 = (uint32_t)j;
            x0 &= ~pb;
            if (JR < 3) { OSD_ELIM_S(A, B, D, c0[A], c0[B], c0[D]); } else { OSD_ELIM(c0[0], c0[1], c0[2]); }
        } else if (pw == 1) {
            used1 |= pb;
            if (lane == pl) own1 = (uint32_t)j;
            x1 &= ~pb;
            if (JR < 3) { OSD_ELIM_S(A, B, D, c1[A], c1[B], c1[D]); } else { OSD_ELIM(c1[0], c1[1], c1[2]); }
        } else {
            used2 |= pb;
            if (lane == pl) own2 = (uint32_t)j;
            x2 &= ~pb;
            if (JR < 3) { OSD_ELIM_S(A, B, D, c2[A], c2[B], c2[D]); } else { OSD_ELIM(c2[0], c2[1], c2[2]); }
        }
        return true;
    };
    uint32_t e_next = s.order[0];
    for (int sp = 0; sp < 174; ++sp) {
        const int c = (int)e_next;
        e_next = s.order[sp + 1];                 // order[] is padded; the entry after the last one is never used
        bool piv;
        if (c < 128) {                            // systematic column c
            const int w = c >> 5;
            const uint32_t b = 1u << (c & 31);
            if ((sel3(w, used0, used1, used2) & b) == 0) {        // untouched unit vector on a free row: nothing to eliminate
                if (w == 0) used0 |= b; else if (w == 1) used1 |= b; else used2 |= b;
                if (lane == 0) { s.piv_row[npiv] = (uint8_t)c; s.piv_col[npiv] = (uint8_t)c; }
                piv = true;
            } else {                                               // its image lives in a basis slot
                const int j = (int)__shfl_sync(FULL, sel3(w, own0, own1, own2), c & 31);
                const int jl = j & 31, jr = j >> 5;
                const uint32_t v0 = __shfl_sync(FULL, sel3(jr, c0[0], c0[1], c0[2]), jl);
                const uint32_t v1 = __shfl_sync(FULL, sel3(jr, c1[0], c1[1], c1[2]), jl);
                const uint32_t v2 = __shfl_sync(FULL, sel3(jr, c2[0], c2[1], c2[2]), jl);
                piv = visit(std::integral_constant<int, 3>{}, v0, v1, v2, j, jl, c);
            }
        } else {                                  // parity column of rank j: slot j / 32 of lane j % 32
            const int j = c - 128, jl = j & 31;
            const int col = s.pcol[j];
            if (j < 32) {
                piv = visit(std::integral_constant<int, 0>{}, __shfl_sync(FULL, c0[0], jl), __shfl_sync(FULL, c1[0], jl), __shfl_sync(FULL, c2[0], jl), j, jl, col);
            } else if (j < 64) {
                piv = visit(std::integral_constant<int, 1>{}, __shfl_sync(FULL, c0[1], jl), __shfl_sync(FULL, c1[1], jl), __shfl_sync(FULL, c2[1], jl), j, jl, col);
            } else {
                piv = visit(std::integral_constant<int, 2>{}, __shfl_sync(FULL, c0[2], jl), __shfl_sync(FULL, c1[2], jl), __shfl_sync(FULL, c2[2], jl), j, jl, col);
            }
        }
        if (piv && ++npiv == 91) break;
    }
    __syncwarp();
    // ---- 4. CRC syndromes of the S flip vectors (vector i = what flip i adds).  Only the 14-bit syndromes are needed to
    //      test a trial; the 91-bit words themselves are built on demand (osd_word) for the rare trials whose syndrome is
    //      zero.  A slot that is not a basis slot contributes nothing (syndrome 0).
    //      Publish the stored columns word-major and let lane i walk the 83 slots for the bit of its pivot row (a per-vector
    //      warp reduction costs 30 x ~40 instructions; this loop ~6 x 83).
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int j = 32 * k + lane;
        s.colw[j] = c0[k]; s.colw[OSD_W_PITCH + j] = c1[k]; s.colw[2 * OSD_W_PITCH + j] = c2[k];
        s.ssyn[j] = (ownrow[k] < 91) ? g.syn[ownrow[k]] : (uint16_t)0;
    }
    __syncwarp();
    for (int i0 = 0; i0 < S; i0 += 32) {
        const int i = i0 + lane;
        const bool act = i < S;
        const int prow = act ? s.piv_row[90 - i] : 0, pcol = act ? s.piv_col[90 - i] : 255;
        const uint32_t* cw = s.colw + (prow >> 5) * OSD_W_PITCH;
        const int sh = prow & 31;
        uint32_t syn = (uint32_t)g.syn[pcol < 91 ? pcol : 95];           // syn[95] = 0: parity pivots add no unit bit
#pragma unroll 4
        for (int q = 0; q < 83; ++q)
            if ((cw[q] >> sh) & 1u) syn ^= (uint32_t)s.ssyn[q];
        if (act) s.syn[i] = (uint16_t)syn;
    }
    __syncwarp();
}

// Step 5 for the hard decisions of llr (llr[c] > 0; NaN and -0 are 0) on the basis osd_basis found for the same |llr|.
// Returns trial index + 1 of the first accepted trial word (0 = none); bits = that word, else the order-0 word.
__device__ __forceinline__ int osd_eval(const OsdWarpScratch& s, const OsdCtaTables& g, const float* llr, int lane, const LaneSyn& ls, int S, int D,
                                        const OsdBasis& ob, uint32_t* bits) {
    constexpr uint32_t FULL = 0xffffffffu;
    const uint32_t (&c0)[3] = ob.c0, (&c1)[3] = ob.c1, (&c2)[3] = ob.c2, (&ownrow)[3] = ob.ownrow;
    // u[row] = hard decision of that row's pivot column; hs = hard decisions of the basis' systematic columns, by column
    uint32_t u0 = 0, u1 = 0, u2 = 0, hs0 = 0, hs1 = 0, hs2 = 0;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int k = 32 * r + lane;
        if (k < 91) {
            const int col = s.piv_col[k];
            if (llr[col] > 0.0f) {
                const int row = s.piv_row[k];
                const uint32_t rb = 1u << (row & 31), cb = 1u << (col & 31);
                if (row < 32) u0 |= rb; else if (row < 64) u1 |= rb; else u2 |= rb;
                if (col < 32) hs0 |= cb; else if (col < 64) hs1 |= cb; else if (col < 91) hs2 |= cb;
            }
        }
    }
    u0 = __reduce_or_sync(FULL, u0); u1 = __reduce_or_sync(FULL, u1); u2 = __reduce_or_sync(FULL, u2);
    hs0 = __reduce_or_sync(FULL, hs0); hs1 = __reduce_or_sync(FULL, hs1); hs2 = __reduce_or_sync(FULL, hs2);
    // CRC syndrome of the order-0 word
    uint32_t bs = (((hs0 >> lane) & 1u) ? ls.s0 : 0u) ^ (((hs1 >> lane) & 1u) ? ls.s1 : 0u) ^ (((hs2 >> lane) & 1u) ? ls.s2 : 0u);
#pragma unroll
    for (int k = 0; k < 3; ++k)
        if ((__popc(c0[k] & u0) + __popc(c1[k] & u1) + __popc(c2[k] & u2)) & 1) bs ^= s.ssyn[32 * k + lane];
    bs = __reduce_xor_sync(FULL, bs);
    // 91-bit word of vector vi (0: order 0, i + 1: flip i, -1: none), XOR-accumulated into w0..w2; every lane gets the result
    auto osd_word = [&](int vi, uint32_t& w0, uint32_t& w1, uint32_t& w2) {
        if (vi < 0) return;
        uint32_t x0 = 0, x1 = 0, x2 = 0;
        const int prow = vi > 0 ? s.piv_row[91 - vi] : 0;
        const int pcol = vi > 0 ? s.piv_col[91 - vi] : 255;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int c = ownrow[k];
            if (c < 91) {
                uint32_t bt;
                if (vi == 0) bt = (__popc(c0[k] & u0) + __popc(c1[k] & u1) + __popc(c2[k] & u2)) & 1u;
                else bt = (((prow < 32) ? c0[k] : ((prow < 64) ? c1[k] : c2[k])) >> (prow & 31)) & 1u;
                if (bt) { const uint32_t bit = 1u << (c & 31); if (c < 32) x0 |= bit; else if (c < 64) x1 |= bit; else x2 |= bit; }
            }
        }
        x0 = __reduce_or_sync(FULL, x0); x1 = __reduce_or_sync(FULL, x1); x2 = __reduce_or_sync(FULL, x2);
        if (vi == 0) { x0 |= hs0; x1 |= hs1; x2 |= hs2; }
        else if (pcol < 91) { const uint32_t bit = 1u << (pcol & 31); if (pcol < 32) x0 |= bit; else if (pcol < 64) x1 |= bit; else x2 |= bit; }
        w0 ^= x0; w1 ^= x1; w2 ^= x2;
    };
    // enumerate trials in the reference's order; first with payload != 0, CRC ok, valid payload
    // trial 0: base; 1..S: single flips i = 0..S-1; then pairs (i, j), j < D, j < i, i-major.
    const int nsingle = S;
    const int npair = (S <= D) ? S * (S - 1) / 2 : D * (D - 1) / 2 + (S - D) * D;      // sum over i < S of min(i, D)
    const int ntrial = 1 + nsingle + npair;
    const int tri = D * (D - 1) / 2;               // pairs of the rows i < D (row i has i of them); every later row has D
    for (int base = 0; base < ntrial; base += 32) {
        const int tr = base + lane;
        bool pass = false;
        int fi = -1, fj = -1;
        if (tr < ntrial) {
            if (tr == 0) { }
            else if (tr <= nsingle) fi = tr - 1;
            else {
                int q = tr - 1 - nsingle;      // q-th pair
                if (q >= tri && D > 0) { q -= tri; fi = D + q / D; fj = q - (fi - D) * D; }
                else { int i = 0; while (q >= i) { q -= i; ++i; } fi = i; fj = q; }
            }
            uint32_t syn = bs;
            if (fi >= 0) syn ^= s.syn[fi];
            if (fj >= 0) syn ^= s.syn[fj];
            pass = (syn == 0);
        }
        uint32_t ballot = __ballot_sync(FULL, pass);
        while (ballot) {
            const int src = __ffs(ballot) - 1;
            ballot &= ballot - 1;
            const int sfi = __shfl_sync(FULL, fi, src), sfj = __shfl_sync(FULL, fj, src);
            uint32_t w[3] = {0u, 0u, 0u};
            osd_word(0, w[0], w[1], w[2]);
            osd_word(sfi >= 0 ? 1 + sfi : -1, w[0], w[1], w[2]);
            osd_word(sfj >= 0 ? 1 + sfj : -1, w[0], w[1], w[2]);
            if ((w[0] | w[1] | (w[2] & 0x1FFFu)) != 0 && payload_valid(w)) {
                bits[0] = w[0]; bits[1] = w[1]; bits[2] = w[2];
                return base + src + 1;
            }
        }
    }
    bits[0] = bits[1] = bits[2] = 0u;
    osd_word(0, bits[0], bits[1], bits[2]);           // nothing accepted: report the order-0 word
    return 0;
}

// Returns trial index + 1 of the first accepted trial word (0 = none); bits = that word.
// llr: 174 floats in shared or global memory.
__device__ __forceinline__ int osd_warp(OsdWarpScratch& s, const OsdCtaTables& g, const float* llr, int lane, const LaneSyn& ls, int S, int D, uint32_t* bits) {
    OsdBasis ob;
    osd_basis(s, g, llr, lane, S, ob);
    return osd_eval(s, g, llr, lane, ls, S, D, ob, bits);
}

}  // namespace ft8
