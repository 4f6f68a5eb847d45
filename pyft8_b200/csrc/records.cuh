// records.cuh -- R1: record packaging on the device (receiver.py:51-66, 389-398).
//
// One CTA per cycle orders that cycle's decoded candidates in the reference's emission order -- pass by pass; inside a
// pass by llr_sd descending (the fine sd from ipass 2 on, all-equal before), ties by candidate rank -- flags later
// duplicates of a payload (receiver.py:53-55) and writes the records contiguously at base[cycle], so the host only copies.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "../../include/ft8_b200.h"
#include "passes.cuh"

using namespace ft8;

constexpr int REC_MAXC = 928, REC_NT = 256;

__global__ void __launch_bounds__(REC_NT) k_rec_count(CandState cs, int32_t* __restrict__ n_per_cycle) {
    __shared__ int cnt;
    const int cyc = blockIdx.x;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    const int n = cs.n_cand[cyc];
    int c = 0;
    for (int r = threadIdx.x; r < n; r += REC_NT) c += cs.status[cyc * cs.K + r] == ST_DECODED;
    if (c) atomicAdd(&cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) n_per_cycle[cyc] = cnt;
}

// exclusive scan of n_per_cycle[B] -> base[B], total -> *total (single CTA)
__global__ void __launch_bounds__(1024) k_rec_scan(const int32_t* __restrict__ n_per_cycle, int B, int32_t* __restrict__ base,
                                                   int32_t* __restrict__ total) {
    __shared__ int warp_sum[32];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int b0 = 0; b0 < B; b0 += 1024) {
        const int i = b0 + threadIdx.x;
        const int v = i < B ? n_per_cycle[i] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
        if (lane == 31) warp_sum[w] = x;
        __syncthreads();
        if (w == 0) {
            int s = warp_sum[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, s, o); if (lane >= o) s += y; }
            warp_sum[lane] = s;
        }
        __syncthreads();
        const int before = carry + (w ? warp_sum[w - 1] : 0) + x - v;
        if (i < B) base[i] = before;
        __syncthreads();
        if (threadIdx.x == 1023) carry = before + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) *total = carry;
}

// The record of decoded candidate `slot` (rank rk of cycle cyc, decoded in pass ip); dup = an earlier record of the cycle has
// the same payload.
__device__ __forceinline__ ft8_record make_record(const CandState& cs, const FineOut* __restrict__ fine, int slot, int cyc, int rk,
                                                  int ip, bool dup) {
    ft8_record r;
    memset(&r, 0, sizeof(r));
    r.bits91[0] = cs.bits91[3 * slot]; r.bits91[1] = cs.bits91[3 * slot + 1]; r.bits91[2] = cs.bits91[3 * slot + 2];
    r.cycle = cyc; r.cand = (int16_t)rk; r.f0_idx = cs.f0[slot]; r.h0_idx = cs.h0[slot];
    r.ipass = (uint8_t)ip; r.ap = cs.r_ap[slot]; r.method = cs.r_method[slot]; r.n_its = cs.r_nits[slot];
    r.score = cs.score[slot]; r.grid_sd = cs.grid_sd[slot];
    r.emitted = dup ? 0 : 1;
    // float(h0/25) and 3.125*f0 like receiver.py:350-351 (python floats; rounded to fp32 for the record)
    double tsec = (double)r.h0_idx / 25.0, fhz = 3.125 * (double)r.f0_idx;
    if (ip >= 2) {
        const FineOut fo = fine[slot];
        r.ttweak = (int8_t)fo.tt; r.ftweak = (int8_t)fo.ff; r.nsync = (uint8_t)fo.nsync; r.fine_sd = fo.sd; r.snr = (int8_t)fo.snr;
        tsec += (double)fo.tt / 200.0; fhz += (double)fo.ff / 16.0;
    } else {
        r.nsync = 100; r.fine_sd = nanf(""); r.snr = cs.grid_snr[slot];
    }
    r.tsec = (float)tsec; r.fHz = (float)fhz;
    return r;
}

// The decoded candidates of cycle cyc in candidate order (ballot scan per warp-sized chunk keeps it deterministic): rank,
// pass, llr_sd at sort time (the fine sd from ipass 2 on, 0 before) and payload of the i-th, their number in s_n (zero on
// entry).  Ends with a barrier.
__device__ __forceinline__ void compact_decoded(const CandState& cs, const FineOut* __restrict__ fine, int cyc, uint16_t* s_rank,
                                                uint8_t* s_ipass, float* s_sd, uint32_t (*s_w)[3], int& s_n) {
    const int lane = threadIdx.x & 31;
    const int n = cs.n_cand[cyc];
    for (int r0 = 0; r0 < n; r0 += REC_NT) {
        const int r = r0 + threadIdx.x;
        const bool dec = r < n && cs.status[cyc * cs.K + r] == ST_DECODED;
        const uint32_t m = __ballot_sync(0xffffffffu, dec);
        __shared__ int wbase[REC_NT / 32];
        if (lane == 0) wbase[threadIdx.x >> 5] = __popc(m);
        __syncthreads();
        int off = s_n;
        for (int w = 0; w < (threadIdx.x >> 5); ++w) off += wbase[w];
        if (dec) {
            const int i = off + __popc(m & ((1u << lane) - 1u));
            const int slot = cyc * cs.K + r;
            s_rank[i] = (uint16_t)r;
            s_ipass[i] = cs.r_ipass[slot];
            s_sd[i] = cs.r_ipass[slot] >= 2 ? fine[slot].sd : 0.0f;
            s_w[i][0] = cs.bits91[3 * slot]; s_w[i][1] = cs.bits91[3 * slot + 1]; s_w[i][2] = cs.bits91[3 * slot + 2] & 0x1FFFu;
        }
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < REC_NT / 32; ++w) t += wbase[w]; s_n += t; }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(REC_NT)
k_rec_write(CandState cs, const FineOut* __restrict__ fine, const int32_t* __restrict__ base, ft8_record* __restrict__ rec,
            DevStats* __restrict__ stats) {
    __shared__ uint16_t s_rank[REC_MAXC];      // candidate rank (index inside the cycle) of the i-th decoded candidate
    __shared__ uint8_t s_ipass[REC_MAXC];
    __shared__ float s_sd[REC_MAXC];
    __shared__ uint32_t s_w[REC_MAXC][3];
    __shared__ int s_n, s_emit;
    const int cyc = blockIdx.x;
    if (threadIdx.x == 0) { s_n = 0; s_emit = 0; }
    __syncthreads();
    compact_decoded(cs, fine, cyc, s_rank, s_ipass, s_sd, s_w, s_n);
    const int nd = s_n;
    int emitted_here = 0;
    for (int i = threadIdx.x; i < nd; i += REC_NT) {
        const int ip = s_ipass[i];
        const float sd = s_sd[i];
        const int rk = s_rank[i];
        int pos = 0;
        bool dup = false;
        for (int j = 0; j < nd; ++j) {
            const int jp = s_ipass[j];
            bool before;                      // does j precede i in emission order?
            if (jp != ip) before = jp < ip;
            else if (ip >= 2 && s_sd[j] != sd) before = s_sd[j] > sd;
            else before = s_rank[j] < rk;
            if (before) {
                ++pos;
                dup = dup || (s_w[j][0] == s_w[i][0] && s_w[j][1] == s_w[i][1] && s_w[j][2] == s_w[i][2]);
            }
        }
        const ft8_record r = make_record(cs, fine, cyc * cs.K + rk, cyc, rk, ip, dup);
        emitted_here += dup ? 0 : 1;
        rec[base[cyc] + pos] = r;
    }
    if (emitted_here) atomicAdd(&s_emit, emitted_here);
    __syncthreads();
    if (threadIdx.x == 0 && s_emit) atomicAdd(&stats->emitted, (unsigned long long)s_emit);
}

// Progressive live decoding (ft8_decode_cycles_live_progress): candidate rank rk is searched at hop S, runs pass k at hop
// d + k with d = max(S + 1, h0 + 285) -- the first hop at which the receiver's grid pointer has left the candidate's payload
// rows -- and a success in pass k comes out at hop e = d + k, inside a hop by llr_sd at sort time descending, then by rank.
// So the emission order of a stream-cycle is the key (e, -sd, rank); with every d equal it is k_rec_write's.
__device__ __forceinline__ int prog_due_hop(int S, int h0) { return max(S + 1, h0 + 285); }

// One CTA per stream: the decoded records with e in (e_lo, e_hi].  WRITE = false: their number to n_out[stream];
// WRITE = true: the records at base[stream] in emission order, e to emit_hop, duplicates flagged against every earlier key
// of the stream-cycle (released by an earlier call or not: a smaller key has a smaller or equal e, so it is final).
template <bool WRITE>
__global__ void __launch_bounds__(REC_NT)
k_prog_rec(CandState cs, const FineOut* __restrict__ fine, int S, int e_lo, int e_hi, int32_t* __restrict__ n_out,
           const int32_t* __restrict__ base, ft8_record* __restrict__ rec, uint16_t* __restrict__ emit_hop,
           DevStats* __restrict__ stats) {
    __shared__ uint16_t s_rank[REC_MAXC];
    __shared__ uint8_t s_ipass[REC_MAXC];
    __shared__ float s_sd[REC_MAXC];
    __shared__ uint32_t s_w[REC_MAXC][3];
    __shared__ int s_n, s_count;
    const int cyc = blockIdx.x;
    if (threadIdx.x == 0) { s_n = 0; s_count = 0; }
    __syncthreads();
    compact_decoded(cs, fine, cyc, s_rank, s_ipass, s_sd, s_w, s_n);
    const int nd = s_n;
    int here = 0;
    for (int i = threadIdx.x; i < nd; i += REC_NT) {
        const int rk = s_rank[i], ip = s_ipass[i];
        const int e = prog_due_hop(S, cs.h0[cyc * cs.K + rk]) + ip;
        if (e <= e_lo || e > e_hi) continue;
        if (!WRITE) { ++here; continue; }
        const float sd = s_sd[i];
        int pos = 0;
        bool dup = false;
        for (int j = 0; j < nd; ++j) {
            const int ej = prog_due_hop(S, cs.h0[cyc * cs.K + s_rank[j]]) + s_ipass[j];
            bool before;                      // does j precede i in emission order?
            if (ej != e) before = ej < e;
            else if (s_sd[j] != sd) before = s_sd[j] > sd;
            else before = s_rank[j] < rk;
            if (before) {
                pos += ej > e_lo;
                dup = dup || (s_w[j][0] == s_w[i][0] && s_w[j][1] == s_w[i][1] && s_w[j][2] == s_w[i][2]);
            }
        }
        rec[base[cyc] + pos] = make_record(cs, fine, cyc * cs.K + rk, cyc, rk, ip, dup);
        emit_hop[base[cyc] + pos] = (uint16_t)e;
        here += dup ? 0 : 1;
    }
    if (here) atomicAdd(&s_count, here);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (!WRITE) n_out[cyc] = s_count;
        else if (s_count) atomicAdd(&stats->emitted, (unsigned long long)s_count);
    }
}
