// passes.cuh -- C1: the per-candidate pass schedule of Candidate.decode (receiver.py:68-107) as device kernels.
//
// The reference advances every candidate one pass per scheduler round (receiver.py:389-398).  Candidates never
// interact before packaging, so the schedule is run here pass by pass over device-side work lists:
//   k_pass0    ipass 0   grid LLRs; for AP in NoAP,CQ,RR73,73,RRR: GOOD91 then LDPC(35,5)      -> list_fine
//   k_fine     ipass 1   fine sync (fine.cuh)
//   k_pass234  ipass 2-4 gate (nsync > 6, sd > sd_min); GOOD91 x2; LDPC(35,5) x2; LDPC(90,20) x5 (+save) -> list_osd
//   k_osd_items ipass 5-6 one warp per (candidate, OSD attempt): 5 AP'd llrs then the saved post-LDPC llrs
//   k_osd_resolve        first successful attempt in reference order wins
// All kernels are persistent: warps pull work from device-resident lists through atomic cursors (the cost per candidate
// varies from nothing to 110 LDPC iterations), so the host never reads a count back between passes (no sync; the
// sequence of launches is fixed and CUDA-graph capturable).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "ldpc.cuh"
#include "osd.cuh"
#include "sync.cuh"
#include "fine.cuh"

namespace ft8 {

constexpr int ST_PENDING = 0, ST_DECODED = 1, ST_STOPPED = 2;
constexpr int WARPS_PER_CTA = 4;

struct ApTables {
    int8_t first[5];          // first llr index of the pattern
    int8_t len[5];
    uint32_t mask[5];         // bit i = i-th forced bit (a word per pattern: a lane-indexed byte table in __constant__
                              // memory would be replayed once per lane)
};
__constant__ ApTables c_ap;

// Candidate._set_AP (receiver.py:109-117): dst = src with known bits forced to +-5
__device__ __forceinline__ void apply_ap(float* dst, const float* src, int ap, int lane) {
    __syncwarp();                 // earlier reads of dst by other lanes (previous attempt) are complete
    for (int i = lane; i < 174; i += 32) dst[i] = src[i];
    __syncwarp();
    if (ap > 0) {
        if (lane < c_ap.len[ap]) dst[c_ap.first[ap] + lane] = ((c_ap.mask[ap] >> lane) & 1u) ? 5.0f : -5.0f;
        if (ap == 1 && lane == 0) { dst[74] = -5.0f; dst[75] = -5.0f; dst[76] = 5.0f; dst[57] = -5.0f; dst[58] = -5.0f; }
    }
    __syncwarp();
}

struct CandState {            // structure-of-arrays views over all B*K slots
    int32_t K;                // slots per cycle (max_cands)
    const int32_t* n_cand;    // [B]
    const int16_t* f0;        // [N]
    const int16_t* h0;
    const float* score;
    uint8_t* status;          // ST_*
    float* llr_grid;          // [N][174]
    float* grid_sd;           // [N]
    int8_t* grid_snr;
    float* llr_fine;          // [N][174]
    FineOut* fine;            // [N]
    float* saved_llr;         // [N][5][174]
    uint8_t* saved_n;         // [N]
    uint8_t* saved_ap;        // [N][5]
    // result
    uint32_t* bits91;         // [N][3]
    uint8_t* r_ipass;
    uint8_t* r_ap;
    uint8_t* r_method;
    uint16_t* r_nits;
    // OSD attempt results
    int32_t* osd_found;       // [N][10]
    uint32_t* osd_bits;       // [N][10][3]
};

struct DevStats {
    unsigned long long candidates, stopped_sd, fine_evals, fine_pass, ldpc_calls, ldpc_iters, osd_calls, decoded, emitted;
};

struct PassSmem {
    LdpcCtaTables tab;
    LdpcWarpScratch w[WARPS_PER_CTA];
    float llr0[WARPS_PER_CTA][176];
};

__device__ __forceinline__ void set_result(const CandState& cs, int slot, const uint32_t* bits, int ipass, int ap, int method, int nits) {
    cs.bits91[3 * slot] = bits[0]; cs.bits91[3 * slot + 1] = bits[1]; cs.bits91[3 * slot + 2] = bits[2];
    cs.r_ipass[slot] = (uint8_t)ipass; cs.r_ap[slot] = (uint8_t)ap; cs.r_method[slot] = (uint8_t)method;
    cs.r_nits[slot] = (uint16_t)(nits < 0 ? 0 : nits);
    cs.status[slot] = ST_DECODED;
}

// ipass 0.  grid: [B][grid_rows][976].  payload_db (optional): [N][58][8].
// prev[] of the decoder in registers needs ~90 registers: 5 CTAs/SM instead of 8 (measured: 5.80 ms with prev in shared
// memory at 8 CTAs, 5.02 with the cheaper quotients, 4.33 with prev in registers at 5 CTAs)
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4)
k_pass0(CandState cs, int n_slots, const float* __restrict__ grid, int grid_rows, int cycle_h0, float sd_min,
        float* __restrict__ payload_db, int llr_only, int32_t* __restrict__ list_fine, int32_t* __restrict__ count_fine,
        int32_t* __restrict__ next_slot, DevStats* __restrict__ stats) {
    extern __shared__ __align__(16) unsigned char pass_smem_raw[];
    PassSmem& sm = *reinterpret_cast<PassSmem*>(pass_smem_raw);
    load_ldpc_tables(sm.tab);
    __syncthreads();
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LaneSyn ls = load_lane_syn(lane);
    LdpcWarpScratch& ws = sm.w[wi];
    float* llr0 = sm.llr0[wi];
    const int warps_total = gridDim.x * WARPS_PER_CTA;
    unsigned long long n_ldpc = 0, n_iter = 0, n_cand = 0, n_stop = 0, n_dec = 0;
    (void)warps_total;
    // candidates cost between ~0 (sd gate, iteration-0 rejects) and 25 LDPC iterations: warps pull batches of 4 slots
    for (int base = 0, sub = 4;; ++sub) {
        if (sub == 4) {
            if (lane == 0) base = atomicAdd(next_slot, 4);
            base = __shfl_sync(0xffffffffu, base, 0);
            sub = 0;
            if (base >= n_slots) break;
        }
        const int slot = base + sub;
        if (slot >= n_slots) continue;
        const int cyc = slot / cs.K, rank = slot - cyc * cs.K;
        if (rank >= cs.n_cand[cyc]) continue;
        ++n_cand;
        const int f0 = cs.f0[slot], h0 = cs.h0[slot];
        const float* g = grid + (size_t)cyc * grid_rows * GRID_COLS;
        // Payload gather (receiver.py:356-363): 58 symbol rows x 8 tones (the upper bin of each tone).  Lane = 8 * sub + tone
        // reads row 4 i + sub: the eight tones of a row share one or two 128-byte lines, so a load instruction touches 4-8
        // lines (one row per lane touched 29: 464 lines per candidate, 2.1x the algorithmic DRAM traffic and most of this
        // kernel's L1 wavefronts).  The values are handed to the symbol-per-lane layout of the LLR step through shared memory
        // (the decoder's delta array, idle until the first LDPC iteration).
        float p[2][8];
        {
            float* stage = ws.dlt;
            const int sub = lane >> 3, t = lane & 7;
            __syncwarp();                         // the previous slot's last LDPC iteration has read dlt
#pragma unroll
            for (int i = 0; i < 15; ++i) {
                const int sidx = 4 * i + sub;                             // payload symbol 0..57
                if (sidx < 58) {
                    const int sym = sidx < 29 ? sidx + 7 : sidx + 14;      // PAYLOAD_SYMB_IDXS = 7..35, 43..71
                    const float v = grid_at(g, grid_rows, cycle_h0 + h0 + 4 + 4 * sym, f0 + 1 + 2 * t);
                    stage[sidx * 8 + t] = v;
                    if (payload_db) payload_db[((size_t)slot * 58 + sidx) * 8 + t] = v;
                }
            }
            __syncwarp();
            if (lane < 29) {
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const float4 a = *reinterpret_cast<const float4*>(stage + (lane + 29 * q) * 8);
                    const float4 b = *reinterpret_cast<const float4*>(stage + (lane + 29 * q) * 8 + 4);
                    p[q][0] = a.x; p[q][1] = a.y; p[q][2] = a.z; p[q][3] = a.w;
                    p[q][4] = b.x; p[q][5] = b.y; p[q][6] = b.z; p[q][7] = b.w;
                }
            }
        }
        float sd; int snr;
        __syncwarp();                             // the previous slot's readers of llr0 are done (racecheck: write-after-read)
        llr_from_payload_warp(p, lane, llr0, sd, snr);
        __syncwarp();
        for (int i = lane; i < 174; i += 32) cs.llr_grid[(size_t)slot * 174 + i] = llr0[i];
        if (lane == 0) { cs.grid_sd[slot] = sd; cs.grid_snr[slot] = (int8_t)snr; cs.status[slot] = ST_PENDING; cs.saved_n[slot] = 0; }
        if (llr_only) continue;
        if (sd <= sd_min) {                       // receiver.py:221-222
            if (lane == 0) cs.status[slot] = ST_STOPPED;
            ++n_stop;
            continue;
        }
        bool done = false;
        for (int ap = 0; ap < 5 && !done; ++ap) {
            apply_ap(ws.llr, llr0, ap, lane);
            uint32_t bits[3];
            if (good91_warp(ws.llr, lane, bits, ls)) {
                if (lane == 0) set_result(cs, slot, bits, 0, ap, 0 /*GOOD91*/, 0);
                done = true;
                break;
            }
            int nits, iters = 0;
            const int st = ldpc_warp(ws, sm.tab, lane, ls, 35, 5, nits, bits, iters);
            ++n_ldpc; n_iter += iters;
            if (st == 1) {
                if (lane == 0) set_result(cs, slot, bits, 0, ap, 1 /*LDPC5*/, nits);
                done = true;
            }
        }
        if (done) ++n_dec;
        else if (lane == 0) list_fine[atomicAdd(count_fine, 1)] = slot;
    }
    if (lane == 0) {
        if (n_cand) atomicAdd(&stats->candidates, n_cand);
        if (n_stop) atomicAdd(&stats->stopped_sd, n_stop);
        if (n_ldpc) atomicAdd(&stats->ldpc_calls, n_ldpc);
        if (n_iter) atomicAdd(&stats->ldpc_iters, n_iter);
        if (n_dec) atomicAdd(&stats->decoded, n_dec);
    }
}

// ipass 2..4 over list_fine.
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 5)
k_pass234(CandState cs, const int32_t* __restrict__ list, const int32_t* __restrict__ count, float sd_min,
          int32_t* __restrict__ list_osd, int32_t* __restrict__ count_osd, int32_t* __restrict__ next_item,
          DevStats* __restrict__ stats) {
    extern __shared__ __align__(16) unsigned char pass_smem_raw[];
    PassSmem& sm = *reinterpret_cast<PassSmem*>(pass_smem_raw);
    load_ldpc_tables(sm.tab);
    __syncthreads();
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LaneSyn ls = load_lane_syn(lane);
    LdpcWarpScratch& ws = sm.w[wi];
    float* llr0 = sm.llr0[wi];
    const int warps_total = gridDim.x * WARPS_PER_CTA;
    const int n_items = *count;
    unsigned long long n_ldpc = 0, n_iter = 0, n_dec = 0, n_fpass = 0, n_feval = 0;
    (void)warps_total;
    // work is very uneven (0 .. 110 LDPC iterations per candidate): warps pull items from a device counter
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(next_item, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int slot = list[item];
        const FineOut fo = cs.fine[slot];
        ++n_feval;
        if (!(fo.nsync > 6) || fo.sd <= sd_min) {            // receiver.py:167-173, 221-222
            if (lane == 0) cs.status[slot] = ST_STOPPED;
            continue;
        }
        ++n_fpass;
        for (int i = lane; i < 174; i += 32) llr0[i] = cs.llr_fine[(size_t)slot * 174 + i];
        __syncwarp();
        bool done = false;
        uint32_t bits[3];
        for (int ap = 0; ap < 2 && !done; ++ap) {             // ipass 2
            apply_ap(ws.llr, llr0, ap, lane);
            if (good91_warp(ws.llr, lane, bits, ls)) {
                if (lane == 0) set_result(cs, slot, bits, 2, ap, 0, 0);
                done = true;
            }
        }
        // ipass 3 (two LDPC(35,5) attempts) and ipass 4 (five LDPC(90,20) attempts) share ONE inlined copy of the decoder
        // (two call sites doubled the kernel's code and its instruction-fetch stalls)
        int nsaved = 0;
        for (int a = 0; a < 7 && !done; ++a) {
            const bool p4 = a >= 2;
            const int ap = p4 ? a - 2 : a;
            apply_ap(ws.llr, llr0, ap, lane);
            int nits, iters = 0;
            const int st = ldpc_warp(ws, sm.tab, lane, ls, p4 ? 90 : 35, p4 ? 20 : 5, nits, bits, iters);
            ++n_ldpc; n_iter += iters;
            if (st == 1) { if (lane == 0) set_result(cs, slot, bits, p4 ? 4 : 3, ap, p4 ? 2 : 1, nits); done = true; }
            else if (p4 && st >= 2) {                         // FAIL or STALL: reference keeps the llr (receiver.py:128-129)
                float* dst = cs.saved_llr + ((size_t)slot * 5 + nsaved) * 174;
                for (int i = lane; i < 174; i += 32) dst[i] = ws.llr[i];
                if (lane == 0) cs.saved_ap[slot * 5 + nsaved] = (uint8_t)ap;
                ++nsaved;
            }
        }
        if (done) ++n_dec;
        else if (lane == 0) { cs.saved_n[slot] = (uint8_t)nsaved; list_osd[atomicAdd(count_osd, 1)] = slot; }
    }
    if (lane == 0) {
        if (n_ldpc) atomicAdd(&stats->ldpc_calls, n_ldpc);
        if (n_iter) atomicAdd(&stats->ldpc_iters, n_iter);
        if (n_dec) atomicAdd(&stats->decoded, n_dec);
        if (n_fpass) atomicAdd(&stats->fine_pass, n_fpass);
        if (n_feval) atomicAdd(&stats->fine_evals, n_feval);
    }
}

struct OsdSmem {
    OsdCtaTables tab;
    OsdWarpScratch w[WARPS_PER_CTA];
    float llr[WARPS_PER_CTA][176];
};

// ipass 5-6: item = 10 * list index + attempt.  attempts 0..4: AP pattern on the fine llr; 5..9: saved llr.
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 8)
k_osd_items(CandState cs, const int32_t* __restrict__ list, const int32_t* __restrict__ count, int S, int D,
            int32_t* __restrict__ next_item, DevStats* __restrict__ stats) {
    extern __shared__ __align__(16) unsigned char pass_smem_raw[];
    OsdSmem& sm = *reinterpret_cast<OsdSmem*>(pass_smem_raw);
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LaneSyn ls = load_lane_syn(lane);
    load_osd_tables(sm.tab);
    __syncthreads();
    const int warps_total = gridDim.x * WARPS_PER_CTA;
    const int n_items = *count * 10;
    unsigned long long n_osd = 0;
    (void)warps_total;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(next_item, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int slot = list[item / 10], k = item % 10;
        int found = 0;
        uint32_t bits[3] = {0, 0, 0};
        const bool run = (k < 5) || (k - 5 < cs.saved_n[slot]);
        if (run) {
            // attempts 0..4: Candidate._set_AP pattern on the fine llr; 5..9: llr saved after a failed LDPC(90,20)
            const float* src = (k < 5) ? cs.llr_fine + (size_t)slot * 174 : cs.saved_llr + ((size_t)slot * 5 + (k - 5)) * 174;
            apply_ap(sm.llr[wi], src, (k < 5) ? k : 0, lane);
            found = osd_warp(sm.w[wi], sm.tab, sm.llr[wi], lane, ls, S, D, bits);
            ++n_osd;
        }
        if (lane == 0) {
            cs.osd_found[slot * 10 + k] = found;
            cs.osd_bits[(slot * 10 + k) * 3] = bits[0];
            cs.osd_bits[(slot * 10 + k) * 3 + 1] = bits[1];
            cs.osd_bits[(slot * 10 + k) * 3 + 2] = bits[2];
        }
        __syncwarp();
    }
    if (lane == 0 && n_osd) atomicAdd(&stats->osd_calls, n_osd);
}

__global__ void k_osd_resolve(CandState cs, const int32_t* __restrict__ list, const int32_t* __restrict__ count,
                              DevStats* __restrict__ stats) {
    const int n = *count;
    for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < n; item += gridDim.x * blockDim.x) {
        const int slot = list[item];
        int win = -1;
        for (int k = 0; k < 10; ++k)
            if (cs.osd_found[slot * 10 + k] > 0) { win = k; break; }
        if (win < 0) { cs.status[slot] = ST_STOPPED; continue; }      // ipass 7
        const uint32_t* b = cs.osd_bits + (slot * 10 + win) * 3;
        if (win < 5) set_result(cs, slot, b, 5, win, 3 /*OSD*/, 0);
        else set_result(cs, slot, b, 6, cs.saved_ap[slot * 5 + win - 5], 4 /*LDPC20_OSD*/, 0);
        atomicAdd(&stats->decoded, 1ull);
    }
}

// ------------------------------------------------------------------ stand-alone stage kernels (parity tests, drop-in ops)
__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
k_llr_batch(const float* __restrict__ payload_db, int N, float* __restrict__ llr, float* __restrict__ sd, int32_t* __restrict__ snr) {
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LaneSyn ls = load_lane_syn(lane);
    for (int n = blockIdx.x * WARPS_PER_CTA + wi; n < N; n += gridDim.x * WARPS_PER_CTA) {
        float p[2][8];
        if (lane < 29) {
#pragma unroll
            for (int q = 0; q < 2; ++q)
#pragma unroll
                for (int t = 0; t < 8; ++t) p[q][t] = payload_db[((size_t)n * 58 + lane + 29 * q) * 8 + t];
        }
        float s; int r;
        llr_from_payload_warp(p, lane, llr + (size_t)n * 174, s, r);
        if (lane == 0) { sd[n] = s; snr[n] = r; }
    }
}

__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
k_ldpc_batch(float* __restrict__ llr, int N, int max_ncheck0, int max_iters, int32_t* __restrict__ status,
             int32_t* __restrict__ nits_out, uint32_t* __restrict__ bits_out) {
    extern __shared__ __align__(16) unsigned char pass_smem_raw[];
    PassSmem& sm = *reinterpret_cast<PassSmem*>(pass_smem_raw);
    load_ldpc_tables(sm.tab);
    __syncthreads();
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LaneSyn ls = load_lane_syn(lane);
    LdpcWarpScratch& ws = sm.w[wi];
    for (int n = blockIdx.x * WARPS_PER_CTA + wi; n < N; n += gridDim.x * WARPS_PER_CTA) {
        for (int i = lane; i < 174; i += 32) ws.llr[i] = llr[(size_t)n * 174 + i];
        __syncwarp();
        uint32_t bits[3];
        int nits, iters = 0;
        const int st = ldpc_warp(ws, sm.tab, lane, ls, max_ncheck0, max_iters, nits, bits, iters);
        __syncwarp();
        for (int i = lane; i < 174; i += 32) llr[(size_t)n * 174 + i] = ws.llr[i];
        if (lane == 0) {
            status[n] = st; nits_out[n] = nits;
            bits_out[3 * n] = bits[0]; bits_out[3 * n + 1] = bits[1]; bits_out[3 * n + 2] = bits[2];
        }
        __syncwarp();
    }
}

__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 8)
k_osd_batch(const float* __restrict__ llr, int N, int S, int D, int32_t* __restrict__ found, uint32_t* __restrict__ bits_out) {
    extern __shared__ __align__(16) unsigned char pass_smem_raw[];
    OsdSmem& sm = *reinterpret_cast<OsdSmem*>(pass_smem_raw);
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LaneSyn ls = load_lane_syn(lane);
    load_osd_tables(sm.tab);
    __syncthreads();
    for (int n = blockIdx.x * WARPS_PER_CTA + wi; n < N; n += gridDim.x * WARPS_PER_CTA) {
        for (int i = lane; i < 174; i += 32) sm.llr[wi][i] = llr[(size_t)n * 174 + i];
        __syncwarp();
        uint32_t bits[3];
        const int f = osd_warp(sm.w[wi], sm.tab, sm.llr[wi], lane, ls, S, D, bits);
        if (lane == 0) { found[n] = f; bits_out[3 * n] = bits[0]; bits_out[3 * n + 1] = bits[1]; bits_out[3 * n + 2] = bits[2]; }
        __syncwarp();
    }
}

__global__ void k_crc_batch(const uint32_t* __restrict__ bits91, int N, int32_t* __restrict__ flags) {
    for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < N; n += gridDim.x * blockDim.x) {
        uint32_t w[3] = {bits91[3 * n], bits91[3 * n + 1], bits91[3 * n + 2] & 0x07FFFFFFu};
        int f = crc_ok_serial(w) ? 1 : 0;
        if (payload_valid(w)) f |= 2;
        flags[n] = f;
    }
}

}  // namespace ft8
