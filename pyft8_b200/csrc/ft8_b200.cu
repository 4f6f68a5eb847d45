// ft8_b200.cu -- handle, table upload and the C ABI (include/ft8_b200.h) of the B200-native FT8 receive path, with the
// ABI's small helper kernels; the stage kernels live in the *.cuh headers.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC (see __graft_entry__.build).
// One handle = one device + one stream + constant tables + scratch sized from ft8_cfg.max_cycles.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/ft8_b200.h"
#include "ft8_tables.h"
#include "fft.cuh"
#include "codec.cuh"
#include "ldpc.cuh"
#include "osd.cuh"
#include "spectrogram.cuh"
#include "sync.cuh"
#include "fine.cuh"
#include "fine_tc.cuh"
#include "passes.cuh"
#include "synth.cuh"
#include "records.cuh"

using namespace ft8;

static thread_local std::string g_create_error;

// Device memory owned by the handle: move-only and freed with its owner.  ensure() only grows: before it frees the old
// block it synchronises the streams that may still read it, and when the new allocation fails it leaves the buffer empty.
template <typename T> class DevBuf {
  public:
    DevBuf() = default;
    DevBuf(DevBuf&& o) noexcept : p_(o.p_), n_(o.n_) { o.p_ = nullptr; o.n_ = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept { std::swap(p_, o.p_); std::swap(n_, o.n_); return *this; }
    ~DevBuf() { if (p_) cudaFree(p_); }
    operator T*() const { return p_; }
    cudaError_t ensure(size_t count, cudaStream_t reader = nullptr, cudaStream_t reader2 = nullptr) {
        if (count <= n_) return cudaSuccess;
        if (p_) {
            cudaError_t e = reader ? cudaStreamSynchronize(reader) : cudaSuccess;
            if (e == cudaSuccess && reader2) e = cudaStreamSynchronize(reader2);
            if (e == cudaSuccess) e = cudaFree(p_);
            if (e != cudaSuccess) return e;
            p_ = nullptr; n_ = 0;
        }
        const cudaError_t e = cudaMalloc((void**)&p_, count * sizeof(T));
        if (e != cudaSuccess) { p_ = nullptr; return e; }
        n_ = count;
        return cudaSuccess;
    }
  private:
    T* p_ = nullptr;
    size_t n_ = 0;
};

// slots of d_counts / h_counts: the work-list lengths of the fine and OSD stages, the records written, the near-tie
// candidates of the frequency scan, the work cursors of k_pass234 / k_osd_items / k_pass0, ft8_fine's out-of-range count
enum CountSlot { CNT_FINE, CNT_OSD, CNT_RECORDS, CNT_NEAR_TIE, CNT_CURSOR_PASS234, CNT_CURSOR_OSD, CNT_CURSOR_PASS0,
                 CNT_FINE_BAD, CNT_SLOTS };

// timing events: event i (1..8) ends stage i of a decode as listed at ft8_last_kernel_ms; then the pair around a stand-alone
// op and the two boundaries inside the three-kernel fine stage
enum Event { EV_START, EV_SPECTROGRAM, EV_SYNC, EV_CYCLE_SPECTRUM, EV_PASS0, EV_FINE, EV_PASS234, EV_OSD, EV_RECORDS,
             EV_OP_BEGIN, EV_OP_END, EV_TSCAN_END, EV_FSCAN_END, EV_COUNT };

// `which` of ft8_last_kernel_ms
enum KernelMs { MS_TOTAL, MS_SPECTROGRAM, MS_SYNC, MS_CYCLE_SPECTRUM, MS_PASS0, MS_FINE, MS_PASS234, MS_OSD, MS_RECORDS,
                MS_FINE_TSCAN, MS_FINE_FSCAN, MS_FINE_FINAL, MS_COUNT };

struct ft8_handle {
    int device = 0;
    int n_sm = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;     // host->device audio copies, overlapped with S1/S2/F1 of earlier chunks
    cudaEvent_t chunk_ev[16] = {};
    ft8_cfg cfg{};
    std::string err;
    // constant-like tables in global memory
    DevBuf<float> d_hann;
    DevBuf<float2> d_W1920, d_W3840, d_W3200, d_W375, d_W256, d_W192000, d_W32;
    DevBuf<float2> d_TS, d_TF, d_TC, d_T256, d_W96000T;   // per-pass twiddle tables [k-1][p]
    DevBuf<float> d_pulse;           // GFSK pulse for the synthetic generator
    // tensor-core frequency scan (fine_tc.cuh): B operand (E | M, tf32 hi/lo), half-sample phase table, per-item intermediates
    DevBuf<float> d_bmat; DevBuf<float2> d_w6400;
    DevBuf<float2> d_zwin; DevBuf<TScanOut> d_tso; DevBuf<int32_t> d_ff;
    DevBuf<int32_t> d_amb;           // [items + 1]: near-tie candidates of the frequency scan ([0] = count, list from [1])
    // batch scratch
    size_t cap_cycles = 0, cap_slots = 0;
    DevBuf<char> d_audio;
    // prefetch slot (ft8_prefetch_audio): the NEXT batch's audio is copied here while the current batch is decoded
    DevBuf<char> d_audio_pf;
    const void* pf_host = nullptr; int pf_B = 0, pf_dtype = -1;
    cudaEvent_t pf_ev = nullptr;
    DevBuf<float> d_grid;
    // live mode (ft8_decode_cycles_live): the reference's two-cycle waterfall ring per stream + the previous cycle's last window
    // (float32 whatever the input dtype; zero for a stream that has no previous cycle)
    DevBuf<float> d_ring, d_tail;
    // consecutive live cycles (ft8_decode_cycles_live_seq): one SEQ_ROWS-row grid and one previous-cycle tail per cycle of a piece
    DevBuf<float> d_seq_grid, d_seq_tail;
    DevBuf<float2> d_Y; size_t y_cycles = 0;
    DevBuf<float2> d_spec;
    DevBuf<float> d_best_score; DevBuf<int16_t> d_best_h0;
    DevBuf<int16_t> d_f0, d_h0; DevBuf<float> d_score; DevBuf<int32_t> d_ncand;
    DevBuf<int32_t> d_cycle_of;
    DevBuf<uint8_t> d_status; DevBuf<float> d_llr_grid, d_grid_sd; DevBuf<int8_t> d_grid_snr;
    DevBuf<float> d_llr_fine; DevBuf<FineOut> d_fine; DevBuf<float> d_saved; DevBuf<uint8_t> d_saved_n;
    DevBuf<uint8_t> d_saved_ap; DevBuf<uint32_t> d_bits; DevBuf<uint8_t> d_ripass, d_rap, d_rmethod;
    DevBuf<uint16_t> d_rnits; DevBuf<int32_t> d_osd_found; DevBuf<uint32_t> d_osd_bits;
    DevBuf<int32_t> d_list_fine, d_list_osd, d_counts;   // d_counts: [CNT_SLOTS]
    DevBuf<DevStats> d_stats;
    DevBuf<ft8_record> d_rec;
    DevBuf<int32_t> d_rec_n, d_rec_base;   // per-cycle record counts / offsets
    int32_t* h_counts = nullptr;      // pinned [CNT_SLOTS]
    DevStats* h_stats = nullptr;      // pinned
    DevBuf<char> arena;               // host buffers and scratch of the stand-alone stage ops (Staging)
    cudaEvent_t ev[EV_COUNT] = {};
    float last_ms[MS_COUNT] = {};
    ft8_stats stats{};
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess) {                                                                  \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e__);                          \
            return FT8_E_CUDA;                                                                     \
        }                                                                                          \
    } while (0)

static int fail(ft8_handle* h, int code, const std::string& msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}

// ------------------------------------------------------------------------------------------ tables
static std::vector<float2> twiddles(int n, int count) {
    std::vector<float2> w(count);
    for (int j = 0; j < count; ++j) {
        const double a = -2.0 * M_PI * (double)j / (double)n;
        w[j] = make_float2((float)cos(a), (float)sin(a));
    }
    return w;
}

static float2 twiddle1(int n, long long j) {
    const double a = -2.0 * M_PI * (double)(j % n) / (double)n;
    return make_float2((float)cos(a), (float)sin(a));
}

// Per-pass twiddle table of Stockham pass (R, S) of a length-n transform, laid out [k-1][p] (fft.cuh, Pass::compute_store
// with TT = true): entry = w_n^(p k S), the same value the plain table holds at index p*k*S.
static void append_pass_table(std::vector<float2>& out, int n, int R, int S) {
    const int M = n / (R * S);
    for (int k = 1; k < R; ++k)
        for (int p = 0; p < M; ++p) out.push_back(twiddle1(n, (long long)p * k * S));
}

template <typename T> static cudaError_t upload(DevBuf<T>& dst, const std::vector<T>& v) {
    cudaError_t e = dst.ensure(v.size());
    if (e != cudaSuccess) return e;
    return cudaMemcpy(dst, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
}

static uint32_t crc14_bits(const uint8_t* msg77) {      // decoders.py:123-129
    uint32_t r = 0;
    for (int i = 0; i < 96; ++i) {
        const uint32_t bit = (i < 77) ? msg77[i] : 0u;
        const uint32_t top = (r >> 13) & 1u;
        r = ((r << 1) & 0x3FFFu) | bit;
        if (top) r ^= 0x2757u;
    }
    return r;
}

static cudaError_t upload_constant_tables() {
    // CRC syndrome contributions
    CodecTables ct;
    memset(&ct, 0, sizeof(ct));
    for (int j = 0; j < 91; ++j) {
        if (j < 77) {
            uint8_t m[77] = {0};
            m[j] = 1;
            ct.crc_syn[j] = (uint16_t)crc14_bits(m);
        } else {
            ct.crc_syn[j] = (uint16_t)(1u << (90 - j));
        }
    }
    memcpy(ct.prefix2, FT8_PREFIX2_BITS, sizeof(ct.prefix2));
    cudaError_t e = cudaMemcpyToSymbol(c_codec, &ct, sizeof(ct));
    if (e != cudaSuccess) return e;
    // LDPC graph; variable -> edge slots in np.add.at order (degree-6 group flattened first, then degree-7)
    LdpcTables lt;
    memset(&lt, 0, sizeof(lt));
    int cnt[174] = {0};
    for (int c = 0; c < 83; ++c)
        for (int k = 0; k < 7; ++k) {
            const uint8_t v = FT8_CHECK_VARS[c][k];
            lt.chk_var[c * 7 + k] = v;
            if (v != 255) lt.var_edge[3 * v + cnt[v]++] = (uint16_t)(c * 7 + k);
        }
    e = cudaMemcpyToSymbol(c_ldpc, &lt, sizeof(lt));
    if (e != cudaSuccess) return e;
    // OSD columns of G0 = [I | A^T]
    OsdTables ot;
    memset(&ot, 0, sizeof(ot));
    for (int c = 0; c < 91; ++c) ot.col[c][c >> 5] = 1u << (c & 31);
    for (int i = 0; i < 83; ++i)
        for (int w = 0; w < 3; ++w) ot.col[91 + i][w] = FT8_GEN_MASK[i][w];
    e = cudaMemcpyToSymbol(c_osd, &ot, sizeof(ot));
    if (e != cudaSuccess) return e;
    // AP patterns (receiver.py:21-27)
    ApTables ap;
    memset(&ap, 0, sizeof(ap));
    const char* pat[5] = {"", "00000000000000000000000000100", "0111111001110101001", "0111111010010100001", "0111111010010010001"};
    const int first[5] = {0, 0, 58, 58, 58};
    for (int a = 0; a < 5; ++a) {
        ap.first[a] = (int8_t)first[a];
        ap.len[a] = (int8_t)strlen(pat[a]);
        for (int i = 0; i < ap.len[a]; ++i) if (pat[a][i] == '1') ap.mask[a] |= 1u << i;
    }
    e = cudaMemcpyToSymbol(c_ap, &ap, sizeof(ap));
    if (e != cudaSuccess) return e;
    // fine-stage tables
    FineTables ft;
    for (int i = 0; i < 100; ++i) {
        const double x = -M_PI + M_PI * (double)i / 99.0;       // np.linspace(-pi, 0, 100); cos is even so the
        ft.taper[i] = (float)(0.5 * (1.0 + cos(x)));             // (pi, 0) variant of receiver.py:183 is identical
    }
    for (int m = 0; m < 32; ++m) {
        const double a = -2.0 * M_PI * m / 32.0;
        ft.w32[m] = make_float2((float)cos(a), (float)sin(a));
    }
    return cudaMemcpyToSymbol(c_fine, &ft, sizeof(ft));
}

// B operand of k_fscan_mma, laid out exactly as one shared-memory stage per K-chunk: [chunk][split hi/lo][k-chunk 0/1][n][4]
// (see fine_tc.cuh for the formulas; tp is the reference's taper incl. the inverted upper ramp, receiver.py:182-183)
static std::vector<float> fscan_bmat() {
    auto taper = [](int i) { return 0.5 * (1.0 + cos(-M_PI + M_PI * (double)i / 99.0)); };
    auto tp = [&](int k) -> double {
        if (k < -150 || k >= 850) return 0.0;
        if (k < -50) return taper(k + 150);
        if (k < 750) return 1.0;
        return taper(k - 750);
    };
    auto split_hi = [](float v) { uint32_t u; memcpy(&u, &v, 4); u = (u + 0x1000u) & 0xFFFFE000u; float r; memcpy(&r, &u, 4); return r; };
    std::vector<float> out((size_t)FS_BMAT_FLOATS, 0.0f);
    for (int n = 0; n < FS_N; ++n) {
        const int f = n >> 3, t = n & 7;
        const int d = -32 + 8 * (f < 4 ? f : f + 1);
        for (int k = 0; k < FS_K; ++k) {
            double v;
            if (k < FS_K1) {
                const int r = k >> 1;
                const double ang = -2.0 * M_PI * (double)(100 * t + d) * ((double)r - 15.5) / 3200.0;
                v = (k & 1) ? sin(ang) : cos(ang);
            } else {
                const int u = fs_u_of(k - FS_K1);
                const int x = u - d - 100 * t;
                const double dir = x == 0 ? 32.0 : sin(M_PI * x / 100.0) / sin(M_PI * x / 3200.0);
                v = (tp(u - d) - tp(u)) * dir;
            }
            const float vf = (float)v, hi = split_hi(vf), lo = split_hi((float)(v - (double)hi));
            const int chunk = k / FS_KC, kc = (k % FS_KC) / 4, e = k % 4;
            const size_t base = (size_t)chunk * (FS_B_STAGE_BYTES / 4);
            out[base + 0 * (FS_B_SPLIT_BYTES / 4) + kc * (FS_N * 4) + n * 4 + e] = hi;
            out[base + 1 * (FS_B_SPLIT_BYTES / 4) + kc * (FS_N * 4) + n * 4 + e] = lo;
        }
    }
    return out;
}

extern "C" void ft8_default_cfg(ft8_cfg* cfg) {
    if (!cfg) return;
    memset(cfg, 0, sizeof(*cfg));
    cfg->max_cycles = 1;
    cfg->max_cands = 200;
    cfg->sync_score_min = 85.0f;
    cfg->llr_sd_min = 5.0f;
    cfg->osd_singleflips = 30;
    cfg->osd_doubleflips = 2;
    cfg->max_codewords = 1 << 16;
}

extern "C" int ft8_create(int device, const ft8_cfg* cfg_in, ft8_handle** out) {
    if (!out) return fail(nullptr, FT8_E_BADARG, "ft8_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, FT8_E_NODEVICE, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, FT8_E_BADARG, "ft8_create: bad device index");
    ft8_cfg cfg;
    ft8_default_cfg(&cfg);
    if (cfg_in) cfg = *cfg_in;
    if (cfg.max_cycles <= 0) cfg.max_cycles = 1;
    if (cfg.max_cands <= 0) cfg.max_cands = 200;
    if (cfg.max_cands > N_F0) cfg.max_cands = N_F0;
    if (cfg.osd_singleflips < 0 || cfg.osd_singleflips > OSD_MAX_FLIPS || cfg.osd_doubleflips < 0)
        return fail(nullptr, FT8_E_BADARG, "ft8_create: osd flips out of range");
    if (cfg.search_f0_lo == 0 && cfg.search_f0_hi == 0) { cfg.search_f0_lo = F0_LO; cfg.search_f0_hi = F0_LO + N_F0; }
    if (cfg.search_h0_lo == 0 && cfg.search_h0_hi == 0) { cfg.search_h0_lo = H0_LO; cfg.search_h0_hi = H0_LO + N_H0; }
    if (cfg.search_f0_lo < F0_LO || cfg.search_f0_hi > F0_LO + N_F0 || cfg.search_f0_lo >= cfg.search_f0_hi ||
        cfg.search_h0_lo < H0_LO || cfg.search_h0_hi > H0_LO + N_H0 || cfg.search_h0_lo >= cfg.search_h0_hi)
        return fail(nullptr, FT8_E_BADARG, "ft8_create: search range outside what the kernels are built for (f0 in [32, 960), h0 in [-37, 87))");
    if (cfg.fine_mode != 0 && cfg.fine_mode != 1) return fail(nullptr, FT8_E_BADARG, "ft8_create: fine_mode must be 0 (tensor-core scan) or 1 (FFT scan)");
    ft8_handle* h = new ft8_handle();
    h->device = device;
    h->cfg = cfg;
#define CKC(call)                                                                              \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            g_create_error = std::string(#call) + ": " + cudaGetErrorString(e__);              \
            ft8_destroy(h);                                                                    \
            return FT8_E_CUDA;                                                                 \
        }                                                                                      \
    } while (0)
    CKC(cudaSetDevice(device));
    cudaDeviceProp prop;
    CKC(cudaGetDeviceProperties(&prop, device));
    h->n_sm = prop.multiProcessorCount;
    CKC(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    for (auto& ev : h->ev) CKC(cudaEventCreate(&ev));
    for (auto& ev : h->chunk_ev) CKC(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&h->pf_ev, cudaEventDisableTiming));
    CKC(upload_constant_tables());
    {
        std::vector<float> w(NFFT_S);
        for (int i = 0; i < NFFT_S; ++i) {          // np.hanning: 0.5 + 0.5*cos(pi*n/(M-1)), n = 1-M, 3-M, ...
            const double n = (double)(1 - NFFT_S + 2 * i);
            w[i] = (float)(0.5 + 0.5 * cos(M_PI * n / (double)(NFFT_S - 1)));
        }
        CKC(upload(h->d_hann, w));
        CKC(upload(h->d_W1920, twiddles(1920, 1920)));
        CKC(upload(h->d_W3840, twiddles(3840, 1921)));
        CKC(upload(h->d_W3200, twiddles(3200, 3200)));
        CKC(upload(h->d_W375, twiddles(375, 375)));
        CKC(upload(h->d_W256, twiddles(256, 256)));
        CKC(upload(h->d_W192000, twiddles(192000, 96001)));
        CKC(upload(h->d_W32, twiddles(32, 32)));
        {   // per-pass tables (coalesced twiddle loads), one buffer per kernel
            std::vector<float2> ts, tf, tc, t256, w96t;
            append_pass_table(ts, 1920, 15, 1); append_pass_table(ts, 1920, 8, 15);                              // SP_T8_OFF
            append_pass_table(tf, 3200, 5, 1); append_pass_table(tf, 3200, 5, 5); append_pass_table(tf, 3200, 8, 25);   // FINE_T*_OFF
            append_pass_table(tc, 375, 3, 1); append_pass_table(tc, 375, 5, 3); append_pass_table(tc, 375, 5, 15);
            append_pass_table(t256, 256, 16, 1);
            w96t.reserve((size_t)CS_N1 * CS_N2);
            for (int k1 = 0; k1 < CS_N1; ++k1)
                for (int n2 = 0; n2 < CS_N2; ++n2) w96t.push_back(twiddle1(96000, (long long)n2 * k1));
            if ((int)ts.size() != SP_T8_OFF + 7 * 16 || (int)tf.size() != FINE_TF_LEN || (int)tc.size() != 370) { ft8_destroy(h); return fail(nullptr, FT8_E_CUDA, "twiddle table layout"); }
            CKC(upload(h->d_TS, ts)); CKC(upload(h->d_TF, tf)); CKC(upload(h->d_TC, tc)); CKC(upload(h->d_T256, t256));
            CKC(upload(h->d_W96000T, w96t));
        }
        CKC(upload(h->d_pulse, synth_pulse_table()));
        CKC(upload(h->d_bmat, fscan_bmat()));
        {
            std::vector<float2> w(FS_W_LEN);
            for (int g = 0; g < FS_W_LEN; ++g) { const double a = 2.0 * M_PI * (double)g / (double)FS_W_LEN; w[g] = make_float2((float)cos(a), (float)sin(a)); }
            CKC(upload(h->d_w6400, w));
        }
    }
    const size_t B = (size_t)cfg.max_cycles, K = (size_t)cfg.max_cands, N = B * K;
    h->cap_cycles = B;
    h->cap_slots = N;
    CKC(h->d_grid.ensure(B * GRID_ROWS * GRID_COLS));
    // four-step scratch Y: 768 KB per cycle, written by k_cs_cols and read back by k_cs_rows, in chunks of up to 1024 cycles.
    // Smaller, L2-resident chunks (VERDICT r1 item 7) were measured and are SLOWER: 3.18 ms per 4096 cycles at 1024, 3.50 at 256,
    // 3.88 at 128, 4.20 at 64, 5.00 at 32 (profiles/r02_experiments.md) -- both kernels sit on the L1/shared data pipe, not on
    // HBM, so the 3x DRAM traffic costs nothing while small grids lose to tail effects.
    h->y_cycles = std::min<size_t>(B, 1024);
    CKC(h->d_Y.ensure(h->y_cycles * CS_N));
    CKC(h->d_spec.ensure(B * FINE_SPEC_STRIDE));
    CKC(h->d_best_score.ensure(B * N_F0 * SY_HS));
    CKC(h->d_best_h0.ensure(B * N_F0 * SY_HS));
    CKC(h->d_f0.ensure(N)); CKC(h->d_h0.ensure(N)); CKC(h->d_score.ensure(N)); CKC(h->d_ncand.ensure(B));
    CKC(h->d_status.ensure(N)); CKC(h->d_llr_grid.ensure(N * 174)); CKC(h->d_grid_sd.ensure(N)); CKC(h->d_grid_snr.ensure(N));
    CKC(h->d_llr_fine.ensure(N * 174)); CKC(h->d_fine.ensure(N)); CKC(h->d_saved.ensure(N * 5 * 174));
    CKC(h->d_saved_n.ensure(N)); CKC(h->d_saved_ap.ensure(N * 5)); CKC(h->d_bits.ensure(N * 3));
    CKC(h->d_ripass.ensure(N)); CKC(h->d_rap.ensure(N)); CKC(h->d_rmethod.ensure(N)); CKC(h->d_rnits.ensure(N));
    CKC(h->d_osd_found.ensure(N * 10)); CKC(h->d_osd_bits.ensure(N * 30));
    CKC(h->d_list_fine.ensure(N)); CKC(h->d_list_osd.ensure(N)); CKC(h->d_counts.ensure(CNT_SLOTS));
    CKC(h->d_stats.ensure(1)); CKC(h->d_rec.ensure(N)); CKC(h->d_rec_n.ensure(B)); CKC(h->d_rec_base.ensure(B));
    CKC(cudaMallocHost((void**)&h->h_counts, CNT_SLOTS * sizeof(int32_t)));
    CKC(cudaMallocHost((void**)&h->h_stats, sizeof(DevStats)));
    {
        std::vector<int32_t> co(N);
        for (size_t i = 0; i < N; ++i) co[i] = (int32_t)(i / K);
        CKC(upload(h->d_cycle_of, co));
    }
    CKC(cudaFuncSetAttribute(k_fine, cudaFuncAttributeMaxDynamicSharedMemorySize, FINE_SMEM_BYTES));
    CKC(cudaFuncSetAttribute(k_fine_tscan, cudaFuncAttributeMaxDynamicSharedMemorySize, FT_SMEM_BYTES));
    CKC(cudaFuncSetAttribute(k_fine_final, cudaFuncAttributeMaxDynamicSharedMemorySize, FF_SMEM_BYTES));
    CKC(cudaFuncSetAttribute(k_fscan_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, FS_SMEM_BYTES));
    if (cfg.fine_mode == 0) {
        CKC(h->d_zwin.ensure(N * FS_WIN)); CKC(h->d_tso.ensure(N)); CKC(h->d_ff.ensure(N)); CKC(h->d_amb.ensure(N + 1));
    }
    {
        const int sp_smem = SP_BUF_LEN * (int)sizeof(float2);
        CKC(cudaFuncSetAttribute(k_spectrogram<int16_t, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sp_smem));
        CKC(cudaFuncSetAttribute(k_spectrogram<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, sp_smem));
        CKC(cudaFuncSetAttribute(k_spectrogram<int16_t, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sp_smem));
        CKC(cudaFuncSetAttribute(k_spectrogram<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, sp_smem));
    }
    CKC(cudaFuncSetAttribute(k_sync_scores, cudaFuncAttributeMaxDynamicSharedMemorySize, SY_SMEM_BYTES));
    CKC(cudaDeviceSynchronize());
#undef CKC
    *out = h;
    return FT8_OK;
}

extern "C" void ft8_destroy(ft8_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->copy_stream) cudaStreamSynchronize(h->copy_stream);
    for (auto& ev : h->ev) if (ev) cudaEventDestroy(ev);
    for (auto& ev : h->chunk_ev) if (ev) cudaEventDestroy(ev);
    if (h->pf_ev) cudaEventDestroy(h->pf_ev);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->stream) cudaStreamDestroy(h->stream);
    if (h->h_counts) cudaFreeHost(h->h_counts);
    if (h->h_stats) cudaFreeHost(h->h_stats);
    delete h;                        // frees the device buffers
}

extern "C" const char* ft8_last_error(ft8_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }
extern "C" void* ft8_stream(ft8_handle* h) { return h ? (void*)h->stream : nullptr; }
extern "C" int ft8_host_alloc(size_t bytes, int flags, void** out) {
    if (!out || bytes == 0) return FT8_E_BADARG;
    *out = nullptr;
    unsigned f = cudaHostAllocPortable;
    if (flags & FT8_HOST_WRITE_COMBINED) f |= cudaHostAllocWriteCombined;
    if (cudaHostAlloc(out, bytes, f) != cudaSuccess) { cudaGetLastError(); *out = nullptr; return FT8_E_CUDA; }
    return FT8_OK;
}
extern "C" int ft8_host_free(void* p) {
    if (!p) return FT8_OK;
    if (cudaFreeHost(p) != cudaSuccess) { cudaGetLastError(); return FT8_E_CUDA; }
    return FT8_OK;
}
extern "C" int ft8_synchronize(ft8_handle* h) {
    if (!h) return FT8_E_BADARG;
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return FT8_OK;
}
extern "C" int ft8_get_stats(ft8_handle* h, ft8_stats* out) {
    if (!h || !out) return FT8_E_BADARG;
    *out = h->stats;
    return FT8_OK;
}
extern "C" int ft8_last_kernel_ms(ft8_handle* h, int which, float* ms) {
    if (!h || !ms || which < 0 || which >= MS_COUNT) return FT8_E_BADARG;
    *ms = h->last_ms[which];
    return FT8_OK;
}

// ------------------------------------------------------------------------------------------ launch helpers
static CandState cand_state(ft8_handle* h) {
    CandState cs;
    cs.K = h->cfg.max_cands; cs.n_cand = h->d_ncand; cs.f0 = h->d_f0; cs.h0 = h->d_h0; cs.score = h->d_score;
    cs.status = h->d_status; cs.llr_grid = h->d_llr_grid; cs.grid_sd = h->d_grid_sd; cs.grid_snr = h->d_grid_snr;
    cs.llr_fine = h->d_llr_fine; cs.fine = h->d_fine; cs.saved_llr = h->d_saved; cs.saved_n = h->d_saved_n;
    cs.saved_ap = h->d_saved_ap; cs.bits91 = h->d_bits; cs.r_ipass = h->d_ripass; cs.r_ap = h->d_rap;
    cs.r_method = h->d_rmethod; cs.r_nits = h->d_rnits; cs.osd_found = h->d_osd_found; cs.osd_bits = h->d_osd_bits;
    return cs;
}

static int launch_spectrogram(ft8_handle* h, const void* d_audio, int dtype, int B, float* d_grid, int row_lo = 1,
                              int row_hi = 375, int out_rows = GRID_ROWS, int out_row0 = 0, int fill_row0 = 1,
                              const float* d_prev_tail = nullptr, int out_wrap = 0) {
    const bool ring = d_prev_tail != nullptr || out_wrap != 0;
    dim3 grid(row_hi - row_lo + 1, B);
    const int smem = SP_BUF_LEN * (int)sizeof(float2);
#define SP_LAUNCH(T, RING)                                                                                                          \
    k_spectrogram<T, RING><<<grid, SP_NT, smem, h->stream>>>((const T*)d_audio, d_grid, h->d_hann, h->d_TS, h->d_W3840, row_lo, \
                                                             row_hi, out_rows, out_row0, fill_row0, d_prev_tail, out_wrap)
    if (dtype == FT8_AUDIO_I16) { if (ring) SP_LAUNCH(int16_t, true); else SP_LAUNCH(int16_t, false); }
    else { if (ring) SP_LAUNCH(float, true); else SP_LAUNCH(float, false); }
#undef SP_LAUNCH
    CK(cudaGetLastError());
    return FT8_OK;
}

// d_grid points at the first of the B cycles; b0 = index of that cycle in the handle's per-cycle arrays; cycle_h0 = grid row
// of the cycle's hop 0
static int launch_sync(ft8_handle* h, const float* d_grid, int grid_rows, int B, int cycle_h0, int b0 = 0) {
    const size_t K = h->cfg.max_cands;
    k_sync_scores<<<dim3(SY_HS * (N_F0 / SY_TF), B), SY_NT, SY_SMEM_BYTES, h->stream>>>(
        d_grid, grid_rows, cycle_h0, h->d_best_score + (size_t)b0 * N_F0 * SY_HS, h->d_best_h0 + (size_t)b0 * N_F0 * SY_HS,
        h->cfg.search_h0_lo, h->cfg.search_h0_hi);
    CK(cudaGetLastError());
    k_topk<<<B, 960, 0, h->stream>>>(h->d_best_score + (size_t)b0 * N_F0 * SY_HS, h->d_best_h0 + (size_t)b0 * N_F0 * SY_HS, h->cfg.sync_score_min,
                                     h->cfg.max_cands, h->d_f0 + b0 * K, h->d_h0 + b0 * K, h->d_score + b0 * K, h->d_ncand + b0,
                                     h->cfg.search_f0_lo, h->cfg.search_f0_hi);
    CK(cudaGetLastError());
    return FT8_OK;
}

// cycle spectra for B cycles into spec[B][stride], processed in chunks bounded by the Y scratch
static int launch_cycle_spectrum(ft8_handle* h, const void* d_audio, int dtype, int B, float2* d_spec, int stride, int kmax) {
    const size_t esz = dtype == FT8_AUDIO_I16 ? 2 : 4;
    for (int b0 = 0; b0 < B; b0 += (int)h->y_cycles) {
        const int nb = std::min<int>((int)h->y_cycles, B - b0);
        const char* a = (const char*)d_audio + (size_t)b0 * CYCLE_SAMPLES * esz;
        const int smem = CS_COLS * CS_N1 * (int)sizeof(float2);
        if (dtype == FT8_AUDIO_I16)
            k_cs_cols<int16_t><<<dim3(CS_N2 / CS_COLS, nb), CS_NT, smem, h->stream>>>((const int16_t*)a, h->d_Y, h->d_TC, h->d_W96000T);
        else
            k_cs_cols<float><<<dim3(CS_N2 / CS_COLS, nb), CS_NT, smem, h->stream>>>((const float*)a, h->d_Y, h->d_TC, h->d_W96000T);
        CK(cudaGetLastError());
        k_cs_rows<<<dim3(24, nb), CS_NT, 0, h->stream>>>(h->d_Y, d_spec + (size_t)b0 * stride, stride, kmax, h->d_T256, h->d_W192000);
        CK(cudaGetLastError());
    }
    return FT8_OK;
}

static int persistent_blocks(ft8_handle* h, int per_sm) { return h->n_sm * per_sm; }

// F2/F3 for a work list (list/count on the device, at most cap_slots items) or for items 0..n_direct-1 (list == nullptr).
// fine_mode 0: time scan -> tensor-core frequency scan -> final transform (fine_tc.cuh); 1: the literal 9-transform kernel.
static int launch_fine(ft8_handle* h, const float2* spec, int spec_stride, const int32_t* list, const int32_t* count, int n_direct,
                       const int32_t* cycle_of, const int16_t* f0, const int16_t* h0, FineOut* fo, float* llr, float* sig_grid) {
    if (h->cfg.fine_mode == 1) {
        const int blocks = list ? persistent_blocks(h, 4) : std::min(persistent_blocks(h, 4), n_direct);
        k_fine<<<blocks, FINE_NT, FINE_SMEM_BYTES, h->stream>>>(spec, spec_stride, list, count, n_direct, cycle_of, f0, h0, h->d_TF, fo, llr, sig_grid);
        CK(cudaGetLastError());
        return FT8_OK;
    }
    const size_t need = list ? h->cap_slots : (size_t)n_direct;
    CK(h->d_zwin.ensure(need * FS_WIN, h->stream)); CK(h->d_tso.ensure(need, h->stream)); CK(h->d_ff.ensure(need, h->stream));
    CK(h->d_amb.ensure(need + 1, h->stream));
    const int nbt = list ? persistent_blocks(h, FT_CTAS) : std::min(persistent_blocks(h, FT_CTAS), n_direct);
    const int nb3 = list ? persistent_blocks(h, FF_CTAS) : std::min(persistent_blocks(h, FF_CTAS), n_direct);
    k_fine_tscan<<<nbt, FT_NT, FT_SMEM_BYTES, h->stream>>>(spec, spec_stride, list, count, n_direct, cycle_of, f0, h0, h->d_TF, h->d_tso, h->d_zwin);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev[EV_TSCAN_END], h->stream));
    const int nb1 = list ? h->n_sm : std::min(h->n_sm, (n_direct + FS_CAND - 1) / FS_CAND);
    CK(cudaMemsetAsync(h->d_amb, 0, sizeof(int32_t), h->stream));
    k_fscan_mma<<<nb1, FS_NT, FS_SMEM_BYTES, h->stream>>>(spec, spec_stride, list, count, n_direct, cycle_of, f0, h0, h->d_tso, h->d_zwin,
                                                         h->d_bmat, h->d_w6400, h->d_ff, h->d_amb + 1, h->d_amb);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev[EV_FSCAN_END], h->stream));
    k_fine_final<<<nb3, FT_NT, FF_SMEM_BYTES, h->stream>>>(spec, spec_stride, list, count, n_direct, cycle_of, f0, h0, h->d_TF, h->d_tso, h->d_ff,
                                                            fo, llr, sig_grid);
    CK(cudaGetLastError());
    // near-tie candidates of the frequency scan: decided by the literal nine-transform kernel (overwrites their results)
    k_fine<<<persistent_blocks(h, 2), FINE_NT, FINE_SMEM_BYTES, h->stream>>>(spec, spec_stride, h->d_amb + 1, h->d_amb, 0, cycle_of, f0, h0, h->d_TF, fo, llr, sig_grid);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->d_counts + CNT_NEAR_TIE, h->d_amb, sizeof(int32_t), cudaMemcpyDeviceToDevice, h->stream));
    return FT8_OK;
}
static int fine_launches(ft8_handle* h) { return h->cfg.fine_mode == 1 ? 1 : 4; }

#define ENTER(h)                                  \
    if (!(h)) return FT8_E_BADARG;                \
    CK(cudaSetDevice((h)->device));
#define TRY(x) do { int r__ = (x); if (r__ != FT8_OK) return r__; } while (0)

static int check_dtype(ft8_handle* h, int dtype) {
    if (dtype != FT8_AUDIO_I16 && dtype != FT8_AUDIO_F32) return fail(h, FT8_E_BADARG, "audio_dtype must be FT8_AUDIO_I16 or FT8_AUDIO_F32");
    return FT8_OK;
}
static size_t sample_bytes(int dtype) { return dtype == FT8_AUDIO_I16 ? 2 : 4; }

// Caller buffers of one stand-alone op.  With FT8_MEM_DEVICE a caller buffer is used in place; with FT8_MEM_HOST it gets a
// slice of the handle's arena: begin() copies the inputs in and finish() copies the outputs back before its final
// synchronise.  Scratch is always a slice of the arena.  begin() sizes the arena from the declarations and grows it, which
// frees the old arena, so every buffer is declared before begin() and the declared pointers are set by it.  A NULL caller
// buffer (an optional output) stays NULL.
class Staging {
  public:
    Staging(ft8_handle* h, int mem) : h_(h), host_(mem == FT8_MEM_HOST) {}
    template <typename T> void in(const T*& dev, const void* user, size_t bytes) { add(dev, user, bytes, true, false); }
    template <typename T> void out(T*& dev, void* user, size_t bytes) { add(dev, user, bytes, false, true); }
    template <typename T> void inout(T*& dev, void* user, size_t bytes) { add(dev, user, bytes, true, true); }
    template <typename T> void scratch(T*& dev, size_t bytes) { add(dev, nullptr, bytes, false, false); }

    int begin() {
        ft8_handle* h = h_;
        CK(h->arena.ensure(bytes_, h->stream));
        for (const Slot& s : slots_) {
            char* p = h->arena + s.off;
            memcpy(s.dev, &p, sizeof(p));
            if (s.in) CK(cudaMemcpyAsync(p, s.user, s.bytes, cudaMemcpyHostToDevice, h->stream));
        }
        return FT8_OK;
    }
    int finish() {
        ft8_handle* h = h_;
        for (const Slot& s : slots_)
            if (s.out) CK(cudaMemcpyAsync((void*)s.user, h->arena + s.off, s.bytes, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return FT8_OK;
    }

  private:
    struct Slot { void* dev; const void* user; size_t off, bytes; bool in, out; };
    template <typename P> void add(P& dev, const void* user, size_t bytes, bool in, bool out) {
        if ((in || out) && (!host_ || !user)) { dev = (P)user; return; }
        const size_t off = (bytes_ + 255) & ~(size_t)255;
        slots_.push_back({&dev, user, off, bytes, in, out});
        bytes_ = off + bytes;
    }
    ft8_handle* h_;
    bool host_;
    std::vector<Slot> slots_;
    size_t bytes_ = 0;
};

// copy of a handle-owned device array to a caller buffer
static int from_device(ft8_handle* h, void* dst, const void* d, size_t bytes, int mem) {
    CK(cudaMemcpyAsync(dst, d, bytes, mem == FT8_MEM_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, h->stream));
    return FT8_OK;
}

// ------------------------------------------------------------------------------------------ stage ops
extern "C" int ft8_spectrogram(ft8_handle* h, const void* audio, int audio_dtype, int B, float* grid_db, int mem) {
    ENTER(h);
    if (!audio || !grid_db || B <= 0) return fail(h, FT8_E_BADARG, "ft8_spectrogram: bad argument");
    if ((size_t)B > h->cap_cycles) return fail(h, FT8_E_CAPACITY, "ft8_spectrogram: B exceeds cfg.max_cycles");
    TRY(check_dtype(h, audio_dtype));
    const char* da; float* dg;
    Staging st(h, mem);
    st.in(da, audio, (size_t)B * CYCLE_SAMPLES * sample_bytes(audio_dtype));
    st.out(dg, grid_db, (size_t)B * GRID_ROWS * GRID_COLS * sizeof(float));
    TRY(st.begin());
    CK(cudaEventRecord(h->ev[EV_OP_BEGIN], h->stream));
    TRY(launch_spectrogram(h, da, audio_dtype, B, dg));
    CK(cudaEventRecord(h->ev[EV_OP_END], h->stream));
    TRY(st.finish());
    CK(cudaEventElapsedTime(&h->last_ms[MS_SPECTROGRAM], h->ev[EV_OP_BEGIN], h->ev[EV_OP_END]));
    return FT8_OK;
}

extern "C" int ft8_hop_spectrum(ft8_handle* h, const void* audio_buffer, int audio_dtype, float* row_db, int mem) {
    ENTER(h);
    if (!audio_buffer || !row_db) return fail(h, FT8_E_BADARG, "ft8_hop_spectrum: bad argument");
    TRY(check_dtype(h, audio_dtype));
    const size_t esz = sample_bytes(audio_dtype);
    const void* da = audio_buffer;
    if (mem == FT8_MEM_HOST) {
        // only the last 3840 samples are read (receiver.py:289): stage those 15 KB at their place in a cycle-sized buffer,
        // not the whole 720 KB ring, every 40 ms hop
        CK(h->d_audio.ensure((size_t)CYCLE_SAMPLES * esz, h->stream));
        const size_t off = (size_t)(CYCLE_SAMPLES - NFFT_S) * esz;
        CK(cudaMemcpyAsync(h->d_audio + off, (const char*)audio_buffer + off, (size_t)NFFT_S * esz, cudaMemcpyHostToDevice, h->stream));
        da = h->d_audio;
    }
    float* dr;
    Staging st(h, mem);
    st.out(dr, row_db, GRID_COLS * sizeof(float));
    TRY(st.begin());
    // the window over the last 3840 samples of a 180000-sample buffer is row 375 of that buffer's waterfall
    TRY(launch_spectrogram(h, da, audio_dtype, 1, dr, 375, 375, 1, 375, 0));
    return st.finish();
}

extern "C" int ft8_sync(ft8_handle* h, const float* grid_db, int grid_rows, int B, int odd_even, int16_t* cand_f0,
                        int16_t* cand_h0, float* cand_score, int32_t* n_cand, float* payload_db, int mem) {
    ENTER(h);
    if (!grid_db || !cand_f0 || !cand_h0 || !cand_score || !n_cand || B <= 0) return fail(h, FT8_E_BADARG, "ft8_sync: bad argument");
    if (grid_rows != GRID_ROWS && grid_rows != LIVE_ROWS) return fail(h, FT8_E_BADARG, "ft8_sync: grid_rows must be 376 or 750");
    if ((size_t)B > h->cap_cycles) return fail(h, FT8_E_CAPACITY, "ft8_sync: B exceeds cfg.max_cycles");
    if (payload_db && mem == FT8_MEM_HOST && grid_rows != GRID_ROWS)
        return fail(h, FT8_E_BADARG, "ft8_sync: payload_db with a host 750-row grid is not supported; pass grid_rows=376 or device memory");
    const size_t K = h->cfg.max_cands, N = (size_t)B * K;
    const float* dg; float* d_pay;
    Staging st(h, mem);
    st.in(dg, grid_db, (size_t)B * grid_rows * GRID_COLS * sizeof(float));
    st.out(d_pay, payload_db, N * 58 * 8 * sizeof(float));
    TRY(st.begin());
    CK(cudaMemsetAsync(h->d_f0, 0, N * 2, h->stream));
    CK(cudaMemsetAsync(h->d_h0, 0, N * 2, h->stream));
    CK(cudaMemsetAsync(h->d_score, 0, N * 4, h->stream));
    CK(cudaEventRecord(h->ev[EV_OP_BEGIN], h->stream));
    TRY(launch_sync(h, dg, grid_rows, B, odd_even ? 375 : 0));
    CK(cudaEventRecord(h->ev[EV_OP_END], h->stream));
    if (payload_db) {
        CK(cudaMemsetAsync(d_pay, 0, N * 58 * 8 * sizeof(float), h->stream));
        CK(cudaMemsetAsync(h->d_stats, 0, sizeof(DevStats), h->stream));
        CK(cudaMemsetAsync(h->d_counts, 0, CNT_SLOTS * sizeof(int32_t), h->stream));
        k_pass0<<<persistent_blocks(h, 8), WARPS_PER_CTA * 32, sizeof(PassSmem), h->stream>>>(
            cand_state(h), (int)N, dg, grid_rows, odd_even ? 375 : 0, h->cfg.llr_sd_min, d_pay, 1, h->d_list_fine,
            h->d_counts + CNT_FINE, h->d_counts + CNT_CURSOR_PASS0, h->d_stats);
        CK(cudaGetLastError());
    }
    TRY(from_device(h, cand_f0, h->d_f0, N * 2, mem));
    TRY(from_device(h, cand_h0, h->d_h0, N * 2, mem));
    TRY(from_device(h, cand_score, h->d_score, N * 4, mem));
    TRY(from_device(h, n_cand, h->d_ncand, (size_t)B * 4, mem));
    TRY(st.finish());
    CK(cudaEventElapsedTime(&h->last_ms[MS_SYNC], h->ev[EV_OP_BEGIN], h->ev[EV_OP_END]));
    return FT8_OK;
}

extern "C" int ft8_llr(ft8_handle* h, const float* payload_db, int N, float* llr, float* sd, int32_t* snr, int mem) {
    ENTER(h);
    if (!payload_db || !llr || !sd || !snr || N <= 0) return fail(h, FT8_E_BADARG, "ft8_llr: bad argument");
    const float* dp; float *dl, *ds; int32_t* dn;
    Staging st(h, mem);
    st.in(dp, payload_db, (size_t)N * 464 * 4);
    st.out(dl, llr, (size_t)N * 174 * 4); st.out(ds, sd, (size_t)N * 4); st.out(dn, snr, (size_t)N * 4);
    TRY(st.begin());
    k_llr_batch<<<std::min(persistent_blocks(h, 8), (N + WARPS_PER_CTA - 1) / WARPS_PER_CTA), WARPS_PER_CTA * 32, 0, h->stream>>>(dp, N, dl, ds, dn);
    CK(cudaGetLastError());
    return st.finish();
}

extern "C" int ft8_cycle_spectrum(ft8_handle* h, const void* audio, int audio_dtype, int B, float* spec, int mem) {
    ENTER(h);
    if (!audio || !spec || B <= 0) return fail(h, FT8_E_BADARG, "ft8_cycle_spectrum: bad argument");
    if ((size_t)B > h->cap_cycles) return fail(h, FT8_E_CAPACITY, "ft8_cycle_spectrum: B exceeds cfg.max_cycles");
    TRY(check_dtype(h, audio_dtype));
    const char* da; float2* ds;
    Staging st(h, mem);
    st.in(da, audio, (size_t)B * CYCLE_SAMPLES * sample_bytes(audio_dtype));
    st.out(ds, spec, (size_t)B * FT8_SPEC_BINS * sizeof(float2));
    TRY(st.begin());
    TRY(launch_cycle_spectrum(h, da, audio_dtype, B, ds, FT8_SPEC_BINS, FT8_SPEC_BINS - 1));
    return st.finish();
}

// ft8_fine helpers: range check of caller-supplied candidates on the device (works for host and device callers alike)
// and the split of FineOut into the ABI's plain arrays.
__global__ void k_fine_validate(const int32_t* __restrict__ cycle_of, const int16_t* __restrict__ f0, const int16_t* __restrict__ h0,
                                int N, int B, int32_t* __restrict__ bad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N && (h0[i] < -100 || h0[i] > 200 || f0[i] < 4 || f0[i] > 1880 || cycle_of[i] < 0 || cycle_of[i] >= B)) atomicAdd(bad, 1);
}
__global__ void k_fine_unpack(const FineOut* __restrict__ fo, int N, int32_t* __restrict__ tt, int32_t* __restrict__ ff,
                              int32_t* __restrict__ ns, float* __restrict__ sd, int32_t* __restrict__ snr) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < N) { const FineOut o = fo[i]; tt[i] = o.tt; ff[i] = o.ff; ns[i] = o.nsync; sd[i] = o.sd; snr[i] = o.snr; }
}

extern "C" int ft8_fine(ft8_handle* h, const float* spec, int B, const int32_t* cycle_of, const int16_t* f0_idx,
                        const int16_t* h0_idx, int N, int32_t* ttweak, int32_t* ftweak, int32_t* nsync, float* signal_grid,
                        float* llr, float* sd, int32_t* snr, int mem) {
    ENTER(h);
    if (!spec || !cycle_of || !f0_idx || !h0_idx || !ttweak || !ftweak || !nsync || !llr || !sd || !snr || N <= 0 || B <= 0)
        return fail(h, FT8_E_BADARG, "ft8_fine: bad argument");
    const float2* sp; const int32_t* dco; const int16_t *df0, *dh0; FineOut* dfo;
    int32_t *dtt, *dff, *dns, *dsn; float *dsd, *dllr, *dsg;
    Staging st(h, mem);
    st.in(sp, spec, (size_t)B * FT8_SPEC_BINS * sizeof(float2));
    st.in(dco, cycle_of, (size_t)N * 4); st.in(df0, f0_idx, (size_t)N * 2); st.in(dh0, h0_idx, (size_t)N * 2);
    st.scratch(dfo, (size_t)N * sizeof(FineOut));
    st.out(dtt, ttweak, (size_t)N * 4); st.out(dff, ftweak, (size_t)N * 4); st.out(dns, nsync, (size_t)N * 4);
    st.out(dsd, sd, (size_t)N * 4); st.out(dsn, snr, (size_t)N * 4);
    st.out(dllr, llr, (size_t)N * 174 * 4); st.out(dsg, signal_grid, (size_t)N * 632 * 4);
    TRY(st.begin());
    // candidates are range-checked on the device before anything gathers with them (host AND device callers)
    CK(cudaMemsetAsync(h->d_counts + CNT_FINE_BAD, 0, 4, h->stream));
    k_fine_validate<<<(N + 255) / 256, 256, 0, h->stream>>>(dco, df0, dh0, N, B, h->d_counts + CNT_FINE_BAD);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(h->h_counts + CNT_FINE_BAD, h->d_counts + CNT_FINE_BAD, 4, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (h->h_counts[CNT_FINE_BAD] != 0)
        return fail(h, FT8_E_BADARG, "ft8_fine: candidate outside the supported range (-100 <= h0 <= 200, 4 <= f0 <= 1880, 0 <= cycle_of < B)");
    TRY(launch_fine(h, sp, FT8_SPEC_BINS, nullptr, nullptr, N, dco, df0, dh0, dfo, dllr, dsg));
    k_fine_unpack<<<(N + 255) / 256, 256, 0, h->stream>>>(dfo, N, dtt, dff, dns, dsd, dsn);
    CK(cudaGetLastError());
    return st.finish();
}

extern "C" int ft8_ldpc(ft8_handle* h, float* llr, int N, int max_ncheck0, int max_iters, int32_t* status, int32_t* nits,
                        uint32_t* bits91, int mem) {
    ENTER(h);
    if (!llr || !status || !nits || !bits91 || N <= 0 || max_iters < 0) return fail(h, FT8_E_BADARG, "ft8_ldpc: bad argument");
    float* dl; int32_t *dst, *dn; uint32_t* db;
    Staging st(h, mem);
    st.inout(dl, llr, (size_t)N * 174 * 4);
    st.out(dst, status, (size_t)N * 4); st.out(dn, nits, (size_t)N * 4); st.out(db, bits91, (size_t)N * 12);
    TRY(st.begin());
    CK(cudaEventRecord(h->ev[EV_OP_BEGIN], h->stream));
    k_ldpc_batch<<<std::min(persistent_blocks(h, 8), (N + WARPS_PER_CTA - 1) / WARPS_PER_CTA), WARPS_PER_CTA * 32, sizeof(PassSmem), h->stream>>>(
        dl, N, max_ncheck0, max_iters, dst, dn, db);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev[EV_OP_END], h->stream));
    TRY(st.finish());
    CK(cudaEventElapsedTime(&h->last_ms[MS_TOTAL], h->ev[EV_OP_BEGIN], h->ev[EV_OP_END]));
    return FT8_OK;
}

extern "C" int ft8_osd(ft8_handle* h, const float* llr, int N, int singleflips, int doubleflips, int32_t* found,
                       uint32_t* bits91, int mem) {
    ENTER(h);
    if (!llr || !found || !bits91 || N <= 0 || singleflips < 0 || singleflips > OSD_MAX_FLIPS || doubleflips < 0)
        return fail(h, FT8_E_BADARG, "ft8_osd: bad argument (singleflips must be 0..91)");
    const float* dl; int32_t* df; uint32_t* db;
    Staging st(h, mem);
    st.in(dl, llr, (size_t)N * 174 * 4);
    st.out(df, found, (size_t)N * 4); st.out(db, bits91, (size_t)N * 12);
    TRY(st.begin());
    CK(cudaEventRecord(h->ev[EV_OP_BEGIN], h->stream));
    k_osd_batch<<<std::min(persistent_blocks(h, 8), (N + WARPS_PER_CTA - 1) / WARPS_PER_CTA), WARPS_PER_CTA * 32, sizeof(OsdSmem), h->stream>>>(
        dl, N, singleflips, doubleflips, df, db);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev[EV_OP_END], h->stream));
    TRY(st.finish());
    CK(cudaEventElapsedTime(&h->last_ms[MS_TOTAL], h->ev[EV_OP_BEGIN], h->ev[EV_OP_END]));
    return FT8_OK;
}

extern "C" int ft8_crc14(ft8_handle* h, const uint32_t* bits91, int N, int32_t* flags, int mem) {
    ENTER(h);
    if (!bits91 || !flags || N <= 0) return fail(h, FT8_E_BADARG, "ft8_crc14: bad argument");
    const uint32_t* db; int32_t* df;
    Staging st(h, mem);
    st.in(db, bits91, (size_t)N * 12);
    st.out(df, flags, (size_t)N * 4);
    TRY(st.begin());
    k_crc_batch<<<std::min(persistent_blocks(h, 8), (N + 127) / 128), 128, 0, h->stream>>>(db, N, df);
    CK(cudaGetLastError());
    return st.finish();
}

// ------------------------------------------------------------------------------------------ whole path
extern "C" int ft8_prefetch_audio(ft8_handle* h, const void* audio_host, int audio_dtype, int B) {
    ENTER(h);
    if (!audio_host || B <= 0 || (audio_dtype != FT8_AUDIO_I16 && audio_dtype != FT8_AUDIO_F32))
        return fail(h, FT8_E_BADARG, "ft8_prefetch_audio: bad argument");
    if ((size_t)B > h->cap_cycles) return fail(h, FT8_E_CAPACITY, "ft8_prefetch_audio: B exceeds cfg.max_cycles");
    const size_t bytes = (size_t)B * CYCLE_SAMPLES * sample_bytes(audio_dtype);
    CK(h->d_audio_pf.ensure(bytes, h->copy_stream, h->stream));
    // the slot may still be read by kernels of the call that consumed the previous prefetch (same stream order)
    CK(cudaEventRecord(h->pf_ev, h->stream));
    CK(cudaStreamWaitEvent(h->copy_stream, h->pf_ev, 0));
    CK(cudaMemcpyAsync(h->d_audio_pf, audio_host, bytes, cudaMemcpyHostToDevice, h->copy_stream));
    CK(cudaEventRecord(h->pf_ev, h->copy_stream));
    h->pf_host = audio_host; h->pf_B = B; h->pf_dtype = audio_dtype;
    return FT8_OK;
}

// the previous cycle's last 3840 samples per stream, kept for the next live call as float32: int16 -> float is exact, so
// the next call reads the same values whichever dtype either call was given
template <typename T>
__global__ void k_save_tails(const T* __restrict__ audio, float* __restrict__ tail) {
    const T* x = audio + (size_t)blockIdx.x * CYCLE_SAMPLES + (CYCLE_SAMPLES - NFFT_S);
    float* t = tail + (size_t)blockIdx.x * NFFT_S;
    for (int i = threadIdx.x; i < NFFT_S; i += blockDim.x) t[i] = (float)x[i];
}

static int save_tails(ft8_handle* h, const void* d_audio, int dtype, int B, float* d_tail) {
    if (dtype == FT8_AUDIO_I16) k_save_tails<<<B, 256, 0, h->stream>>>((const int16_t*)d_audio, d_tail);
    else k_save_tails<<<B, 256, 0, h->stream>>>((const float*)d_audio, d_tail);
    CK(cudaGetLastError());
    return FT8_OK;
}

// Consecutive live cycles (ft8_decode_cycles_live_seq) are decoded in pieces: `steps` cycle steps of `streams` streams, one
// batch of steps * streams cycles, cycle i = step * streams + stream, the first step of parity `parity`.  Each cycle gets a
// SEQ_ROWS-row grid: rows 0..5 are the previous cycle's hops 370..375, rows 6..380 its own hops 1..375.  The search runs on
// it with cycle_h0 = SEQ_H0, so row SEQ_H0 + d holds what the live ring holds at 375 p + d: the sync search reads d in
// 111..258, payload rows d = h0 + 4 + 4 s lie in [-5, 374], and d <= 0 is the previous cycle's hop 375 + d.
struct SeqPiece { int streams, steps, parity; };
constexpr int SEQ_BOUND = 6, SEQ_H0 = SEQ_BOUND - 1, SEQ_ROWS = SEQ_BOUND + 375;
constexpr int ROW_F4 = GRID_COLS / 4;           // a grid row as float4 (3904 bytes: every row starts 16-byte aligned)

// Rows 0..5 of cycles b0 .. b0 + gridDim.y - 1 of a piece: for a cycle after the piece's first step, rows 375..380 of the same
// stream's cycle one step earlier (its hops 370..375); for the first step, the ring rows (375 p + d) mod 750, d = -5..0, that
// a live call of parity p reads there.  Runs after S1 has written the own rows of those cycles.
__global__ void k_seq_boundary(float* grid, const float* __restrict__ ring, int streams, int b0, int parity) {
    const int i = b0 + blockIdx.y, r = blockIdx.x;
    const float* src = i >= streams ? grid + ((size_t)(i - streams) * SEQ_ROWS + 375 + r) * GRID_COLS
                                    : ring + ((size_t)i * LIVE_ROWS + (375 * parity + r - SEQ_H0 + LIVE_ROWS) % LIVE_ROWS) * GRID_COLS;
    const float4* s = reinterpret_cast<const float4*>(src);
    float4* d = reinterpret_cast<float4*>(grid + ((size_t)i * SEQ_ROWS + r) * GRID_COLS);
    for (int k = threadIdx.x; k < ROW_F4; k += blockDim.x) d[k] = s[k];
}

// Ring write-back of gridDim.y / streams consecutive steps (grid points at the first, of parity `parity`): ring row
// (375 p + h) mod 750 <- grid row SEQ_H0 + h, h = 1..375 -- the half a live call of that step would have written.
__global__ void k_seq_store_ring(const float* __restrict__ grid, float* __restrict__ ring, int streams, int parity) {
    const int j = blockIdx.y, hop = blockIdx.x + 1;
    const int b = j % streams, p = parity ^ ((j / streams) & 1);
    const float4* s = reinterpret_cast<const float4*>(grid + ((size_t)j * SEQ_ROWS + SEQ_H0 + hop) * GRID_COLS);
    float4* d = reinterpret_cast<float4*>(ring + ((size_t)b * LIVE_ROWS + (375 * p + hop) % LIVE_ROWS) * GRID_COLS);
    for (int k = threadIdx.x; k < ROW_F4; k += blockDim.x) d[k] = s[k];
}

// Front end of cycles b0 .. b0 + nb - 1 of a piece (d_audio = the whole piece): their tails (the last 3840 samples of the same
// stream one step earlier; the piece's first step has its tails copied from d_tail already), S1 into rows 6..380 and the
// boundary rows.  Adds its kernel launches other than S1 to *launches.
static int seq_front(ft8_handle* h, const SeqPiece& sp, const char* d_audio, int dtype, int b0, int nb, int* launches) {
    const size_t esz = sample_bytes(dtype);
    const int lo = std::max(b0, sp.streams), hi = b0 + nb;
    if (lo < hi) {
        TRY(save_tails(h, d_audio + (size_t)(lo - sp.streams) * CYCLE_SAMPLES * esz, dtype, hi - lo, h->d_seq_tail + (size_t)lo * NFFT_S));
        ++*launches;
    }
    float* g = h->d_seq_grid + (size_t)b0 * SEQ_ROWS * GRID_COLS;
    TRY(launch_spectrogram(h, d_audio + (size_t)b0 * CYCLE_SAMPLES * esz, dtype, nb, g, 1, 375, SEQ_ROWS, -SEQ_H0, 0,
                           h->d_seq_tail + (size_t)b0 * NFFT_S, 0));
    k_seq_boundary<<<dim3(SEQ_BOUND, nb), 256, 0, h->stream>>>(h->d_seq_grid, h->d_ring, sp.streams, b0, sp.parity);
    CK(cudaGetLastError());
    ++*launches;
    return FT8_OK;
}

// After the piece's kernels: the ring halves of its last two steps (one when it has one step; the half before that was
// written by the previous piece or call) and every stream's tail, as the live calls of those steps leave them.
static int seq_store(ft8_handle* h, const SeqPiece& sp, const char* d_audio, int dtype, int* launches) {
    const int last = sp.steps - 1, first = std::max(0, last - 1);
    TRY(save_tails(h, d_audio + (size_t)last * sp.streams * CYCLE_SAMPLES * sample_bytes(dtype), dtype, sp.streams, h->d_tail));
    k_seq_store_ring<<<dim3(375, (last - first + 1) * sp.streams), 256, 0, h->stream>>>(
        h->d_seq_grid + (size_t)first * sp.streams * SEQ_ROWS * GRID_COLS, h->d_ring, sp.streams, sp.parity ^ (first & 1));
    CK(cudaGetLastError());
    *launches += 2;
    return FT8_OK;
}

__global__ void k_fill(float* p, size_t n, float v) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// A fresh ring is all 1.0 like np.ones (receiver.py:238).  A stream without a previous cycle reads zeros before its first
// sample, as a fresh Receiver does; so does a stream that joins a later call with a larger B.
static int clear_live(ft8_handle* h) {
    k_fill<<<h->n_sm * 8, 256, 0, h->stream>>>(h->d_ring, h->cap_cycles * (size_t)LIVE_ROWS * GRID_COLS, 1.0f);
    CK(cudaGetLastError());
    CK(cudaMemsetAsync(h->d_tail, 0, h->cap_cycles * (size_t)NFFT_S * sizeof(float), h->stream));
    return FT8_OK;
}

// Decode prologue.  A pending prefetch is consumed only by the streaming entry (consume_pf), whose caller named this very
// buffer as the next batch and so promises it has not been rewritten since; every other call drops it -- after waiting for
// its copy, which may still be reading the caller's host buffer.  *d_audio is where the batch is on the device (for host
// audio that was not prefetched: where it is to be copied); *prefetched says whether it came from the prefetch.
static int take_audio(ft8_handle* h, const void* audio, int dtype, int B, int mem, bool consume_pf, const void** d_audio,
                      bool* prefetched) {
    *prefetched = consume_pf && mem == FT8_MEM_HOST && h->pf_host == audio && h->pf_B == B && h->pf_dtype == dtype;
    if (!*prefetched && h->pf_host) CK(cudaStreamSynchronize(h->copy_stream));
    h->pf_host = nullptr;                        // a pending prefetch this call does not consume is dropped, never decoded later
    *d_audio = audio;
    if (*prefetched) {
        // this batch was copied by ft8_prefetch_audio while the previous call was computing: swap it in and go on as if
        // the audio were device-resident
        std::swap(h->d_audio, h->d_audio_pf);
        CK(cudaStreamWaitEvent(h->stream, h->pf_ev, 0));
        *d_audio = h->d_audio;
    } else if (mem == FT8_MEM_HOST) {
        CK(h->d_audio.ensure((size_t)B * CYCLE_SAMPLES * sample_bytes(dtype), h->stream));
        *d_audio = h->d_audio;
    }
    return FT8_OK;
}

// Decode epilogue: counts, records and statistics back to the host.  Records are cycle-major, so when rec_capacity cuts
// them the per-cycle counts are trimmed to what was copied.
static int finish_decode(ft8_handle* h, int B, ft8_record* rec, int rec_capacity, int32_t* n_rec, int launches) {
    CK(cudaMemcpyAsync(h->h_counts, h->d_counts, (CNT_NEAR_TIE + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(h->h_stats, h->d_stats, sizeof(DevStats), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(n_rec, h->d_rec_n, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    const int nrec = h->h_counts[CNT_RECORDS];
    const int ncopy = std::min(nrec, rec_capacity);
    if (ncopy > 0) {
        CK(cudaMemcpyAsync(rec, h->d_rec, (size_t)ncopy * sizeof(ft8_record), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    const bool overflow = nrec > rec_capacity;
    if (overflow) {
        int left = rec_capacity;
        for (int b = 0; b < B; ++b) { const int t = std::min(n_rec[b], left); n_rec[b] = t; left -= t; }
    }
    const int64_t emitted = (int64_t)h->h_stats->emitted;
    CK(cudaEventElapsedTime(&h->last_ms[MS_TOTAL], h->ev[EV_START], h->ev[EV_RECORDS]));
    for (int i = MS_SPECTROGRAM; i <= MS_RECORDS; ++i) CK(cudaEventElapsedTime(&h->last_ms[i], h->ev[i - 1], h->ev[i]));
    h->last_ms[MS_FINE_TSCAN] = h->last_ms[MS_FINE_FSCAN] = h->last_ms[MS_FINE_FINAL] = 0.0f;
    if (h->cfg.fine_mode == 0) {
        CK(cudaEventElapsedTime(&h->last_ms[MS_FINE_TSCAN], h->ev[EV_PASS0], h->ev[EV_TSCAN_END]));
        CK(cudaEventElapsedTime(&h->last_ms[MS_FINE_FSCAN], h->ev[EV_TSCAN_END], h->ev[EV_FSCAN_END]));
        CK(cudaEventElapsedTime(&h->last_ms[MS_FINE_FINAL], h->ev[EV_FSCAN_END], h->ev[EV_FINE]));
    }
    ft8_stats& s = h->stats;
    memset(&s, 0, sizeof(s));
    s.cycles = B; s.candidates = (int64_t)h->h_stats->candidates; s.stopped_sd = (int64_t)h->h_stats->stopped_sd;
    s.fine_evals = (int64_t)h->h_stats->fine_evals; s.fine_pass = (int64_t)h->h_stats->fine_pass;
    s.ldpc_calls = (int64_t)h->h_stats->ldpc_calls; s.ldpc_iters = (int64_t)h->h_stats->ldpc_iters;
    s.osd_calls = (int64_t)h->h_stats->osd_calls; s.decoded = nrec; s.emitted = emitted; s.kernel_launches = launches;
    s.fine_rechecked = h->cfg.fine_mode == 0 ? h->h_counts[CNT_NEAR_TIE] : 0;
    if (overflow) return fail(h, FT8_E_CAPACITY, "ft8_decode_cycles: rec_capacity too small (records truncated)");
    return FT8_OK;
}

static int decode_cycles_core(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even, ft8_record* rec,
                              int rec_capacity, int32_t* n_rec, int mem, const void* next_audio_host, bool consume_pf,
                              bool live = false, const SeqPiece* seq = nullptr) {
    ENTER(h);
    if (!audio || !rec || !n_rec || B <= 0 || rec_capacity < 0) return fail(h, FT8_E_BADARG, "ft8_decode_cycles: bad argument");
    if ((size_t)B > h->cap_cycles) return fail(h, FT8_E_CAPACITY, "ft8_decode_cycles: B exceeds cfg.max_cycles");
    const int K = h->cfg.max_cands, N = B * K;
    // Isolated mode (default): every cycle is decoded on its own 376-row waterfall (SURVEY H5), the search runs with
    // cycle_h0 = 0 and odd_even only labels the records on the host side (their_tx_cycle, receiver.py:62).
    // Live mode: stream b keeps the reference's 750-row two-cycle ring (receiver.py:238, 295-306); this call's rows go to the
    // half odd_even selects, rows of the other half still hold the previous cycle, and the first hops' windows reach back into
    // the previous cycle's last samples -- so candidates with h0 < -32 read real rows, exactly as a live Receiver does.
    // Consecutive live cycles (seq): one piece of ft8_decode_cycles_live_seq on SEQ_ROWS-row grids (see SeqPiece), chained
    // to the calls before and after it through the same ring and tails.
    TRY(check_dtype(h, audio_dtype));
    const size_t esz = sample_bytes(audio_dtype);
    const int cycle_h0 = seq ? SEQ_H0 : live ? (odd_even ? 375 : 0) : 0;
    const int grows = seq ? SEQ_ROWS : live ? LIVE_ROWS : GRID_ROWS;
    float* gbase = h->d_grid;
    if (live || seq) {
        if (!h->d_ring) {
            CK(h->d_ring.ensure(h->cap_cycles * (size_t)LIVE_ROWS * GRID_COLS, h->stream));
            CK(h->d_tail.ensure(h->cap_cycles * (size_t)NFFT_S, h->stream));
            TRY(clear_live(h));
        }
        gbase = h->d_ring;
    }
    if (seq) {
        CK(h->d_seq_grid.ensure(h->cap_cycles * (size_t)SEQ_ROWS * GRID_COLS, h->stream));
        CK(h->d_seq_tail.ensure(h->cap_cycles * (size_t)NFFT_S, h->stream));
        gbase = h->d_seq_grid;
    }
    const void* da;
    bool prefetched;
    TRY(take_audio(h, audio, audio_dtype, B, mem, consume_pf, &da, &prefetched));
    const bool copy = mem == FT8_MEM_HOST && !prefetched;
    // streaming callers name the next batch: its copy is queued now and runs underneath this batch's kernels
    // (after this batch's own copies when it was not prefetched itself, so that they are not queued behind it)
    if (next_audio_host && prefetched) TRY(ft8_prefetch_audio(h, next_audio_host, audio_dtype, B));
    int launches = 0;
    CK(cudaMemsetAsync(h->d_counts, 0, CNT_SLOTS * sizeof(int32_t), h->stream));
    CK(cudaMemsetAsync(h->d_stats, 0, sizeof(DevStats), h->stream));
    CK(cudaEventRecord(h->ev[EV_START], h->stream));
    if (seq) CK(cudaMemcpyAsync(h->d_seq_tail, h->d_tail, (size_t)seq->streams * NFFT_S * sizeof(float), cudaMemcpyDeviceToDevice,
                                h->stream));           // the tails of the piece's first step
    // Front end (S1, S2, F1) chunk by chunk.  Host audio is copied on the copy stream in up to 16 equal chunks, and a chunk's
    // kernels start as soon as it has landed, so the PCIe transfer hides behind the front end of the chunks before it
    // (measured best for a single handle: 28.6 k cycles/s vs 27.3-28.0 k for growing chunks); callers that stream batch
    // after batch should use ft8_prefetch_audio, which hides the whole transfer.  Device-resident or prefetched audio is one
    // chunk.  With one chunk the stage events fall between S1, S2 and F1; with several, stage 1 covers the whole front end.
    const int nchunk = copy ? std::min(16, (B + 255) / 256) : 1;
    const int per = (B + nchunk - 1) / nchunk;
    if (copy) {
        CK(cudaEventRecord(h->chunk_ev[0], h->stream));
        CK(cudaStreamWaitEvent(h->copy_stream, h->chunk_ev[0], 0));        // previous users of d_audio on the main stream are done
        for (int c = 0, b0 = 0; b0 < B; ++c, b0 += per) {
            const size_t off = (size_t)b0 * CYCLE_SAMPLES * esz;
            CK(cudaMemcpyAsync(h->d_audio + off, (const char*)audio + off, (size_t)std::min(per, B - b0) * CYCLE_SAMPLES * esz,
                               cudaMemcpyHostToDevice, h->copy_stream));
            CK(cudaEventRecord(h->chunk_ev[c], h->copy_stream));
        }
    }
    for (int c = 0, b0 = 0; b0 < B; ++c, b0 += per) {
        const int nb = std::min(per, B - b0);
        const char* a = (const char*)da + (size_t)b0 * CYCLE_SAMPLES * esz;
        if (copy) CK(cudaStreamWaitEvent(h->stream, h->chunk_ev[c], 0));
        float* gc = gbase + (size_t)b0 * grows * GRID_COLS;
        if (seq) TRY(seq_front(h, *seq, (const char*)da, audio_dtype, b0, nb, &launches));
        else if (live) TRY(launch_spectrogram(h, a, audio_dtype, nb, gc, 1, 375, LIVE_ROWS, -cycle_h0, 0, h->d_tail + (size_t)b0 * NFFT_S, 1));
        else TRY(launch_spectrogram(h, a, audio_dtype, nb, gc));
        ++launches;
        if (nchunk == 1) CK(cudaEventRecord(h->ev[EV_SPECTROGRAM], h->stream));
        TRY(launch_sync(h, gc, grows, nb, cycle_h0, b0)); launches += 2;
        if (nchunk == 1) CK(cudaEventRecord(h->ev[EV_SYNC], h->stream));
        // F1 (independent of S1/S2; same stream)
        TRY(launch_cycle_spectrum(h, a, audio_dtype, nb, h->d_spec + (size_t)b0 * FINE_SPEC_STRIDE, FINE_SPEC_STRIDE, FINE_SPEC_STRIDE - 1));
        launches += 2 * ((nb + (int)h->y_cycles - 1) / (int)h->y_cycles);
    }
    if (nchunk > 1) {
        CK(cudaEventRecord(h->ev[EV_SPECTROGRAM], h->stream));
        CK(cudaEventRecord(h->ev[EV_SYNC], h->stream));
    }
    CK(cudaEventRecord(h->ev[EV_CYCLE_SPECTRUM], h->stream));
    if (next_audio_host && !prefetched) TRY(ft8_prefetch_audio(h, next_audio_host, audio_dtype, B));
    if (seq) TRY(seq_store(h, *seq, (const char*)da, audio_dtype, &launches));
    else if (live) { TRY(save_tails(h, da, audio_dtype, B, h->d_tail)); ++launches; }   // after S1 has read the old tails
    CandState cs = cand_state(h);
    // ipass 0
    k_pass0<<<persistent_blocks(h, 8), WARPS_PER_CTA * 32, sizeof(PassSmem), h->stream>>>(
        cs, N, gbase, grows, cycle_h0, h->cfg.llr_sd_min, nullptr, 0, h->d_list_fine, h->d_counts + CNT_FINE,
        h->d_counts + CNT_CURSOR_PASS0, h->d_stats);
    CK(cudaGetLastError()); ++launches;
    CK(cudaEventRecord(h->ev[EV_PASS0], h->stream));
    // ipass 1
    TRY(launch_fine(h, h->d_spec, FINE_SPEC_STRIDE, h->d_list_fine, h->d_counts + CNT_FINE, 0, h->d_cycle_of, h->d_f0, h->d_h0, h->d_fine,
                    h->d_llr_fine, nullptr));
    launches += fine_launches(h);
    CK(cudaEventRecord(h->ev[EV_FINE], h->stream));
    // ipass 2-4
    k_pass234<<<persistent_blocks(h, 8), WARPS_PER_CTA * 32, sizeof(PassSmem), h->stream>>>(
        cs, h->d_list_fine, h->d_counts + CNT_FINE, h->cfg.llr_sd_min, h->d_list_osd, h->d_counts + CNT_OSD,
        h->d_counts + CNT_CURSOR_PASS234, h->d_stats);
    CK(cudaGetLastError()); ++launches;
    CK(cudaEventRecord(h->ev[EV_PASS234], h->stream));
    // ipass 5-6
    k_osd_items<<<persistent_blocks(h, 8), WARPS_PER_CTA * 32, sizeof(OsdSmem), h->stream>>>(
        cs, h->d_list_osd, h->d_counts + CNT_OSD, h->cfg.osd_singleflips, h->cfg.osd_doubleflips, h->d_counts + CNT_CURSOR_OSD,
        h->d_stats);
    CK(cudaGetLastError()); ++launches;
    k_osd_resolve<<<persistent_blocks(h, 2), 128, 0, h->stream>>>(cs, h->d_list_osd, h->d_counts + CNT_OSD, h->d_stats);
    CK(cudaGetLastError()); ++launches;
    CK(cudaEventRecord(h->ev[EV_OSD], h->stream));
    k_rec_count<<<B, REC_NT, 0, h->stream>>>(cs, h->d_rec_n);
    CK(cudaGetLastError()); ++launches;
    k_rec_scan<<<1, 1024, 0, h->stream>>>(h->d_rec_n, B, h->d_rec_base, h->d_counts + CNT_RECORDS);
    CK(cudaGetLastError()); ++launches;
    k_rec_write<<<B, REC_NT, 0, h->stream>>>(cs, h->d_fine, h->d_rec_base, h->d_rec, h->d_stats);
    CK(cudaGetLastError()); ++launches;
    CK(cudaEventRecord(h->ev[EV_RECORDS], h->stream));
    return finish_decode(h, B, rec, rec_capacity, n_rec, launches);
}

extern "C" int ft8_decode_cycles(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even, ft8_record* rec,
                                 int rec_capacity, int32_t* n_rec, int mem) {
    return decode_cycles_core(h, audio, audio_dtype, B, odd_even, rec, rec_capacity, n_rec, mem, nullptr, false);
}

extern "C" int ft8_decode_cycles_live(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even, ft8_record* rec,
                                      int rec_capacity, int32_t* n_rec, int mem) {
    if (odd_even != 0 && odd_even != 1) return fail(h, FT8_E_BADARG, "ft8_decode_cycles_live: odd_even must be 0 or 1");
    return decode_cycles_core(h, audio, audio_dtype, B, odd_even, rec, rec_capacity, n_rec, mem, nullptr, false, true);
}

// C steps of B streams in pieces of floor(max_cycles / B) steps; each piece is one decode batch.  Records of a piece land after
// those of the pieces before it (cycle-major, so the capacity cut of finish_decode stays cycle-major over the whole call);
// their cycle index is the piece's local one and is shifted here.
extern "C" int ft8_decode_cycles_live_seq(ft8_handle* h, const void* audio, int audio_dtype, int B, int C, int odd_even,
                                          ft8_record* rec, int rec_capacity, int32_t* n_rec, int mem) {
    ENTER(h);
    if (odd_even != 0 && odd_even != 1) return fail(h, FT8_E_BADARG, "ft8_decode_cycles_live_seq: odd_even must be 0 or 1");
    if (!audio || !rec || !n_rec || B <= 0 || C <= 0 || rec_capacity < 0)
        return fail(h, FT8_E_BADARG, "ft8_decode_cycles_live_seq: bad argument");
    if ((size_t)B > h->cap_cycles) return fail(h, FT8_E_CAPACITY, "ft8_decode_cycles_live_seq: B exceeds cfg.max_cycles");
    TRY(check_dtype(h, audio_dtype));
    const int per = (int)(h->cap_cycles / B);
    const size_t step_bytes = (size_t)B * CYCLE_SAMPLES * sample_bytes(audio_dtype);
    ft8_stats total{};
    float ms[MS_COUNT] = {};
    int written = 0;
    bool overflow = false;
    CK(cudaEventRecord(h->ev[EV_OP_BEGIN], h->stream));
    for (int c0 = 0; c0 < C; c0 += per) {
        const SeqPiece sp{B, std::min(per, C - c0), odd_even ^ (c0 & 1)};
        const int nb = sp.steps * B;
        ft8_record* r = rec + written;
        int32_t* n = n_rec + (size_t)c0 * B;
        const int rc = decode_cycles_core(h, (const char*)audio + (size_t)c0 * step_bytes, audio_dtype, nb, sp.parity, r,
                                          rec_capacity - written, n, mem, nullptr, false, false, &sp);
        if (rc != FT8_OK && rc != FT8_E_CAPACITY) return rc;
        overflow = overflow || rc == FT8_E_CAPACITY;
        int got = 0;
        for (int i = 0; i < nb; ++i) got += n[i];
        for (int i = 0; i < got; ++i) r[i].cycle += c0 * B;
        written += got;
        const ft8_stats& s = h->stats;
        total.cycles += s.cycles; total.candidates += s.candidates; total.stopped_sd += s.stopped_sd;
        total.fine_evals += s.fine_evals; total.fine_pass += s.fine_pass; total.ldpc_calls += s.ldpc_calls;
        total.ldpc_iters += s.ldpc_iters; total.osd_calls += s.osd_calls; total.decoded += s.decoded; total.emitted += s.emitted;
        total.kernel_launches += s.kernel_launches; total.fine_rechecked += s.fine_rechecked;
        for (int i = MS_SPECTROGRAM; i < MS_COUNT; ++i) ms[i] += h->last_ms[i];
    }
    CK(cudaEventRecord(h->ev[EV_OP_END], h->stream));
    CK(cudaEventSynchronize(h->ev[EV_OP_END]));
    CK(cudaEventElapsedTime(&ms[MS_TOTAL], h->ev[EV_OP_BEGIN], h->ev[EV_OP_END]));
    h->stats = total;
    memcpy(h->last_ms, ms, sizeof(ms));
    if (overflow) return fail(h, FT8_E_CAPACITY, "ft8_decode_cycles_live_seq: rec_capacity too small (records truncated)");
    return FT8_OK;
}

extern "C" int ft8_live_reset(ft8_handle* h) {
    ENTER(h);
    if (h->d_ring) TRY(clear_live(h));
    CK(cudaStreamSynchronize(h->stream));
    return FT8_OK;
}

extern "C" int ft8_decode_cycles_stream(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even, ft8_record* rec,
                                        int rec_capacity, int32_t* n_rec, const void* next_audio_host) {
    return decode_cycles_core(h, audio, audio_dtype, B, odd_even, rec, rec_capacity, n_rec, FT8_MEM_HOST, next_audio_host, true);
}

// ------------------------------------------------------------------------------------------ generator + test hook
extern "C" int ft8_synth_cycles(ft8_handle* h, const uint8_t* symbols, const float* f_hz, const float* dt_s, const float* amp,
                                int B, int n_sig, float noise_sigma, uint64_t seed, int16_t* audio, int mem) {
    ENTER(h);
    if (!symbols || !f_hz || !dt_s || !amp || !audio || B <= 0 || n_sig < 0 || n_sig > SYNTH_MAX_SIG)
        return fail(h, FT8_E_BADARG, "ft8_synth_cycles: bad argument (n_sig <= 128)");
    const size_t ns = (size_t)B * n_sig;
    uint8_t* dsym; float *df, *dd, *dam; int16_t* da;
    Staging st(h, mem);
    st.scratch(dsym, ns * 79); st.scratch(df, ns * 4); st.scratch(dd, ns * 4); st.scratch(dam, ns * 4);
    st.out(da, audio, (size_t)B * CYCLE_SAMPLES * 2);
    TRY(st.begin());
    // parameters are small and always copied, from host or device memory
    CK(cudaMemcpyAsync(dsym, symbols, ns * 79, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpyAsync(df, f_hz, ns * 4, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpyAsync(dd, dt_s, ns * 4, cudaMemcpyDefault, h->stream));
    CK(cudaMemcpyAsync(dam, amp, ns * 4, cudaMemcpyDefault, h->stream));
    k_synth<<<dim3((CYCLE_SAMPLES + SYNTH_TILE - 1) / SYNTH_TILE, B), SYNTH_NT, 0, h->stream>>>(dsym, df, dd, dam, n_sig, noise_sigma, seed, h->d_pulse, da);
    CK(cudaGetLastError());
    return st.finish();
}

template <int N, int NT, bool INV>
__global__ void k_debug_fft(const float2* __restrict__ in, float2* __restrict__ out, const float2* __restrict__ W) {
    extern __shared__ float2 dbg_smem[];
    const float2* x = in + (size_t)blockIdx.x * N;
    for (int i = threadIdx.x; i < N; i += NT) dbg_smem[i] = x[i];
    __syncthreads();
    if (N == 1920) fft1920<NT, INV>(dbg_smem, threadIdx.x, W);
    if (N == 3200) fft3200<NT, INV>(dbg_smem, threadIdx.x, W);
    if (N == 375) fft375<NT, INV>(dbg_smem, threadIdx.x, W);
    if (N == 256) fft256<NT, INV>(dbg_smem, threadIdx.x, W);
    if (N == 32) fft32<NT, INV>(dbg_smem, threadIdx.x, W);
    for (int i = threadIdx.x; i < N; i += NT) out[(size_t)blockIdx.x * N + i] = dbg_smem[i];
}

extern "C" int ft8_debug_fft(ft8_handle* h, int n, int inverse, const float* in, float* out, int batch) {
    ENTER(h);
    if (!in || !out || batch <= 0) return fail(h, FT8_E_BADARG, "ft8_debug_fft: bad argument");
    const size_t bytes = (size_t)batch * n * sizeof(float2);
    const float2* di; float2* dout;
    Staging st(h, FT8_MEM_HOST);
    st.in(di, in, bytes);
    st.out(dout, out, bytes);
    TRY(st.begin());
#define DBG(NN, NT, WT)                                                                                                    \
    if (n == NN) {                                                                                                         \
        if (inverse) k_debug_fft<NN, NT, true><<<batch, NT, NN * sizeof(float2), h->stream>>>(di, dout, WT);               \
        else k_debug_fft<NN, NT, false><<<batch, NT, NN * sizeof(float2), h->stream>>>(di, dout, WT);                      \
    }
    DBG(1920, 128, h->d_W1920) else DBG(3200, 256, h->d_W3200) else DBG(375, 128, h->d_W375) else DBG(256, 64, h->d_W256)
    else DBG(32, 32, h->d_W32) else return fail(h, FT8_E_BADARG, "ft8_debug_fft: n must be 32, 256, 375, 1920 or 3200");
#undef DBG
    CK(cudaGetLastError());
    return st.finish();
}

#ifdef FS_PROFILE
extern "C" int ft8_debug_fs_prof(unsigned long long* out16, int reset) {
    cudaMemcpyFromSymbol(out16, ft8::g_fs_prof, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(ft8::g_fs_prof, z, sizeof(z)); }
    return 0;
}
#endif

#ifdef FINE_PROFILE
// debug build only: read (and optionally reset) the k_fine phase counters
extern "C" int ft8_debug_fine_prof(unsigned long long* out16, int reset) {
    cudaMemcpyFromSymbol(out16, ft8::g_fine_prof, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(ft8::g_fine_prof, z, sizeof(z)); }
    return 0;
}
#endif
