/* ft8_b200.h -- C ABI of the B200-native FT8 receive hot path (libft8_b200.so).
 *
 * Drop-in boundary for G1OJS/PyFT8's receive chain (reference paths are PyFT8/...):
 * each entry point replaces one reference function, batched, and is what the
 * reference-side ctypes binding (INTEGRATION.md) loads.  Plain pointers and sizes only.
 *
 * Conventions
 *   - every function returns FT8_OK (0) or a negative FT8_E* code; ft8_last_error(h)
 *     gives the text.  "No decode" is data (status / n == 0), never an error.
 *   - `mem` says where the caller's buffers live: FT8_MEM_HOST (numpy / malloc; the
 *     library stages them through its own device scratch, copies included in the call)
 *     or FT8_MEM_DEVICE (pointers on the handle's CUDA device, e.g. torch .data_ptr()).
 *   - the caller owns every buffer; the library owns only the handle (tables + scratch).
 *   - a handle is one CUDA device + one stream; calls on one handle are serialised by
 *     the caller, different handles are independent.  No global mutable state.
 *   - there is no CPU fallback: without a usable CUDA device ft8_create fails.
 *   - bit packing: a 91-bit word (77 message + 14 CRC bits, codeword order) is stored
 *     LSB-first in three uint32: bit j (0 = first transmitted) is (w[j>>5] >> (j&31)) & 1.
 */
#ifndef FT8_B200_H
#define FT8_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FT8_OK            0
#define FT8_E_BADARG     -1
#define FT8_E_CUDA       -2
#define FT8_E_CAPACITY   -3
#define FT8_E_NODEVICE   -4

#define FT8_MEM_HOST      0
#define FT8_MEM_DEVICE    1

#define FT8_AUDIO_I16     0      /* int16 samples, as PyAudio delivers them (receiver.py:296) */
#define FT8_AUDIO_F32     1      /* float32 samples in int16 scale (receiver.py:248)          */

/* geometry (receiver.py:228-243, 319-327; SURVEY.md section 8) */
#define FT8_SAMPLES_PER_CYCLE 180000
#define FT8_GRID_ROWS         376     /* rows 0..375 of one cycle; row h = window ending at sample 480*h; row 0 == 1.0 */
#define FT8_GRID_ROWS_LIVE    750     /* two-cycle ring of the live receiver (receiver.py:238) */
#define FT8_GRID_COLS         976
#define FT8_N_F0              928     /* f0 bins 32..959 */
#define FT8_N_H0              124     /* h0 offsets -37..86 */
#define FT8_SPEC_BINS         96001   /* rfft of 192000 samples */
#define FT8_PAYLOAD_ROWS      58
#define FT8_N_LLR             174

/* LDPC status codes (decoders.py:153-171) */
#define FT8_LDPC_REJECT   0   /* iteration-0 syndrome weight > max_ncheck0: llr untouched, reference returns (None,-1,[]) */
#define FT8_LDPC_OK       1   /* syndrome 0, CRC-14 ok, payload accepted by unpack: reference returns (msg, n_its, [])     */
#define FT8_LDPC_FAIL     2   /* max_iters reached: reference returns (None,-1,llr)                                         */
#define FT8_LDPC_STALL    3   /* syndrome 0 but CRC/unpack rejected: llr frozen, reference returns (None,-1,llr)            */

/* how a record was decoded (decode_notes of receiver.py:121,126,133) */
#define FT8_METHOD_GOOD91     0
#define FT8_METHOD_LDPC5      1
#define FT8_METHOD_LDPC20     2
#define FT8_METHOD_OSD        3   /* OSD on the AP'd llr (ipass 5)          */
#define FT8_METHOD_LDPC20_OSD 4   /* OSD on a saved post-LDPC llr (ipass 6) */

typedef struct ft8_handle ft8_handle;

/* Mirrors Receiver(...) / Candidate(...) / osd_012(...) keyword arguments (receiver.py:30,311-313; decoders.py:223). */
typedef struct ft8_cfg {
    int32_t max_cycles;        /* scratch capacity: cycles per ft8_decode_cycles / stage call          */
    int32_t max_cands;         /* Receiver(max_cands=200)                                              */
    float   sync_score_min;    /* Receiver(sync_score_min=85)                                          */
    float   llr_sd_min;        /* Candidate(llr_sd_min=5)                                              */
    int32_t osd_singleflips;   /* osd_012(singleflips=30)                                              */
    int32_t osd_doubleflips;   /* osd_012(doubleflips=2)                                               */
    int32_t max_codewords;     /* unused; kept for the layout of this struct                                               */
    int32_t fine_mode;         /* fine sync (receiver.py:140-206): 0 = time scan + tensor-core frequency scan + final transform
                                  (default); 1 = the literal nine-inverse-FFT kernel (A/B reference for the former)            */
    /* Receiver(search_freq_range, search_time_range) as index ranges (receiver.py:311-319): coarse frequency bins
     * f0 in [search_f0_lo, search_f0_hi) (3.125 Hz each; int(Hz / 3.125)) and hop offsets h0 in [search_h0_lo, search_h0_hi)
     * (40 ms each; int((t + 0.5) * 25)).  All four zero = the reference defaults [100, 3000] Hz -> [32, 960) and
     * [-2, 3] s -> [-37, 87), which are also the widest ranges the kernels are built for: any sub-range is honoured,
     * anything wider is FT8_E_BADARG. */
    int16_t search_f0_lo, search_f0_hi, search_h0_lo, search_h0_hi;
    int32_t reserved[2];
} ft8_cfg;

/* One decoded candidate, as Candidate.check_and_package would see it (receiver.py:51-66). 64 bytes. */
typedef struct ft8_record {
    uint32_t bits91[3];   /* message + CRC bits, LSB-first packing (see top)                               */
    int32_t  cycle;       /* index of the cycle inside the batch                                           */
    int16_t  cand;        /* rank of the candidate in Receiver.search order (score descending)             */
    int16_t  f0_idx;      /* coarse frequency bin (3.125 Hz)                                               */
    int16_t  h0_idx;      /* coarse hop offset (40 ms)                                                     */
    int8_t   snr;         /* Candidate.snr at decode time (receiver.py:212)                                */
    uint8_t  ipass;       /* pass in which it decoded, 0..6 (receiver.py:72-103)                           */
    uint8_t  ap;          /* a-priori pattern 0 NoAP, 1 CQ, 2 RR73, 3 73, 4 RRR (receiver.py:21-27)        */
    uint8_t  method;      /* FT8_METHOD_*                                                                  */
    int8_t   ttweak;      /* fine time tweak in 5 ms steps (0 before the fine stage)                       */
    int8_t   ftweak;      /* fine frequency tweak in 1/16 Hz steps                                         */
    uint8_t  nsync;       /* Costas symbols matched by the fine stage (100 before it, receiver.py:45)      */
    uint8_t  emitted;     /* 1 = first occurrence of this payload in emission order, 0 = duplicate         */
    uint16_t n_its;       /* LDPC iteration at which it converged (LDPC methods)                           */
    float    score;       /* coarse sync score                                                             */
    float    tsec;        /* origin['tsec'] after tweaks (all_txt prints tsec - 0.6)                       */
    float    fHz;         /* origin['fHz'] after tweaks                                                    */
    float    grid_sd;     /* llr_sd of the grid-stage LLRs                                                 */
    float    fine_sd;     /* llr_sd of the fine-stage LLRs (NaN before the fine stage)                     */
    uint32_t reserved[3];
} ft8_record;

/* Work counters of the last ft8_decode_cycles call (SURVEY.md section 5: metrics). */
typedef struct ft8_stats {
    int64_t cycles, candidates, stopped_sd, fine_evals, fine_pass, ldpc_calls, ldpc_iters, osd_calls,
            decoded, emitted, kernel_launches;
    int64_t fine_rechecked;      /* candidates whose frequency scan was a near-tie and was decided by the literal kernel */
    int64_t reserved[4];
} ft8_stats;

/* Fills cfg with the reference defaults (max_cycles = 1). */
void ft8_default_cfg(ft8_cfg* cfg);
int  ft8_create(int device, const ft8_cfg* cfg, ft8_handle** out);
void ft8_destroy(ft8_handle* h);
const char* ft8_last_error(ft8_handle* h);       /* h may be NULL: error of the last failed ft8_create on this thread */
int  ft8_get_stats(ft8_handle* h, ft8_stats* out);
int  ft8_synchronize(ft8_handle* h);
/* CUDA stream of the handle (cudaStream_t as void*), for callers that enqueue their own work / events on it. */
void* ft8_stream(ft8_handle* h);
/* Milliseconds spent on the device (CUDA events on the handle's stream).  After ft8_decode_cycles: which = 0 whole
 * device section, 1 spectrogram, 2 sync (scores + top-K), 3 cycle spectrum, 4 pass 0 (grid LLR + GOOD91 + LDPC5),
 * 5 fine sync, 6 passes 2-4 (LDPC), 7 passes 5-6 (OSD), 8 record collection, 9 / 10 / 11 the three kernels of the fine stage
 * (time scan, tensor-core frequency scan, final transform; 0 with fine_mode 1).  Host audio of more than 256 cycles that was
 * not prefetched is copied and processed in chunks: then 1 covers the whole front end (1-3) and 2 and 3 are 0.
 * After ft8_decode_cycles_live_seq: 0 = the whole call (all its pieces), 1-11 = the sums of those entries over the pieces.
 * After a stand-alone ft8_spectrogram / ft8_sync call: 1 / 2 = that kernel.  After ft8_ldpc / ft8_osd: 0 = that kernel. */
int  ft8_last_kernel_ms(ft8_handle* h, int which, float* ms);

/* S1  AudioIn.get_hop_spectrum x375 (receiver.py:288-293): audio[B][180000] -> grid_db[B][376][976] float32 dB. */
int ft8_spectrogram(ft8_handle* h, const void* audio, int audio_dtype, int B, float* grid_db, int mem);

/* S1, live form: exactly AudioIn.get_hop_spectrum (receiver.py:288-293) -- audio_buffer[180000] is the receiver's ring
 *     buffer (receiver.py:248, 296-299); row_db[976] = 20*log10(|rfft(audio_buffer[-3840:] * hanning)[:976]| + 1e-12). */
int ft8_hop_spectrum(ft8_handle* h, const void* audio_buffer, int audio_dtype, float* row_db, int mem);

/* S2  Receiver.search (receiver.py:338-367): grid_db[B][grid_rows][976] (grid_rows 376: rows beyond read as 1.0,
 *     or 750: the live ring) -> per cycle up to max_cands candidates sorted by score descending.
 *     cand_f0/cand_h0: int16 [B][max_cands]; cand_score: float [B][max_cands]; n_cand: int32 [B];
 *     payload_db: float [B][max_cands][58][8] or NULL. */
int ft8_sync(ft8_handle* h, const float* grid_db, int grid_rows, int B, int odd_even,
             int16_t* cand_f0, int16_t* cand_h0, float* cand_score, int32_t* n_cand, float* payload_db, int mem);

/* L0  Candidate._dB_to_llr (receiver.py:208-222): payload_db[N][58][8] -> llr[N][174], sd[N], snr[N] (int32). */
int ft8_llr(ft8_handle* h, const float* payload_db, int N, float* llr, float* sd, int32_t* snr, int mem);

/* F1  AudioIn.get_cycle_spectrum (receiver.py:280-286): audio[B][180000] -> spec[B][96001] complex64 (re,im). */
int ft8_cycle_spectrum(ft8_handle* h, const void* audio, int audio_dtype, int B, float* spec, int mem);

/* F2+F3  Candidate._get_llr_fine (receiver.py:140-206) for N candidates: cycle_of[N] indexes spec[B][96001];
 *     f0_idx/h0_idx[N] are the coarse origin.  Outputs: ttweak/ftweak/nsync int32 [N]; signal_grid[N][79][8]
 *     (linear magnitudes, may be NULL); llr[N][174], sd[N], snr[N] valid where nsync > 6. */
int ft8_fine(ft8_handle* h, const float* spec, int B, const int32_t* cycle_of, const int16_t* f0_idx,
             const int16_t* h0_idx, int N, int32_t* ttweak, int32_t* ftweak, int32_t* nsync,
             float* signal_grid, float* llr, float* sd, int32_t* snr, int mem);

/* L1+L2  ldpc_decode (decoders.py:153-171), llr[N][174] updated in place; status/nits int32 [N]; bits91 uint32 [N][3]
 *     (hard decisions of llr[:91] at exit). */
int ft8_ldpc(ft8_handle* h, float* llr, int N, int max_ncheck0, int max_iters,
             int32_t* status, int32_t* nits, uint32_t* bits91, int mem);

/* O1+K1  osd_012 (decoders.py:223-272): llr[N][174] -> found[N] (trial index + 1 of the first trial word that has a
 *     non-zero payload, passes CRC-14 and is accepted by unpack; 0 = none), bits91[N][3]. */
int ft8_osd(ft8_handle* h, const float* llr, int N, int singleflips, int doubleflips,
            int32_t* found, uint32_t* bits91, int mem);

/* K1  crc_unpack91 minus the text (decoders.py:117-131): bits91[N][3] -> flags[N]: bit0 payload != 0 and CRC-14
 *     matches, bit1 payload accepted by unpack (decoders.py:16-115 as a predicate). */
int ft8_crc14(ft8_handle* h, const uint32_t* bits91, int N, int32_t* flags, int mem);

/* Whole path, Receiver.search + Candidate.decode passes 0..7 for every candidate (receiver.py:68-107, 389-398):
 * audio[B][180000] -> records.  rec has room for rec_capacity records; records of one cycle are contiguous and in
 * the reference's emission order; n_rec[B] (int32) counts per cycle; duplicates of a payload are kept with
 * emitted = 0.  The output arrays are HOST memory in every mode; `mem` describes `audio` only.  Each cycle is decoded in
 * isolation (no rows from a neighbouring cycle); odd_even is carried as a label only (their_tx_cycle, receiver.py:62). */
int ft8_decode_cycles(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even,
                      ft8_record* rec, int rec_capacity, int32_t* n_rec, int mem);

/* Live form of ft8_decode_cycles (what a running Receiver sees, receiver.py:238, 295-306, 338-367): the handle keeps, per
 * stream b < B, the reference's 750-row two-cycle waterfall ring and the previous cycle's last 3840 samples.  Each call
 * decodes the NEXT 15 s of every stream: its rows are written into the half `odd_even` selects (rows of the other half
 * still hold the previous cycle; a fresh ring is all 1.0 like np.ones), the first hops' windows reach back into the
 * previous cycle's audio, the search runs with cycle_h0 = 375 * odd_even, and payload rows wrap mod 750 into the other
 * half -- so a signal that starts before the cycle boundary (h0 < -32) is read from real rows, as in the reference.
 * Callers alternate odd_even 0, 1, 0, ... per stream position; ft8_live_reset forgets all streams' history.  A stream
 * without a previous cycle (first call, after a reset, or beyond the B of every earlier call) reads zeros before its first
 * sample, like a fresh Receiver; the audio dtype may change from one call to the next. */
int ft8_decode_cycles_live(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even,
                           ft8_record* rec, int rec_capacity, int32_t* n_rec, int mem);
int ft8_live_reset(ft8_handle* h);

/* Progressive form of ft8_decode_cycles_live: the live decode of the open cycle of B streams, released hop by hop at the
 * hop a running reference Receiver emits each message (receiver.py:376-412, its scheduler loop run once after every hop,
 * with the clock one microsecond after the hop).  audio is each stream's cycle buffer [B][180000]: only samples
 * < 480 * hop are valid, and the call reads only those that arrived since its previous call.  hop increases strictly
 * within a cycle (1..375); B and odd_even stay.  The call that passes hop S = search_h0_hi + 173 (260 by default) searches
 * the ring as it is then and runs pass 0 on that snapshot; a candidate then runs pass k at hop d + k,
 * d = max(S + 1, h0 + 285), its fine stage on the audio buffer as the receiver holds it at hop d + 1.  A call returns the
 * records with emission hop e <= hop that earlier calls have not released, stream-major (ft8_record.cycle = stream) and in
 * emission order -- e, then llr_sd at that hop descending, then candidate rank -- with n_rec[B] per stream and emit_hop[i]
 * = e.  A record is a duplicate (emitted = 0) if an earlier one of the same stream-cycle, released or not, has its payload.
 * The call with hop = 375 completes the cycle: it releases everything left (e up to 377, in the next cycle's first hops)
 * and leaves ring, tail and previous cycle of every stream exactly as ft8_decode_cycles_live of the same audio does, so the
 * two entries can follow each other at cycle boundaries.  FT8_E_BADARG: hop not increasing, B or odd_even changed within a
 * cycle, odd_even equal to the last completed live cycle's, or ft8_decode_cycles_live / _seq called while a cycle is open
 * (ft8_live_reset abandons it).  Other calls (isolated decodes, stage ops) may come in between and do not disturb it.
 * Capacity as in ft8_decode_cycles (the released records count as released even when cut).  ft8_get_stats: the work of
 * this call (cycles = B only in the completing call); ft8_last_kernel_ms(0): the call's device time. */
int ft8_decode_cycles_live_progress(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even, int hop,
                                    ft8_record* rec, uint16_t* emit_hop, int rec_capacity, int32_t* n_rec, int mem);
/* The search hop S of ft8_decode_cycles_live_progress for this handle's search range (260 for the default range): the first
 * hop whose call searches; records can be released from hop S + 1 on. */
int ft8_progress_search_hop(ft8_handle* h, int* hop);

/* C consecutive live cycles of B streams in one call.  audio is [C][B][180000] (time-major: audio + c*B*180000 is the
 * batch a c-th ft8_decode_cycles_live call would get), so one stream's recording (B = 1) is one contiguous array.
 * Equivalent to, and bit-identical with:
 *     for c in 0..C-1: ft8_decode_cycles_live(h, audio + c*B*180000, audio_dtype, B, odd_even ^ (c & 1), ...)
 * records concatenated in that order, n_rec[C][B], and ft8_record.cycle = c*B + b.  The handle's live state (both ring
 * halves and the tail of each stream b < B) is left exactly as those C calls leave it, so ft8_decode_cycles_live and this
 * entry can follow each other in any order.  C*B may exceed cfg.max_cycles; B may not (FT8_E_CAPACITY).  The call works in
 * pieces of floor(max_cycles / B) consecutive cycles per stream, each one decode batch.  When rec_capacity is too small,
 * all C cycles are still decoded and the live state still advances past them; records beyond rec_capacity are dropped
 * cycle-major (n_rec trimmed to what was copied) and the call returns FT8_E_CAPACITY.  ft8_get_stats gives totals over the
 * call; ft8_last_kernel_ms: 0 = the whole call, 1-11 summed over the pieces. */
int ft8_decode_cycles_live_seq(ft8_handle* h, const void* audio, int audio_dtype, int B, int C, int odd_even,
                               ft8_record* rec, int rec_capacity, int32_t* n_rec, int mem);

/* Optional double buffering for callers that stream batches from host memory: starts the host->device copy of the NEXT
 * batch on a second stream and returns at once.  The host buffer must stay valid and UNCHANGED until the copy has been
 * consumed or dropped; pinned memory is needed for the copy to be asynchronous.  A pending prefetch is consumed only by
 * the next ft8_decode_cycles_stream call whose `audio`, dtype and B are the ones that were prefetched -- by naming the
 * buffer again through the streaming entry the caller states that it has not been rewritten.  Any other decode call
 * (plain ft8_decode_cycles included, or a streaming call on a different buffer) waits for the pending copy to finish and
 * drops it, so a stale device copy is never decoded and the host buffer is never read after that call returns. */
int ft8_prefetch_audio(ft8_handle* h, const void* audio_host, int audio_dtype, int B);

/* Page-locked host memory for the streaming entry points (the audio batches a caller refills, the record buffer):
 * flags bit 0 (FT8_HOST_WRITE_COMBINED) asks for write-combined memory -- meant for INPUT staging buffers the CPU only
 * writes and the GPU only reads; CPU reads of such memory are very slow.  Memory is portable across devices.  Replaces
 * nothing in the reference (its audio arrives through PyAudio callbacks, receiver.py:295-306); it exists so that a C or
 * ctypes caller does not need the CUDA runtime to get DMA-able buffers. */
#define FT8_HOST_WRITE_COMBINED 1
int  ft8_host_alloc(size_t bytes, int flags, void** out);
int  ft8_host_free(void* p);

/* Streaming form of ft8_decode_cycles for host audio: decodes `audio` (consuming its prefetched copy when there is one) and
 * at the same time starts the copy of `next_audio_host` (same dtype and B; NULL = none), i.e. one call per batch with a
 * one-batch look-ahead keeps the PCIe transfer entirely underneath the kernels. */
int ft8_decode_cycles_stream(ft8_handle* h, const void* audio, int audio_dtype, int B, int odd_even,
                             ft8_record* rec, int rec_capacity, int32_t* n_rec, const void* next_audio_host);

/* Workload generator on the device (SURVEY.md 8f rank 4; restates transmitter.py:52-70 + the 8d mixing recipe):
 * sums n_sig GFSK signals per cycle and white Gaussian noise into int16 audio[B][180000] (device or host per mem).
 * symbols: uint8 [B][n_sig][79]; f_hz, dt_s, amp: float [B][n_sig]. */
int ft8_synth_cycles(ft8_handle* h, const uint8_t* symbols, const float* f_hz, const float* dt_s, const float* amp,
                     int B, int n_sig, float noise_sigma, uint64_t seed, int16_t* audio, int mem);

/* Test hook: batched complex FFT through the library's shared-memory kernels (n in {32, 256, 375, 1920, 3200}). */
int ft8_debug_fft(ft8_handle* h, int n, int inverse, const float* in, float* out, int batch);

/* Test hook: the OSD attempts of pass 5 (the five AP patterns on one llr, with RR73, 73 and RRR sharing one reliability order
 * and basis, as the decode runs them) on host llr[N][174] -> found[N][5], bits91[N][5][3], attempt k as ft8_osd gives it
 * for the llr with AP pattern k applied. */
int ft8_debug_osd_ap(ft8_handle* h, const float* llr, int N, int singleflips, int doubleflips, int32_t* found,
                     uint32_t* bits91);

#ifdef __cplusplus
}
#endif
#endif /* FT8_B200_H */
