"""Engine: numpy-facing wrapper of one ft8_handle (one CUDA device + stream).

Every method passes caller-owned numpy buffers (FT8_MEM_HOST) through the C ABI; ``*_dev`` variants take raw
device pointers (e.g. ``torch.Tensor.data_ptr()``), PyTorch being only an optional carrier.  Errors raise
RuntimeError(ft8_last_error()).  Reference call sites replaced by each method are cited in include/ft8_b200.h.
"""
import ctypes as C
import threading

import numpy as np

from . import _lib as L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def bits91_to_int(w):
    """three LSB-first uint32 words -> python int whose bit 90-j is codeword bit j (reference's bits91_int)."""
    v = 0
    for j in range(91):
        v = (v << 1) | ((int(w[j >> 5]) >> (j & 31)) & 1)
    return v


def int_to_bits91(v):
    w = [0, 0, 0]
    for j in range(91):
        if (v >> (90 - j)) & 1:
            w[j >> 5] |= 1 << (j & 31)
    return np.array(w, np.uint32)


class _SerialisedLib:
    """Per-handle call gate.  One ft8_handle = one stream + one scratch arena, so its entry points must not run
    concurrently (INTEGRATION.md section 5) -- but ctypes releases the GIL, and the live Receiver calls the same handle
    from the audio callback (`hop_spectrum`) and from `manage_cycle` (`ft8_llr/ldpc/osd/fine`).  Every library call of
    an Engine therefore goes through this proxy, which holds the engine's lock for the duration of the call and, on
    failure, reads ft8_last_error while still holding it (kept per thread for `_check`)."""

    def __init__(self, lib, lock):
        self._lib, self._lock, self._tls = lib, lock, threading.local()

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        takes_handle = name not in ("ft8_default_cfg", "ft8_create")

        def call(*args):
            with self._lock:
                rc = fn(*args)
                if takes_handle and fn.restype is C.c_int and rc != L.OK:
                    self._tls.err = self._lib.ft8_last_error(args[0]).decode()
                return rc
        setattr(self, name, call)
        return call

    def last_error(self):
        return getattr(self._tls, "err", "")


class PinnedArray:
    """Page-locked host array from the library's allocator (ft8_host_alloc): `.array` is a numpy view, freed on close() /
    garbage collection.  write_combined=True is for input staging buffers the CPU only writes (CPU reads are very slow)."""

    def __init__(self, shape, dtype, write_combined=False):
        lib = L.load()
        self._lib = lib
        dtype = np.dtype(dtype)
        nbytes = int(np.prod(shape)) * dtype.itemsize
        p = C.c_void_p()
        rc = lib.ft8_host_alloc(nbytes, L.HOST_WRITE_COMBINED if write_combined else 0, C.byref(p))
        if rc != L.OK or not p.value:
            raise RuntimeError("ft8_host_alloc(%d bytes) failed: rc %d" % (nbytes, rc))
        self._p = p
        self.array = np.frombuffer((C.c_uint8 * nbytes).from_address(p.value), dtype=dtype).reshape(shape)

    def close(self):
        if getattr(self, "_p", None) is not None:
            self.array = None
            self._lib.ft8_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass



class Engine:
    def __init__(self, device=0, max_cycles=1, max_cands=200, sync_score_min=85.0, llr_sd_min=5.0,
                 osd_singleflips=30, osd_doubleflips=2, fine_mode=0,
                 search_f0_range=None, search_h0_range=None):
        self._lock = threading.RLock()
        self._lib = _SerialisedLib(L.load(), self._lock)
        cfg = L.Cfg()
        self._lib.ft8_default_cfg(C.byref(cfg))
        cfg.max_cycles, cfg.max_cands = int(max_cycles), int(max_cands)
        cfg.sync_score_min, cfg.llr_sd_min = float(sync_score_min), float(llr_sd_min)
        cfg.osd_singleflips, cfg.osd_doubleflips = int(osd_singleflips), int(osd_doubleflips)
        if search_f0_range is not None:                   # [lo, hi) in 3.125 Hz bins; None = reference default [32, 960)
            cfg.search_f0_lo, cfg.search_f0_hi = int(search_f0_range[0]), int(search_f0_range[1])
        if search_h0_range is not None:                   # [lo, hi) in 40 ms hops; None = reference default [-37, 87)
            cfg.search_h0_lo, cfg.search_h0_hi = int(search_h0_range[0]), int(search_h0_range[1])
        cfg.fine_mode = int(fine_mode)                    # 0: tensor-core frequency scan (default), 1: nine-FFT kernel (A/B)
        self.cfg = cfg
        self._h = C.c_void_p()
        rc = self._lib.ft8_create(int(device), C.byref(cfg), C.byref(self._h))
        if rc != L.OK:
            msg = self._lib.ft8_last_error(None).decode()
            self._h = None
            raise RuntimeError(f"ft8_create failed ({rc}): {msg}")
        self.device = int(device)
        self.max_cycles, self.max_cands = int(max_cycles), int(max_cands)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.ft8_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != L.OK:
            raise RuntimeError(f"libft8_b200 error {rc}: {self._lib.last_error()}")

    @staticmethod
    def _audio(audio):
        a = np.ascontiguousarray(audio)
        if a.ndim == 1:
            a = a[None, :]
        if a.shape[1] != 180000:
            raise ValueError("audio must be [B, 180000] (one 15 s cycle at 12 kHz per row)")
        if a.dtype == np.int16:
            return a, L.AUDIO_I16
        if a.dtype == np.float32:
            return a, L.AUDIO_F32
        raise ValueError("audio dtype must be int16 or float32")

    # ---- S1
    def spectrogram(self, audio):
        a, dt = self._audio(audio)
        out = np.empty((a.shape[0], L.GRID_ROWS, L.GRID_COLS), np.float32)
        self._check(self._lib.ft8_spectrogram(self._h, _ptr(a), dt, a.shape[0], _ptr(out), L.MEM_HOST))
        return out

    def hop_spectrum(self, audio_buffer):
        """AudioIn.get_hop_spectrum: dB row of the window over the last 3840 samples of the 180000-sample ring buffer."""
        a, dt = self._audio(audio_buffer)
        out = np.empty(L.GRID_COLS, np.float32)
        self._check(self._lib.ft8_hop_spectrum(self._h, _ptr(a), dt, _ptr(out), L.MEM_HOST))
        return out

    # ---- S2
    def sync(self, grid, odd_even=0, want_payload=True):
        g = np.ascontiguousarray(grid, np.float32)
        if g.ndim == 2:
            g = g[None]
        B, rows, cols = g.shape
        assert cols == L.GRID_COLS and rows in (L.GRID_ROWS, L.GRID_ROWS_LIVE)
        K = self.max_cands
        f0 = np.zeros((B, K), np.int16)
        h0 = np.zeros((B, K), np.int16)
        sc = np.zeros((B, K), np.float32)
        n = np.zeros(B, np.int32)
        pay = np.zeros((B, K, 58, 8), np.float32) if want_payload else None
        self._check(self._lib.ft8_sync(self._h, _ptr(g), rows, B, int(odd_even), _ptr(f0), _ptr(h0), _ptr(sc), _ptr(n),
                                       _ptr(pay), L.MEM_HOST))
        return f0, h0, sc, n, pay

    # ---- L0
    def llr(self, payload_db):
        p = np.ascontiguousarray(payload_db, np.float32).reshape(-1, 58, 8)
        N = p.shape[0]
        llr = np.empty((N, 174), np.float32)
        sd = np.empty(N, np.float32)
        snr = np.empty(N, np.int32)
        self._check(self._lib.ft8_llr(self._h, _ptr(p), N, _ptr(llr), _ptr(sd), _ptr(snr), L.MEM_HOST))
        return llr, sd, snr

    # ---- F1
    def cycle_spectrum(self, audio):
        a, dt = self._audio(audio)
        out = np.empty((a.shape[0], L.SPEC_BINS), np.complex64)
        self._check(self._lib.ft8_cycle_spectrum(self._h, _ptr(a), dt, a.shape[0], _ptr(out), L.MEM_HOST))
        return out

    # ---- F2/F3
    def fine(self, spec, cycle_of, f0_idx, h0_idx, want_grid=True):
        s = np.ascontiguousarray(spec, np.complex64)
        if s.ndim == 1:
            s = s[None]
        assert s.shape[1] == L.SPEC_BINS
        co = np.ascontiguousarray(cycle_of, np.int32)
        f0 = np.ascontiguousarray(f0_idx, np.int16)
        h0 = np.ascontiguousarray(h0_idx, np.int16)
        N = len(co)
        tt, ff, ns, snr = (np.empty(N, np.int32) for _ in range(4))
        sd = np.empty(N, np.float32)
        llr = np.empty((N, 174), np.float32)
        sg = np.empty((N, 79, 8), np.float32) if want_grid else None
        self._check(self._lib.ft8_fine(self._h, _ptr(s), s.shape[0], _ptr(co), _ptr(f0), _ptr(h0), N, _ptr(tt), _ptr(ff),
                                       _ptr(ns), _ptr(sg), _ptr(llr), _ptr(sd), _ptr(snr), L.MEM_HOST))
        return dict(tt=tt, ff=ff, nsync=ns, grid=sg, llr=llr, sd=sd, snr=snr)

    # ---- L1/L2
    def ldpc(self, llr, max_ncheck0, max_iters):
        """llr [N,174] float32 is updated in place (like the reference). Returns status, nits, bits91[N,3]."""
        assert llr.dtype == np.float32 and llr.flags.c_contiguous and llr.shape[-1] == 174
        N = llr.size // 174
        st = np.empty(N, np.int32)
        ni = np.empty(N, np.int32)
        bits = np.empty((N, 3), np.uint32)
        self._check(self._lib.ft8_ldpc(self._h, _ptr(llr), N, int(max_ncheck0), int(max_iters), _ptr(st), _ptr(ni),
                                       _ptr(bits), L.MEM_HOST))
        return st, ni, bits

    # ---- O1
    def osd(self, llr, singleflips=30, doubleflips=2):
        x = np.ascontiguousarray(llr, np.float32).reshape(-1, 174)
        N = x.shape[0]
        found = np.empty(N, np.int32)
        bits = np.empty((N, 3), np.uint32)
        self._check(self._lib.ft8_osd(self._h, _ptr(x), N, int(singleflips), int(doubleflips), _ptr(found), _ptr(bits),
                                      L.MEM_HOST))
        return found, bits

    # ---- K1
    def crc14(self, bits91):
        b = np.ascontiguousarray(bits91, np.uint32).reshape(-1, 3)
        flags = np.empty(b.shape[0], np.int32)
        self._check(self._lib.ft8_crc14(self._h, _ptr(b), b.shape[0], _ptr(flags), L.MEM_HOST))
        return flags

    # ---- whole path
    def _outputs(self, B, rec, n):
        """The record and count outputs of a decode of B cycles: new arrays, or the caller's after checking them (the library
        writes up to len(rec) 64-byte records into `rec` and B int32 counts into `n`)."""
        if rec is None:
            rec = np.zeros(B * self.max_cands, L.RECORD_DTYPE)
        elif rec.dtype != L.RECORD_DTYPE or not rec.flags.c_contiguous:
            raise ValueError("rec must be a contiguous RECORD_DTYPE array")
        if n is None:
            n = np.zeros(B, np.int32)
        elif n.dtype != np.int32 or len(n) < B or not n.flags.c_contiguous:
            raise ValueError("n must be a contiguous int32 array of at least B entries")
        return rec, n

    def decode_cycles(self, audio, odd_even=0, next_audio=None, rec=None, n=None):
        """audio [B,180000] int16/float32 -> (records structured array in emission order, n_rec[B]).

        `rec` / `n`: optional caller-owned output arrays (RECORD_DTYPE[>= B*max_cands is always enough], int32[B]); pass
        pinned ones to make the record copy-back a straight DMA.  The returned records are a view of `rec`.

        Streaming: pass the following batch as `next_audio` (same shape/dtype, ideally pinned); its host->device copy runs
        underneath this batch's kernels and the next call consumes it (ft8_decode_cycles_stream)."""
        a, dt = self._audio(audio)
        B = a.shape[0]
        rec, n = self._outputs(B, rec, n)
        cap = len(rec)
        pending = getattr(self, "_pf_ref", None)
        # a prefetched copy is consumed only through the streaming entry, and only for the very array that was named
        mine = pending is not None and pending.ctypes.data == a.ctypes.data and pending.shape == a.shape
        if next_audio is None and not mine:
            self._check(self._lib.ft8_decode_cycles(self._h, _ptr(a), dt, B, int(odd_even), _ptr(rec), cap, _ptr(n), L.MEM_HOST))
            self._pf_ref = None                            # the library waited for (and dropped) any pending copy
        else:
            nx = None
            if next_audio is not None:
                nx, ndt = self._audio(next_audio)
                if ndt != dt or nx.shape != a.shape:
                    raise ValueError("next_audio must have the dtype and shape of audio")
            self._check(self._lib.ft8_decode_cycles_stream(self._h, _ptr(a), dt, B, int(odd_even), _ptr(rec), cap, _ptr(n), _ptr(nx)))
            self._pf_ref = nx                              # keeps the host buffer alive until its copy is consumed or dropped
        return rec[:int(n[:B].sum())], n[:B]

    def decode_cycles_live(self, audio, odd_even, rec=None, n=None):
        """Next 15 s of B live streams (row b = stream b): like decode_cycles, but against the handle's per-stream two-cycle
        waterfall ring and previous-cycle tail (ft8_decode_cycles_live) -- what a running reference Receiver decodes.
        Alternate odd_even 0, 1, 0, ... call after call; live_reset() forgets the history."""
        a, dt = self._audio(audio)
        B = a.shape[0]
        rec, n = self._outputs(B, rec, n)
        self._check(self._lib.ft8_decode_cycles_live(self._h, _ptr(a), dt, B, int(odd_even), _ptr(rec), len(rec), _ptr(n), L.MEM_HOST))
        return rec[:int(n[:B].sum())], n[:B]

    def decode_cycles_live_seq(self, audio, odd_even, rec=None, n=None):
        """C consecutive live cycles of B streams in one call (ft8_decode_cycles_live_seq): audio [C, B, 180000], or
        [C, 180000] for one stream, int16/float32, cycle c of parity odd_even ^ (c & 1).  Bit-identical with C
        decode_cycles_live calls, and leaves the same live state.  Returns (records, n[C, B]); a record's `cycle` is c*B + b.
        `n`, when given, is a flat int32 array of at least C*B entries."""
        a = np.ascontiguousarray(audio)
        if a.ndim == 2:
            a = a[:, None, :]
        if a.ndim != 3 or a.shape[2] != 180000 or a.shape[0] == 0 or a.shape[1] == 0:
            raise ValueError("audio must be [C, B, 180000] or [C, 180000] (C consecutive 15 s cycles of B streams)")
        if a.dtype == np.int16:
            dt = L.AUDIO_I16
        elif a.dtype == np.float32:
            dt = L.AUDIO_F32
        else:
            raise ValueError("audio dtype must be int16 or float32")
        C_, B = a.shape[:2]
        rec, n = self._outputs(C_ * B, rec, n)
        self._check(self._lib.ft8_decode_cycles_live_seq(self._h, _ptr(a), dt, B, C_, int(odd_even), _ptr(rec), len(rec), _ptr(n),
                                                         L.MEM_HOST))
        return rec[:int(n[:C_ * B].sum())], n[:C_ * B].reshape(C_, B)

    def live_reset(self):
        self._check(self._lib.ft8_live_reset(self._h))

    def prefetch(self, audio):
        """Start copying the NEXT batch (host array, ideally pinned) while the current one is being decoded; the following
        decode_cycles(audio) with the same array consumes the copy (ft8_prefetch_audio)."""
        a, dt = self._audio(audio)
        self._pf_ref = a                               # keep the host buffer alive until it is consumed
        self._check(self._lib.ft8_prefetch_audio(self._h, _ptr(a), dt, a.shape[0]))

    def decode_cycles_dev(self, audio_ptr, dtype, B, odd_even=0, rec=None, n=None):
        """Same, with audio already resident on this engine's device (raw pointer)."""
        rec, n = self._outputs(B, rec, n)
        self._check(self._lib.ft8_decode_cycles(self._h, C.c_void_p(audio_ptr), dtype, B, int(odd_even), _ptr(rec), len(rec),
                                                _ptr(n), L.MEM_DEVICE))
        return rec[:int(n[:B].sum())], n[:B]

    def stats(self):
        s = L.Stats()
        self._check(self._lib.ft8_get_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in L.Stats._fields_ if k != "reserved"}

    def last_kernel_ms(self, which):
        v = C.c_float()
        self._check(self._lib.ft8_last_kernel_ms(self._h, int(which), C.byref(v)))
        return float(v.value)

    def synchronize(self):
        self._check(self._lib.ft8_synchronize(self._h))

    # ---- generator / test hook
    def synth_cycles(self, symbols, f_hz, dt_s, amp, noise_sigma=1000.0, seed=0, out_ptr=None):
        sym = np.ascontiguousarray(symbols, np.uint8)
        B, n_sig = sym.shape[0], sym.shape[1]
        f = np.ascontiguousarray(f_hz, np.float32)
        d = np.ascontiguousarray(dt_s, np.float32)
        am = np.ascontiguousarray(amp, np.float32)
        if out_ptr is None:
            out = np.empty((B, 180000), np.int16)
            self._check(self._lib.ft8_synth_cycles(self._h, _ptr(sym), _ptr(f), _ptr(d), _ptr(am), B, n_sig, float(noise_sigma),
                                                   int(seed), _ptr(out), L.MEM_HOST))
            return out
        self._check(self._lib.ft8_synth_cycles(self._h, _ptr(sym), _ptr(f), _ptr(d), _ptr(am), B, n_sig, float(noise_sigma),
                                               int(seed), C.c_void_p(out_ptr), L.MEM_DEVICE))
        return None

    def debug_fft(self, x, inverse=False):
        a = np.ascontiguousarray(x, np.complex64)
        if a.ndim == 1:
            a = a[None]
        out = np.empty_like(a)
        self._check(self._lib.ft8_debug_fft(self._h, a.shape[1], int(bool(inverse)), _ptr(a), _ptr(out), a.shape[0]))
        return out
