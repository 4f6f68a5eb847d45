"""The handle's host layer: how the stand-alone entry points stage caller buffers, how its scratch grows, its argument
errors, and the caller-supplied outputs of the Engine's decode methods.

- Every stand-alone entry point gives bit-identical results with device buffers (torch tensors, FT8_MEM_DEVICE) and with
  host buffers (numpy, FT8_MEM_HOST), on golden cycles.
- A handle whose scratch grows and shrinks over a sequence of calls answers each call as a fresh handle does.
- Bad calls return their error codes and messages.
- Without a GPU: Engine's decode methods reject a wrong `rec` / `n` before calling the library.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import cycle_audio
from pyft8_b200 import _lib as L
from pyft8_b200.engine import Engine, _ptr


def _call(eng, name, args, mem):
    """Calls `name`(handle, *args, mem).  Numpy arrays in `args` are copied first and, for FT8_MEM_DEVICE, passed as torch
    tensors on the engine's device; returns the arrays as they are after the call."""
    arrays = [a.copy() if isinstance(a, np.ndarray) else a for a in args]
    if mem == L.MEM_DEVICE:
        import torch
        dev = torch.device("cuda", eng.device)
        tensors = [torch.from_numpy(a.reshape(-1).view(np.uint8)).to(dev) if isinstance(a, np.ndarray) else None
                   for a in arrays]
        torch.cuda.synchronize(dev)
        cargs = [C.c_void_p(t.data_ptr()) if t is not None else a for a, t in zip(arrays, tensors)]
    else:
        cargs = [_ptr(a) if isinstance(a, np.ndarray) else a for a in arrays]
    eng._check(getattr(eng._lib, name)(eng._h, *cargs, mem))
    if mem == L.MEM_DEVICE:
        for a, t in zip(arrays, tensors):
            if t is not None:
                a[...] = t.cpu().numpy().view(a.dtype).reshape(a.shape)
    return [a for a in arrays if isinstance(a, np.ndarray)]


def _same(x, y):
    return x.shape == y.shape and x.tobytes() == y.tobytes()


def _both(eng, name, *args):
    """Results of one call with host and with device buffers; asserts they are bit-identical."""
    host = _call(eng, name, args, L.MEM_HOST)
    dev = _call(eng, name, args, L.MEM_DEVICE)
    for i, (a, b) in enumerate(zip(host, dev)):
        assert _same(a, b), (name, i)
    return host


@pytest.fixture(scope="module")
def inputs():
    audio = np.stack([cycle_audio("test_09"), cycle_audio("syn20")])
    return audio


@pytest.mark.gpu
def test_device_buffers_give_the_host_results(inputs):
    audio = inputs
    B, K = audio.shape[0], 200
    eng = Engine(max_cycles=B, max_cands=K)
    try:
        _both(eng, "ft8_spectrogram", audio, L.AUDIO_I16, B, np.zeros((B, L.GRID_ROWS, L.GRID_COLS), np.float32))
        _both(eng, "ft8_spectrogram", audio.astype(np.float32), L.AUDIO_F32, B,
              np.zeros((B, L.GRID_ROWS, L.GRID_COLS), np.float32))
        _both(eng, "ft8_hop_spectrum", audio[0], L.AUDIO_I16, np.zeros(L.GRID_COLS, np.float32))
        grid = eng.spectrogram(audio)
        cand = [np.zeros((B, K), np.int16), np.zeros((B, K), np.int16), np.zeros((B, K), np.float32), np.zeros(B, np.int32)]
        _, f0, h0, _, n, pay = _both(eng, "ft8_sync", grid, L.GRID_ROWS, B, 0, *cand, np.zeros((B, K, 58, 8), np.float32))
        assert n.min() > 0
        ring = np.concatenate([grid[:, 1:], grid[:, 1:]], axis=1)[:, :L.GRID_ROWS_LIVE]
        _both(eng, "ft8_sync", np.ascontiguousarray(ring), L.GRID_ROWS_LIVE, B, 1, *cand, None)
        N = int(n.sum())
        sel = np.concatenate([np.arange(b * K, b * K + n[b]) for b in range(B)])
        _, llr, _, _ = _both(eng, "ft8_llr", pay.reshape(-1, 58, 8)[sel], N, np.zeros((N, 174), np.float32),
                          np.zeros(N, np.float32), np.zeros(N, np.int32))
        _, spec = _both(eng, "ft8_cycle_spectrum", audio, L.AUDIO_I16, B, np.zeros((B, L.SPEC_BINS), np.complex64))
        _both(eng, "ft8_cycle_spectrum", audio.astype(np.float32), L.AUDIO_F32, B, np.zeros((B, L.SPEC_BINS), np.complex64))
        cyc = (sel // K).astype(np.int32)
        f0s, h0s = f0.reshape(-1)[sel], h0.reshape(-1)[sel]
        for want_grid in (True, False):
            args = [spec, B, cyc, f0s, h0s, N, np.zeros(N, np.int32), np.zeros(N, np.int32), np.zeros(N, np.int32),
                    np.zeros((N, 79, 8), np.float32) if want_grid else None,
                    np.zeros((N, 174), np.float32), np.zeros(N, np.float32), np.zeros(N, np.int32)]
            host = _call(eng, "ft8_fine", args, L.MEM_HOST)[4:]           # tt, ff, nsync, [grid], llr, sd, snr
            dev = _call(eng, "ft8_fine", args, L.MEM_DEVICE)[4:]
            ok = host[2] > 6
            assert 0 < ok.sum() < N
            for i, (x, y) in enumerate(zip(host, dev)):
                if not want_grid and i == 3:          # without a signal grid, llr is written only where nsync > 6
                    x, y = x[ok], y[ok]
                assert _same(x, y), ("ft8_fine", want_grid, i)
        st, _, bits = _both(eng, "ft8_ldpc", llr, N, 90, 20, np.zeros(N, np.int32), np.zeros(N, np.int32),
                            np.zeros((N, 3), np.uint32))[1:]
        assert (st == L.LDPC_OK).any()
        _both(eng, "ft8_osd", llr, N, 30, 2, np.zeros(N, np.int32), np.zeros((N, 3), np.uint32))
        _both(eng, "ft8_crc14", bits, N, np.zeros(N, np.int32))
        rng = np.random.default_rng(5)
        sym = rng.integers(0, 8, (B, 3, 79)).astype(np.uint8)
        f = rng.uniform(300, 2500, (B, 3)).astype(np.float32)
        d = rng.uniform(-0.5, 1.0, (B, 3)).astype(np.float32)
        am = np.full((B, 3), 300.0, np.float32)
        _both(eng, "ft8_synth_cycles", sym, f, d, am, B, 3, 1000.0, 17, np.zeros((B, 180000), np.int16))
    finally:
        eng.close()


def _fine(eng, spec, cands, N):
    """ft8_fine on the first N of `cands` (repeated as often as needed)."""
    cyc, f0, h0 = (np.resize(c, N) for c in cands)
    return eng.fine(spec, cyc, f0, h0)


def _decode(eng, audio, **kw):
    rec, n = eng.decode_cycles(audio, **kw)
    return rec.copy(), n.copy()


def _equal(x, y):
    if isinstance(x, dict):
        return x.keys() == y.keys() and all(_equal(x[k], y[k]) for k in x)
    if isinstance(x, (tuple, list)):
        return len(x) == len(y) and all(_equal(a, b) for a, b in zip(x, y))
    return (x is None and y is None) or _same(x, y)


@pytest.mark.gpu
def test_growing_and_shrinking_scratch_answers_like_a_fresh_handle(inputs):
    """The arena, the fine-stage temporaries (N above max_cycles * max_cands) and the prefetch slot (a larger B than any
    before) grow on one handle over a sequence of calls whose needs rise and fall; every call must answer as it does on a
    fresh handle."""
    audio = inputs
    cfg = dict(max_cycles=2, max_cands=50)
    ref = Engine(**cfg)
    grid = ref.spectrogram(audio)
    spec = ref.cycle_spectrum(audio)
    f0, h0, _, n, pay = ref.sync(grid)
    ref.close()
    sel = np.concatenate([np.arange(b * 50, b * 50 + n[b]) for b in range(2)])
    cands = ((sel // 50).astype(np.int32), f0.reshape(-1)[sel], h0.reshape(-1)[sel])
    payload = np.ascontiguousarray(np.resize(pay.reshape(-1, 58, 8)[sel], (300, 58, 8)))
    bits = np.random.default_rng(3).integers(0, 2 ** 32, (300, 3), dtype=np.uint64).astype(np.uint32)
    a1, a1_next, a2 = audio[:1].copy(), audio[1:].copy(), audio.copy()
    steps = [
        ("llr 4", lambda e: e.llr(payload[:4])),
        ("spectrogram B=2", lambda e: e.spectrogram(audio)),
        ("llr 300", lambda e: e.llr(payload)),
        ("crc 3", lambda e: e.crc14(bits[:3])),
        ("fine N=300", lambda e: _fine(e, spec, cands, 300)),
        ("fine N=20", lambda e: _fine(e, spec[:1], [c[cands[0] == 0] for c in cands], 20)),
        ("cycle spectrum B=1", lambda e: e.cycle_spectrum(audio[1:])),
        ("hop spectrum", lambda e: e.hop_spectrum(audio[1])),
        ("sync 376 rows", lambda e: e.sync(grid)),
        ("osd 8", lambda e: e.osd(e.llr(payload[:8])[0])),
        ("decode B=1 naming the next batch", lambda e: _decode(e, a1, next_audio=a1_next)),
        ("decode of the prefetched batch", lambda e: _decode(e, a1_next)),
    ]
    eng = Engine(**cfg)
    try:
        for name, fn in steps:
            got = fn(eng)
            fresh = Engine(**cfg)
            want = fn(fresh)
            fresh.close()
            assert _equal(got, want), name
        eng.prefetch(a2)                                    # B = 2: the prefetch slot grows
        got = _decode(eng, a2)
        assert eng.stats()["cycles"] == 2
        fresh = Engine(**cfg)
        assert _equal(got, _decode(fresh, a2))
        fresh.close()
    finally:
        eng.close()


@pytest.mark.gpu
def test_bad_calls_return_their_codes_and_messages(inputs):
    eng = Engine(max_cycles=2, max_cands=50)
    lib, h, P = eng._lib, eng._h, _ptr
    a3 = np.zeros((3, 180000), np.int16)
    grid3 = np.zeros((3, L.GRID_ROWS_LIVE, L.GRID_COLS), np.float32)
    big = np.zeros(3 * L.SPEC_BINS * 2, np.float32)
    k = [np.zeros(3 * 50, np.int32) for _ in range(4)]
    pay = np.zeros((2, 50, 58, 8), np.float32)
    rec = np.zeros(100, L.RECORD_DTYPE)
    nrec = np.zeros(3, np.int32)
    spec = np.zeros((1, L.SPEC_BINS), np.complex64)
    one = lambda v, t: np.array([v], t)
    out = [np.zeros(1, np.int32) for _ in range(3)] + [np.zeros((1, 79, 8), np.float32), np.zeros((1, 174), np.float32),
                                                        np.zeros(1, np.float32), np.zeros(1, np.int32)]
    fine = lambda cyc, f0, h0: lib.ft8_fine(h, P(spec), 1, P(one(cyc, np.int32)), P(one(f0, np.int16)), P(one(h0, np.int16)), 1,
                                            *map(P, out), L.MEM_HOST)
    capacity = "B exceeds cfg.max_cycles"
    dtype = "audio_dtype must be FT8_AUDIO_I16 or FT8_AUDIO_F32"
    fine_range = "ft8_fine: candidate outside the supported range (-100 <= h0 <= 200, 4 <= f0 <= 1880, 0 <= cycle_of < B)"
    table = [
        (lambda: lib.ft8_spectrogram(h, P(a3), 0, 3, P(big), L.MEM_HOST), L.E_CAPACITY, "ft8_spectrogram: " + capacity),
        (lambda: lib.ft8_cycle_spectrum(h, P(a3), 0, 3, P(big), L.MEM_HOST), L.E_CAPACITY, "ft8_cycle_spectrum: " + capacity),
        (lambda: lib.ft8_sync(h, P(grid3), L.GRID_ROWS, 3, 0, *map(P, k), None, L.MEM_HOST), L.E_CAPACITY, "ft8_sync: " + capacity),
        (lambda: lib.ft8_prefetch_audio(h, P(a3), 0, 3), L.E_CAPACITY, "ft8_prefetch_audio: " + capacity),
        (lambda: lib.ft8_decode_cycles(h, P(a3), 0, 3, 0, P(rec), 100, P(nrec), L.MEM_HOST), L.E_CAPACITY,
         "ft8_decode_cycles: " + capacity),
        (lambda: lib.ft8_spectrogram(h, P(a3), 2, 1, P(big), L.MEM_HOST), L.E_BADARG, dtype),
        (lambda: lib.ft8_hop_spectrum(h, P(a3), 2, P(big), L.MEM_HOST), L.E_BADARG, dtype),
        (lambda: lib.ft8_cycle_spectrum(h, P(a3), 2, 1, P(big), L.MEM_HOST), L.E_BADARG, dtype),
        (lambda: lib.ft8_decode_cycles(h, P(a3), 2, 1, 0, P(rec), 100, P(nrec), L.MEM_HOST), L.E_BADARG, dtype),
        (lambda: lib.ft8_decode_cycles_live(h, P(a3), 2, 1, 0, P(rec), 100, P(nrec), L.MEM_HOST), L.E_BADARG, dtype),
        (lambda: lib.ft8_prefetch_audio(h, P(a3), 2, 1), L.E_BADARG, "ft8_prefetch_audio: bad argument"),
        (lambda: lib.ft8_sync(h, P(grid3), L.GRID_ROWS_LIVE, 2, 0, *map(P, k), P(pay), L.MEM_HOST), L.E_BADARG,
         "ft8_sync: payload_db with a host 750-row grid is not supported; pass grid_rows=376 or device memory"),
        (lambda: lib.ft8_sync(h, P(grid3), 100, 1, 0, *map(P, k), None, L.MEM_HOST), L.E_BADARG,
         "ft8_sync: grid_rows must be 376 or 750"),
        (lambda: fine(0, 100, 201), L.E_BADARG, fine_range),
        (lambda: fine(0, 100, -101), L.E_BADARG, fine_range),
        (lambda: fine(0, 1881, 10), L.E_BADARG, fine_range),
        (lambda: fine(0, 3, 10), L.E_BADARG, fine_range),
        (lambda: fine(1, 100, 10), L.E_BADARG, fine_range),
        (lambda: lib.ft8_decode_cycles_live(h, P(a3), 0, 1, 2, P(rec), 100, P(nrec), L.MEM_HOST), L.E_BADARG,
         "ft8_decode_cycles_live: odd_even must be 0 or 1"),
        (lambda: lib.ft8_osd(h, P(big), 1, 92, 2, P(k[0]), P(k[1]), L.MEM_HOST), L.E_BADARG,
         "ft8_osd: bad argument (singleflips must be 0..91)"),
        (lambda: lib.ft8_synth_cycles(h, P(big), P(big), P(big), P(big), 1, 129, 1.0, 0, P(a3), L.MEM_HOST), L.E_BADARG,
         "ft8_synth_cycles: bad argument (n_sig <= 128)"),
        (lambda: lib.ft8_debug_fft(h, 100, 0, P(big), P(big), 1), L.E_BADARG,
         "ft8_debug_fft: n must be 32, 256, 375, 1920 or 3200"),
        (lambda: lib.ft8_decode_cycles(h, P(inputs[:1].copy()), 0, 1, 0, P(rec), 1, P(nrec), L.MEM_HOST), L.E_CAPACITY,
         "ft8_decode_cycles: rec_capacity too small (records truncated)"),
    ]
    try:
        for i, (call, code, msg) in enumerate(table):
            assert call() == code, (i, msg)
            assert lib.ft8_last_error(h).decode() == msg, i
        assert nrec[0] == 1                                # the truncated decode's counts are trimmed to what was copied
        assert lib.ft8_last_kernel_ms(h, 12, C.byref(C.c_float())) == L.E_BADARG
        rec, n = eng.decode_cycles(inputs[:1])             # the handle still decodes after every refusal
        assert n[0] > 0
    finally:
        eng.close()


class _FakeLib:
    """Stands in for the library: records the names of the calls and returns FT8_OK without touching any buffer."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def call(*args):
            self.calls.append(name)
            return L.OK
        return call

    def last_error(self):
        return ""


@pytest.mark.parametrize("method", ["decode_cycles", "decode_cycles_live", "decode_cycles_dev"])
def test_decode_methods_reject_bad_caller_outputs(method):
    B = 2
    eng = Engine.__new__(Engine)
    eng._lib, eng._h, eng.max_cands = _FakeLib(), None, 4
    audio = np.zeros((B, 180000), np.int16)
    decode = {"decode_cycles": lambda **kw: eng.decode_cycles(audio, **kw),
              "decode_cycles_live": lambda **kw: eng.decode_cycles_live(audio, 0, **kw),
              "decode_cycles_dev": lambda **kw: eng.decode_cycles_dev(0, L.AUDIO_I16, B, **kw)}[method]
    bad = [dict(rec=np.zeros(B * 4 * 64, np.uint8)),
           dict(rec=np.zeros((B * 4, 2), L.RECORD_DTYPE)[:, 0]),
           dict(n=np.zeros(B, np.int64)),
           dict(n=np.zeros(B - 1, np.int32)),
           dict(n=np.zeros(2 * B, np.int32)[::2])]
    for kw in bad:
        with pytest.raises(ValueError):
            decode(**kw)
    assert eng._lib.calls == []
    decode(rec=np.zeros(B * 4, L.RECORD_DTYPE), n=np.zeros(B, np.int32))
    assert eng._lib.calls == ["ft8_decode_cycles_live" if method == "decode_cycles_live" else "ft8_decode_cycles"]
