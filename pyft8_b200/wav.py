"""WAV ingest / export for the batch path (SURVEY.md 8f rank 4): 12 kHz mono int16 recordings <-> [n_cycles, 180000] arrays.

The reference's fixtures (tests/pipeline/*.wav) and its own writer (transmitter.py:79-85) use 12 kHz, mono, 16 bit; a
recording is cut into consecutive 15 s cycles (the last one zero-padded), which is exactly the `audio` argument of
Engine.decode_cycles / decode_cycles_live / Receiver.decode_cycles.  Standard library only.
"""
import wave

import numpy as np

SAMP_RATE = 12000
CYCLE_SAMPLES = 180000


def read_wav(path, start_sample=0):
    """-> int16 [n_cycles, 180000].  `start_sample` aligns the first cycle (e.g. a recording that starts mid-cycle)."""
    with wave.open(path, "rb") as w:
        if w.getframerate() != SAMP_RATE or w.getnchannels() != 1 or w.getsampwidth() != 2:
            raise ValueError(f"{path}: need 12 kHz mono 16-bit PCM (got {w.getframerate()} Hz, {w.getnchannels()} ch, "
                             f"{8 * w.getsampwidth()} bit)")
        x = np.frombuffer(w.readframes(w.getnframes()), dtype="<i2")
    x = x[start_sample:]
    n = max(1, -(-len(x) // CYCLE_SAMPLES))
    out = np.zeros((n, CYCLE_SAMPLES), np.int16)
    out.reshape(-1)[:len(x)] = x
    return out


def write_wav(path, audio):
    """int16 [n_cycles, 180000] or [n_samples] -> 12 kHz mono 16-bit WAV (the format transmitter.py:79-85 writes)."""
    a = np.ascontiguousarray(audio, dtype="<i2").reshape(-1)
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(SAMP_RATE)
        w.writeframes(a.tobytes())


def decode_wav(path, receiver=None, live=False, **kw):
    """Decode a recording: list (per 15 s cycle) of message dicts.  live=True keeps the two-cycle waterfall ring across the
    recording's consecutive cycles (Engine.decode_cycles_live_seq, the first cycle even) instead of decoding each cycle in
    isolation."""
    from .receiver import Receiver, format_records
    audio = read_wav(path)
    rx = receiver or Receiver("", None, **kw)
    if not live:
        return rx.decode_cycles(audio, emit=False)
    from .engine import Engine
    # the library decodes the recording in pieces of max_cycles cycles, chained through the live state
    eng = Engine(device=rx._device, max_cycles=min(len(audio), 256), max_cands=rx.max_cands, sync_score_min=rx.sync_score_min,
                 search_f0_range=rx._search_ranges[0], search_h0_range=rx._search_ranges[1])
    rec, n = eng.decode_cycles_live_seq(audio, 0)
    eng.close()
    out, off = [], 0
    for k in n[:, 0].tolist():
        # one cycle per unpacking batch, like a live receiver, so that hashed calls ('<...>') resolve as they do there
        mb = format_records(rec[off:off + k])
        off += k
        out.append([t for t, keep in zip(mb.text.tolist(), mb.keep.tolist()) if keep])
    return out
