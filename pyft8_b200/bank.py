"""Many live receivers multiplexed onto one GPU (SURVEY.md section 8f rank 3).

The reference runs one `Receiver` per audio device: a PyAudio callback appends 480-sample hops (receiver.py:295-306) and
`manage_cycle` (receiver.py:372-412) searches and decodes once enough of the cycle has arrived.  A skimmer-scale
deployment has hundreds of such streams; one B200 decodes ~30 k cycles/s, so the natural shape is: every stream appends
into its own 15-s slot of a pinned [R, 180000] int16 batch, and when a cycle closes the whole batch goes through
`ft8_decode_cycles_stream` once (isolated-cycle semantics, SURVEY H5) while the streams keep filling the other half of
the double buffer.  Decoding runs on a worker thread; `feed()` only waits when it has to write into the half the decoder
is still reading (a stream that runs a whole cycle ahead of the decoder).  `feed`/`feed_all` may be called from
several audio threads: the ring positions and the close-of-cycle decision are guarded by one lock.

What is kept from the reference surface: `on_message(dict)` with the keys of `check_and_package` (receiver.py:61-64)
plus 'receiver'; `set_band(r, band)`; per-receiver waterfall rows on request (`waterfall(r)`, the 376 x 976 dB grid the
GUI reads, receiver.py:272-278); and the live waterfall semantics: each receiver's 750-row two-cycle ring lives on the
device (`live_ring=True`, ft8_decode_cycles_live), so the first hops of a cycle see the previous cycle's audio and early
candidates (h0 < -32) read the previous cycle's rows, exactly like a running reference Receiver (receiver.py:295-306,
360).  By default a cycle is searched and decoded when its 15 s are complete (the reference starts searching 10.4 s into
the cycle and decodes candidates as their payload region fills, receiver.py:389-407): the messages are the same and come
out in the same order, up to 4.6 s later.  With `progressive=True` the bank follows the reference's schedule too
(ft8_decode_cycles_live_progress): once the slowest receiver has passed the search hop, a progress call every
`progress_hops` hops releases each message at the hop a running Receiver emits it (its 'decode_hop'), and the final call
at the end of the cycle releases the rest.  Calls are lock-step over all receivers, at the slowest one's hop.  What stays
different in either mode: "ran out of decoding time" cannot happen.
"""
import queue
import threading

import numpy as np

from .engine import Engine
from .receiver import format_records, record_to_message
from .time_utils import TimeUtils

CYCLE_SAMPLES = 180000


def _pinned(shape):
    import torch                      # device/pinned memory plumbing only
    t = torch.zeros(shape, dtype=torch.int16)
    try:
        t = t.pin_memory()
    except RuntimeError:              # no CUDA runtime (host-logic tests): pageable memory works, only slower
        pass
    return t, t.numpy()


class ReceiverBank:
    def __init__(self, n_receivers, on_message=None, bands=None, device=0, engine=None, clock=None, sync_score_min=85,
                 max_cands=200, columnar=False, decoder=None, live_ring=True, progressive=False, progress_hops=1):
        self.n = int(n_receivers)
        self.on_message = on_message
        self.bands = list(bands) if bands is not None else [None] * self.n
        self.columnar = columnar
        self.live_ring = live_ring    # True: every receiver keeps the reference's two-cycle waterfall ring on the device
                                      # (ft8_decode_cycles_live); False: each cycle decoded in isolation (SURVEY H5)
        if progressive and not live_ring:
            raise ValueError("progressive=True needs live_ring=True")
        if int(progress_hops) < 1:
            raise ValueError("progress_hops must be >= 1")
        self.progressive = progressive    # release messages during the cycle at the reference's hops (see module docstring)
        self.progress_hops = int(progress_hops)
        self._tu = TimeUtils(clock)
        self._decoder = decoder       # test seam: callable(audio[R,180000]) -> record array; progressive:
                                      # callable(audio[R,180000], hop) -> (record array, emission hops)
        self.engine = engine
        if decoder is None and engine is None:
            self.engine = Engine(device=device, max_cycles=self.n, max_cands=max_cands, sync_score_min=sync_score_min)
        self._hold = [_pinned((self.n, CYCLE_SAMPLES)) for _ in range(2)]
        self._buf = [h[1] for h in self._hold]
        self._open = 0                                    # oldest cycle not yet handed to the decoder (lives in half open & 1)
        self._cyc = np.zeros(self.n, np.int64)            # cycle each receiver is writing (open or open + 1)
        self._pos = np.zeros(self.n, np.int64)            # samples of that cycle received so far
        self._q = queue.Queue()
        self._results = queue.Queue()
        self._busy = {}                                   # half -> cycle handed to the decoder and not yet released
        # progressive mode: search hop, last progress hop requested for the open cycle, the latest requested hop and the
        # last decoded hop per cycle (queued calls of one cycle collapse into the latest), the cycle's label
        self._search_hop = self.engine.search_hop if self.engine is not None else 260
        self._req = 0
        self._latest, self._done, self._label = {}, {}, {}
        self._seen = {}                                   # cycle -> (receiver, text) released by its earlier calls
        self._cv = threading.Condition()
        self._state = threading.RLock()                   # guards _cyc/_pos/_open and the close-of-cycle decision
        self._eng_lock = threading.Lock()                 # one handle = one stream: calls are serialised
        self._worker = threading.Thread(target=self._run, daemon=True)
        self._worker.start()

    # ------------------------------------------------------------------------------------------------ feeding
    def set_band(self, r, band):
        self.bands[r] = band

    def _half_for(self, c):
        """Buffer half of cycle c, once the decoder has released it (it held cycle c - 2)."""
        with self._cv:
            while self._busy.get(c & 1, c) != c:
                self._cv.wait(0.05)
        return self._buf[c & 1]

    def feed(self, r, samples):
        """Append int16 samples of receiver r (any block size; the reference's callback delivers 480).  Samples past the
        end of a cycle spill into the next one; a receiver may run at most one cycle ahead of the slowest receiver.
        Returns the number of cycles this call closed."""
        x = np.asarray(samples)
        if x.dtype != np.int16 or x.ndim != 1:
            raise TypeError("feed() takes a 1-D int16 block, as the reference's audio callback does")
        with self._state:
            return self._feed_locked(r, x)

    def _feed_locked(self, r, x):
        closed = 0
        while len(x):
            c, p = int(self._cyc[r]), int(self._pos[r])
            if c > self._open + 1:
                raise BufferError("receiver %d is more than one cycle ahead of the slowest receiver" % r)
            k = min(len(x), CYCLE_SAMPLES - p)
            self._half_for(c)[r, p:p + k] = x[:k]
            x = x[k:]
            if p + k == CYCLE_SAMPLES:
                self._cyc[r], self._pos[r] = c + 1, 0
                if np.all(self._cyc > self._open):
                    self._close_cycle()
                    closed += 1
            else:
                self._pos[r] = p + k
                self._progress()
        return closed

    def feed_all(self, block):
        """block [R, k] int16: the same number of new samples for every receiver (one call per hop for a sound-card
        style source, or whole cycles for file replay)."""
        b = np.asarray(block)
        if b.dtype != np.int16 or b.ndim != 2 or b.shape[0] != self.n:
            raise TypeError("feed_all() takes an int16 [n_receivers, k] block")
        with self._state:
            return self._feed_all_locked(b)

    def _feed_all_locked(self, b):
        closed = 0
        while b.shape[1]:
            c, p = int(self._cyc[0]), int(self._pos[0])
            if not (np.all(self._pos == p) and np.all(self._cyc == c)):
                raise BufferError("feed_all() needs all receivers at the same position")
            k = min(b.shape[1], CYCLE_SAMPLES - p)
            self._half_for(c)[:, p:p + k] = b[:, :k]
            b = b[:, k:]
            if p + k == CYCLE_SAMPLES:
                self._cyc += 1
                self._pos[:] = 0
                self._close_cycle()
                closed += 1
            else:
                self._pos += k
                self._progress()
        return closed

    def _label_of(self, no, in_cycle):
        """(cyclestart string, odd_even label) of cycle `no`, read from the clock during the cycle or just after it"""
        if no not in self._label:
            t = self._tu.time() - (0.0 if in_cycle else 1.0)
            self._label[no] = (self._tu.cyclestart_string(t), self._tu.odd_even() ^ (0 if in_cycle else 1))
        return self._label[no]

    def _request(self, no, hop, in_cycle):
        cs, odd_even = self._label_of(no, in_cycle)
        with self._cv:
            self._busy[no & 1] = no
            self._latest[no] = hop
        self._q.put((no, no & 1, cs, odd_even, list(self.bands)))

    def _progress(self):
        """progressive mode: a progress call when the slowest receiver's hop in the open cycle crosses a multiple of
        progress_hops at or after the first hop that can release a message (search hop + 1)"""
        if not self.progressive:
            return
        o = self._open
        pos = np.where(self._cyc > o, 180000, self._pos)
        hop = int(pos.min()) // 480
        hop -= hop % self.progress_hops
        if self._search_hop + 1 <= hop < 375 and hop > self._req:
            self._req = hop
            self._request(o, hop, True)

    def _close_cycle(self, cyclestart_string=None):
        if self.progressive:
            self._request(self._open, 375, self._req > 0)
            self._req = 0
            self._open += 1
            return
        cs = cyclestart_string if cyclestart_string is not None else self._tu.cyclestart_string(self._tu.time() - 1.0)
        half = self._open & 1
        with self._cv:
            self._busy[half] = self._open
        self._q.put((self._open, half, cs, self._tu.odd_even() ^ 1, list(self.bands)))
        self._open += 1

    # ------------------------------------------------------------------------------------------------ decoding thread
    def _run(self):
        while True:
            item = self._q.get()
            if item is None:
                return
            no, half, cs, odd_even, bands = item
            if self.progressive:
                self._run_progress(no, half, cs, odd_even, bands)
                continue
            try:
                audio = self._buf[half]
                if self._decoder is not None:
                    rec = self._decoder(audio)
                else:
                    with self._eng_lock:
                        if self.live_ring:
                            # ring half = cycle number parity (strictly alternating); `odd_even` from the clock is only the label
                            rec, _ = self.engine.decode_cycles_live(audio, no & 1)
                        else:
                            rec, _ = self.engine.decode_cycles(audio, odd_even)
                self._release(half)                       # audio consumed: the feeder may reuse this half
                mb = format_records(rec, [cs] * self.n)
                out = mb if self.columnar else self._messages(rec, mb, cs, odd_even, bands)
                self._results.put((no, out))
            except Exception as e:                        # surface decoder failures to the feeding thread
                self._results.put((no, e))
            finally:
                self._release(half)

    def _release(self, half):
        with self._cv:
            self._busy.pop(half, None)
            self._cv.notify_all()

    def _messages(self, rec, mb, cs, odd_even, bands, emit_hop=None, seen=None):
        """message dicts of the kept rows of a formatted batch (and on_message for each); in progressive mode also
        'decode_hop', and rows whose (receiver, text) an earlier call of the cycle released are dropped"""
        out = []
        kept = np.flatnonzero(mb.keep)
        for i, txt in zip(kept.tolist(), mb.msg_tuple[kept].tolist()):
            r = rec[i]
            if seen is not None:
                key = (int(r["cycle"]), " ".join(txt))
                if key in seen:
                    continue
                seen.add(key)
            m = record_to_message(r, cs, bands[int(r["cycle"])], odd_even, self._tu.time(), msg=txt)
            m["receiver"] = int(r["cycle"])
            if emit_hop is not None:
                m["decode_hop"] = int(emit_hop[i])
            out.append(m)
            if self.on_message:
                self.on_message(m)
        return out

    def _run_progress(self, no, half, cs, odd_even, bands):
        with self._cv:
            hop = self._latest.get(no)
        if hop is None or hop <= self._done.get(no, 0):
            return                                    # collapsed into a later call of the same cycle
        try:
            audio = self._buf[half]
            if self._decoder is not None:
                rec, eh = self._decoder(audio, hop)
            else:
                with self._eng_lock:
                    rec, _, eh = self.engine.decode_cycles_live_progress(audio, no & 1, hop)
            self._done[no] = hop
            seen = self._seen.setdefault(no, set())
            mb = format_records(rec, [cs] * self.n)
            self._results.put((no, hop, self._messages(rec, mb, cs, odd_even, bands, eh, seen)))
        except Exception as e:                        # surface decoder failures to the feeding thread
            self._done[no] = hop
            self._results.put((no, hop, e))
        finally:
            if hop == 375:
                self._release(half)
                with self._cv:
                    self._latest.pop(no, None)
                self._done.pop(no, None)
                self._label.pop(no, None)
                self._seen.pop(no, None)

    def results(self, block=True, timeout=None):
        """(cycle number, list of message dicts | MessageBatch) of the next decoded cycle; in progressive mode (cycle number,
        hop, list of message dicts) of the next progress call.  Raises what the decoder raised."""
        item = self._results.get(block, timeout)
        if isinstance(item[-1], Exception):
            raise item[-1]
        return item

    # ------------------------------------------------------------------------------------------------ GUI support
    def waterfall(self, r):
        """376 x 976 dB grid of receiver r's open cycle so far (rows past the received audio see zeros, i.e. -240 dB)."""
        if self.engine is None:
            raise RuntimeError("waterfall() needs the CUDA engine")
        a = np.zeros((1, CYCLE_SAMPLES), np.int16)
        p = int(self._pos[r])
        a[0, :p] = self._buf[int(self._cyc[r]) & 1][r, :p]
        with self._eng_lock:
            return self.engine.spectrogram(a)[0]

    def close(self):
        self._q.put(None)
        self._worker.join(5)
        if self.engine is not None and self._decoder is None:
            self.engine.close()
