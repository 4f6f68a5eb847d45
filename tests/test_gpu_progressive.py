"""Progressive live decoding (ft8_decode_cycles_live_progress) against the reference scheduler made deterministic.

A running reference Receiver runs its scheduler loop (receiver.py:376-412) while the audio arrives: it searches once the hop
counter passes search_start_hop and decodes each candidate one pass per loop as soon as its payload rows are on the grid.
With the loop body run once after every hop and the clock one microsecond after it, the messages and the hop each one comes
out at are a function of the audio: tests/golden/progressive.npz holds them for the unmodified reference, and
Receiver.tick reproduces them one stream at a time.  The progressive entry must give exactly the same for many streams at
once, whatever hops it is called at.
"""
import numpy as np
import pytest

from conftest import cycle_audio, load_golden
from pyft8_b200 import _lib as L
from pyft8_b200 import messages, synth
from pyft8_b200.engine import Engine
from pyft8_b200.receiver import Receiver, record_to_message

pytestmark = pytest.mark.gpu

T0 = 30.0 * 1000000                     # a multiple of 30 s: cycle 0 is even
S_DEFAULT = 260


def stream_audio(seed, n_cycles, per=4, late=3, early=4):
    """Continuous int16 audio of n_cycles cycles: per cycle `per` stations starting 0.0-1.5 s after its boundary (the
    search finds a station starting s seconds in at h0 ~ 25 s + 2: here about 2..40, so d = h0 + 285 in about 287..325),
    `late` ones starting 2.0-2.9 s after it (h0 about 52..75, d about 337..360: due in the cycle's last hops), and, after
    the first cycle, `early` ones starting 1.30-1.48 s before it (they straddle the boundary; h0 about -35..-30, so d = 261:
    due right after the search)."""
    rng = np.random.default_rng(seed)
    x = rng.normal(0.0, 1000.0, 180000 * n_cycles)
    sig = []
    for k in range(n_cycles):
        sig += [(15.0 * k + float(rng.uniform(0.0, 1.5)), (-16, 0)) for _ in range(per)]
        sig += [(15.0 * k + float(rng.uniform(2.0, 2.9)), (-14, 0)) for _ in range(late)]
        if k:
            sig += [(15.0 * k - float(rng.uniform(1.30, 1.48)), (-19, -6)) for _ in range(early)]
    for t0, (lo, hi) in sig:
        b77 = synth.pack77(*synth.random_message(rng))
        snr = float(rng.uniform(lo, hi))
        f = float(rng.uniform(250, 2900))
        amp = 1000.0 * np.sqrt(2.0 * (2500.0 / 6000.0) * 10.0 ** (snr / 10.0))
        wf = np.imag(synth.shift_carrier(synth.gfsk_baseband(synth.symbols_from_bits77(b77)), f)) * amp
        s0 = int(t0 * 12000)
        a, b = max(s0, 0), min(s0 + len(wf), len(x))
        x[a:b] += wf[a - s0:b - s0]
    return np.clip(np.round(x), -32768, 32767).astype(np.int16).reshape(n_cycles, 180000)


def one_hop_schedule(S=S_DEFAULT):
    """the benchmark's schedule: one rows-only call for hops 1..S-1, then one call per hop"""
    return [S - 1] + list(range(S, 376))


def run_cycle(eng, audio, odd_even, hops, dev=None):
    """One cycle of B streams through progress calls at `hops` (ending with 375).  Returns (per-stream lists of
    (record, e) in release order, the concatenated record bytes, emit hops, and the summed work counters)."""
    B = audio.shape[0]
    per = [[] for _ in range(B)]
    recs, hopsout, tot = [], [], {}
    for hop in hops:
        if dev is None:
            rec, n, eh = eng.decode_cycles_live_progress(audio, odd_even, hop)
        else:
            rec, n, eh = eng.decode_cycles_live_progress_dev(dev.data_ptr(), L.AUDIO_I16 if audio.dtype == np.int16 else L.AUDIO_F32,
                                                             B, odd_even, hop)
        rec, eh = rec.copy(), eh.copy()
        assert np.all(eh <= (hop if hop < 375 else 377))
        i = 0
        for b in range(B):
            for _ in range(int(n[b])):
                assert rec[i]["cycle"] == b
                per[b].append((rec[i], int(eh[i])))
                i += 1
        recs.append(rec)
        hopsout.append(eh)
        for k, v in eng.stats().items():
            tot[k] = tot.get(k, 0) + v
    return per, np.concatenate(recs), np.concatenate(hopsout), tot


def messages_of(per_stream):
    """[(text, notes, snr, tsec, fHz, e)] of one stream-cycle's released records, text de-duplicated like check_and_package"""
    out = []
    seen = set()
    recs = [r for r, _ in per_stream]
    if not recs:
        return out
    texts = messages.unpack_words(np.stack([r["bits91"] for r in recs]))
    for (r, e), txt in zip(per_stream, texts):
        m = record_to_message(r, msg=txt)
        if m is None:
            continue
        if " ".join(m["msg_tuple"]) in seen:
            continue
        seen.add(" ".join(m["msg_tuple"]))
        out.append((" ".join(m["msg_tuple"]), m["decode_notes"], int(m["their_snr"]), m["tsec"], m["fHz"], e))
    return out


def receiver_messages(audio_cycles, rx_kw=None, engine=None):
    """One stream's consecutive cycles through Receiver.tick once per hop (clock t0 + 15 c + 0.04 T + 1e-6), two hops of
    silence after the last.  Returns per cycle [(text, notes, snr, tsec, fHz, e)], e = emission hop counted from that
    cycle's start (376, 377: the next cycle's first hops)."""
    now = [T0]
    got = []
    where = [0, 0]
    rx = Receiver("", lambda m: got.append((m, where[0], where[1])), clock=lambda: now[0], engine=engine, **(rx_kw or {}))
    ai = rx.audio_in
    st = rx.new_cycle_state()
    C = audio_cycles.shape[0]
    for c in range(C + 1):
        for T in range(1, 376 if c < C else 3):
            now[0] = T0 + 15.0 * c + T * 0.04 + 1e-6
            where[:] = [c, T]
            blk = audio_cycles[c, 480 * (T - 1):480 * T] if c < C else np.zeros(480, np.int16)
            ai._callback(blk.tobytes(), 480, None, None)
            rx.tick(st)
    out = [[] for _ in range(C)]
    starts = [rx._tu.cyclestart_string(T0 + 15.0 * c + 1.0) for c in range(C)]
    for m, c, T in got:
        k = starts.index(m["cyclestart_string"])
        e = T if k == c else 375 + T
        out[k].append((" ".join(m["msg_tuple"]), m["decode_notes"], int(m["their_snr"]), m["tsec"], m["fHz"], e))
    return out


def engine_messages(eng, seq, schedule=None):
    """seq [S, C, 180000]: C consecutive cycles of S streams through progress calls.  Returns per stream per cycle the
    messages as receiver_messages gives them (text decoded per stream in release order, hashes per stream)."""
    S_, C = seq.shape[:2]
    raw = [[None] * C for _ in range(S_)]
    for c in range(C):
        per, _, _, _ = run_cycle(eng, np.ascontiguousarray(seq[:, c]), c % 2, schedule or one_hop_schedule())
        for s in range(S_):
            raw[s][c] = per[s]
    out = []
    for s in range(S_):
        messages.call_hashes.clear()
        flat = [(r, e, c) for c in range(C) for r, e in raw[s][c]]
        res = [[] for _ in range(C)]
        if flat:
            texts = messages.unpack_words(np.stack([r["bits91"] for r, _, _ in flat]))
            seen = set()
            for (r, e, c), txt in zip(flat, texts):
                m = record_to_message(r, msg=txt)
                if m is None or (c, " ".join(m["msg_tuple"])) in seen:
                    continue
                seen.add((c, " ".join(m["msg_tuple"])))
                res[c].append((" ".join(m["msg_tuple"]), m["decode_notes"], int(m["their_snr"]), m["tsec"], m["fHz"], e))
        out.append(res)
    return out


@pytest.fixture(scope="module")
def seq3():
    return np.stack([stream_audio(7000 + s, 3) for s in range(6)])


def test_golden_cycles_among_other_streams():
    """test_08 and syn20 as streams 1 and 3 of a 5-stream batch (noise, other cycles around them), one-hop calls: per
    stream the messages, notes, SNR and emission hops of the unmodified reference's scheduler (progressive.npz)."""
    g = load_golden("progressive.npz")
    rng = np.random.default_rng(5)
    noise = np.clip(np.round(rng.normal(0, 1000, 180000)), -32768, 32767).astype(np.int16)
    batch = np.stack([noise, cycle_audio("test_08"), cycle_audio("syn50"), cycle_audio("syn20"), stream_audio(11, 1)[0]])
    eng = Engine(max_cycles=5)
    per, _, eh, _ = run_cycle(eng, batch, 0, one_hop_schedule())
    for b, name in ((1, "test_08"), (3, "syn20")):
        messages.call_hashes.clear()
        got = messages_of(per[b])
        assert [m[0] for m in got] == g[f"{name}_text"].tolist()
        assert [m[1] for m in got] == g[f"{name}_notes"].tolist()
        assert [m[2] for m in got] == g[f"{name}_snr"].tolist()
        assert [m[5] for m in got] == g[f"{name}_hop"].tolist()
    assert min(eh) > 260 and min(eh) < 375
    eng.close()


def test_many_streams_equal_single_stream_receivers(seq3):
    """6 streams x 3 consecutive cycles (boundary stations due right after the search, late stations emitted in the next
    cycle's hops, a third cycle whose pass-0 snapshots read ring rows two cycles old): every stream-cycle equals its own
    Receiver driven hop by hop -- text, notes, SNR, tsec, fHz, emission hop and order, exactly."""
    eng = Engine(max_cycles=seq3.shape[0])
    got = engine_messages(eng, seq3)
    eng.close()
    n_late = n_early = 0
    for s in range(seq3.shape[0]):
        messages.call_hashes.clear()
        want = receiver_messages(seq3[s])
        assert got[s] == want, f"stream {s}"
        for c in range(3):
            n_late += sum(m[5] > 331 for m in want[c])
            n_early += sum(m[5] < 285 for m in want[c])
    # both ends of the schedule are exercised: a station that starts inside the cycle has h0 >= 0, so d >= 285, and the
    # stations starting 0-1.5 s in have h0 <= ~40, so e <= ~331; e < 285 comes from a boundary station, e > 331 from a late one
    assert n_late > 0 and n_early > 0
    assert sum(len(x) for w in got for x in w) > 40


def test_releases_in_the_next_cycles_first_hops_equal_receiver():
    """Stations starting 3.32-3.38 s into the cycle are found at h0 = 85 or 86, the end of the search range, so d = 370 or
    371: a decode in
    pass 5 or 6 (OSD) can come out at hop 376 or 377, in the next cycle's first hops, from the call that completes the cycle.
    From a seeded pool of 512 such streams (10 stations each near the decode threshold, made by the library's generator),
    those with a release past hop 375 go through the one-hop schedule and each equals its own Receiver driven hop by hop
    (two more hops of silence after the cycle), emission hops included."""
    R, n_sig = 512, 10
    rng = np.random.default_rng(4242)
    table = np.array([synth.symbols_from_bits77(synth.pack77(*synth.random_message(rng))) for _ in range(R * n_sig)], np.uint8)
    snr = rng.uniform(-21.0, -15.0, (R, n_sig))
    amp = (1000.0 * np.sqrt(2.0 * (2500.0 / 6000.0) * 10.0 ** (snr / 10.0))).astype(np.float32)
    f = rng.uniform(250.0, 2900.0, (R, n_sig)).astype(np.float32)
    dt = rng.uniform(2.82, 2.88, (R, n_sig)).astype(np.float32)       # start 0.5 + dt s: 3.32-3.38 s
    eng = Engine(max_cycles=R)
    pool = eng.synth_cycles(table.reshape(R, n_sig, 79), f, dt, amp, 1000.0, seed=4242)
    per, _, _, _ = run_cycle(eng, pool, 0, [375])
    eng.close()
    late = [b for b in range(R) if any(e > 375 and r["emitted"] for r, e in per[b])][:3]
    assert late, "no stream of the pool has a release past hop 375"
    eng = Engine(max_cycles=len(late))
    got = engine_messages(eng, pool[late][:, None])
    eng.close()
    n_next = 0
    for i, b in enumerate(late):
        messages.call_hashes.clear()
        want = receiver_messages(pool[b][None])
        assert got[i] == want, f"stream {b}"
        n_next += sum(m[5] > 375 for m in want[0])
    assert n_next > 0


@pytest.mark.parametrize("dtype", ["int16", "float32", "device"])
def test_call_granularity_changes_nothing(seq3, dtype):
    """Calls every 1, 7 and 40 hops, at irregular hops, and one single hop-375 call: byte-identical records, emission hops
    and summed work counters, for two consecutive cycles; int16 / float32 / device-resident audio alike."""
    import torch
    schedules = [list(range(1, 376)), list(range(7, 375, 7)) + [375], list(range(40, 375, 40)) + [375],
                 [3, 100, 259, 260, 261, 262, 300, 301, 374, 375], [375], one_hop_schedule()]
    ref = None
    eng = Engine(max_cycles=seq3.shape[0])
    for sch in schedules:
        eng.live_reset()
        outs = []
        for c in range(2):
            a = np.ascontiguousarray(seq3[:, c])
            if dtype == "float32":
                a = a.astype(np.float32)
            dev = torch.from_numpy(a).cuda() if dtype == "device" else None
            per, _, _, tot = run_cycle(eng, a, c % 2, sch, dev)
            rec = np.array([r for p in per for r, _ in p], L.RECORD_DTYPE)          # per stream, in release order
            eh = np.array([e for p in per for _, e in p], np.uint16)
            outs.append((rec.tobytes(), eh.tobytes(), {k: v for k, v in tot.items() if k != "kernel_launches"}))
        if ref is None:
            ref = outs
            assert len(rec) > 0
        else:
            assert outs == ref, sch
    if dtype != "int16":
        eng2 = Engine(max_cycles=seq3.shape[0])
        base = []
        for c in range(2):
            _, rec, eh, _ = run_cycle(eng2, np.ascontiguousarray(seq3[:, c]), c % 2, [375])    # one call: stream-major
            base.append((rec.tobytes(), eh.tobytes()))
        assert [o[:2] for o in ref] == base
        eng2.close()
    eng.close()


def _live_state_after(eng, seq, kinds):
    """run cycles 0..len(kinds)-1 with 'p' (progressive, one-hop) or 'l' (live); returns the last cycle's records"""
    eng.live_reset()
    for c, k in enumerate(kinds):
        a = np.ascontiguousarray(seq[:, c])
        if k == "l":
            rec, n = eng.decode_cycles_live(a, c % 2)
            last = rec.copy()
        else:
            _, last, _, _ = run_cycle(eng, a, c % 2, one_hop_schedule())
    return last


def test_state_at_cycle_boundaries(seq3):
    """Progressive and live calls follow each other at cycle boundaries: the state a progressive cycle leaves is the one a
    live call leaves (so the next cycle decodes the same, either way), and the next progressive cycle reads the live
    cycle's audio and rows exactly as if it had been progressive."""
    eng = Engine(max_cycles=seq3.shape[0])
    assert _live_state_after(eng, seq3, "pl").tobytes() == _live_state_after(eng, seq3, "ll").tobytes()
    assert _live_state_after(eng, seq3, "lp").tobytes() == _live_state_after(eng, seq3, "pp").tobytes()
    assert _live_state_after(eng, seq3, "plp").tobytes() == _live_state_after(eng, seq3, "ppp").tobytes()
    eng.close()


def test_other_calls_between_progress_calls_change_nothing(seq3):
    """Stage calls and an isolated decode between two progress calls of an open cycle do not disturb it."""
    B = seq3.shape[0]
    eng = Engine(max_cycles=B)
    a0, a1 = np.ascontiguousarray(seq3[:, 0]), np.ascontiguousarray(seq3[:, 1])
    ref = [run_cycle(eng, a, c, one_hop_schedule())[1].tobytes() for c, a in enumerate((a0, a1))]
    eng.live_reset()
    out = []
    for c, a in enumerate((a0, a1)):
        recs = []
        for hop in one_hop_schedule():
            rec, _, _ = eng.decode_cycles_live_progress(a, c, hop)
            recs.append(rec.copy())
            if hop in (259, 262, 300, 371):
                eng.spectrogram(seq3[:2, 2])
                eng.cycle_spectrum(seq3[:3, 2])
                eng.decode_cycles(seq3[:, 2])
        out.append(np.concatenate(recs).tobytes())
    assert out == ref
    eng.close()


def test_errors_and_reset(seq3):
    B = seq3.shape[0]
    eng = Engine(max_cycles=B)
    a = np.ascontiguousarray(seq3[:, 0])
    lib, h = eng._lib, eng._h
    rec = np.zeros(B * 200, L.RECORD_DTYPE)
    eh = np.zeros(B * 200, np.uint16)
    n = np.zeros(B, np.int32)

    def call(x, B_, oe, hop):
        return lib.ft8_decode_cycles_live_progress(h, x.ctypes.data, L.AUDIO_I16, B_, oe, hop, rec.ctypes.data, eh.ctypes.data,
                                                   len(rec), n.ctypes.data, L.MEM_HOST)
    assert call(a, B, 0, 0) == L.E_BADARG and call(a, B, 0, 376) == L.E_BADARG and call(a, B, 2, 10) == L.E_BADARG
    assert call(a, B, 0, 100) == L.OK
    assert call(a, B, 0, 100) == L.E_BADARG            # not increasing
    assert call(a, B, 0, 99) == L.E_BADARG
    assert call(a, B - 1, 0, 150) == L.E_BADARG        # B changed
    assert call(a, B, 1, 150) == L.E_BADARG            # odd_even changed
    with pytest.raises(RuntimeError):
        eng.decode_cycles_live(a, 0)                   # a progressive cycle is open
    with pytest.raises(RuntimeError):
        eng.decode_cycles_live_seq(seq3[:, :2].transpose(1, 0, 2), 0)
    assert call(a, B, 0, 375) == L.OK
    assert call(a, B, 0, 10) == L.E_BADARG             # parity does not alternate
    # a reset in the middle of a cycle abandons it: the stream is fresh again
    assert call(np.ascontiguousarray(seq3[:, 1]), B, 1, 300) == L.OK
    eng.live_reset()
    fresh = Engine(max_cycles=B)
    x = np.ascontiguousarray(seq3[:, 2])
    assert run_cycle(eng, x, 0, one_hop_schedule())[1].tobytes() == run_cycle(fresh, x, 0, one_hop_schedule())[1].tobytes()
    fresh.close()
    eng.close()


@pytest.mark.parametrize("knob", ["time_range", "freq_range", "max_cands", "fine_mode"])
def test_knobs_against_receiver(seq3, knob):
    """Search ranges (a narrower time range moves the search hop), max_cands and fine_mode 1, each against Receiver.tick
    built with the same settings."""
    rx_kw, eng_kw = {}, {}
    if knob == "time_range":
        rx_kw = dict(search_time_range=[-1.5, 2.0])
        eng_kw = dict(search_h0_range=[int((t + 0.5) * 25) for t in rx_kw["search_time_range"]])
    elif knob == "freq_range":
        rx_kw = dict(search_freq_range=[400, 2200])
        eng_kw = dict(search_f0_range=[int(f / 3.125) for f in rx_kw["search_freq_range"]])
    elif knob == "max_cands":
        rx_kw = dict(max_cands=25)
        eng_kw = dict(max_cands=25)
    else:
        eng_kw = dict(fine_mode=1)
    seq = seq3[:3, :2]
    eng = Engine(max_cycles=seq.shape[0], **eng_kw)
    S = eng.search_hop
    got = engine_messages(eng, seq, one_hop_schedule(S))
    eng.close()
    for s in range(seq.shape[0]):
        messages.call_hashes.clear()
        rx_engine = None
        if knob == "fine_mode":
            rx_engine = Engine(max_cycles=1, max_cands=928, fine_mode=1)
        want = receiver_messages(seq[s], rx_kw, rx_engine)
        assert got[s] == want, f"stream {s}"
        if rx_engine is not None:
            rx_engine.close()


def test_bank_progressive_equals_engine(seq3):
    """ReceiverBank(progressive=True) fed 480 samples per hop over two cycles: its messages and decode hops are the
    engine-level ones, and the first messages arrive while the cycle is still running."""
    from pyft8_b200.bank import ReceiverBank
    seq = seq3[:, :2]
    B = seq.shape[0]
    eng = Engine(max_cycles=B)
    want = engine_messages(eng, seq)
    eng.close()
    messages.call_hashes.clear()
    now = [T0]
    bank = ReceiverBank(B, clock=lambda: now[0], progressive=True)
    calls = []
    for c in range(2):
        for T in range(1, 376):
            now[0] = T0 + 15.0 * c + T * 0.04 + 1e-6
            bank.feed_all(np.ascontiguousarray(seq[:, c, 480 * (T - 1):480 * T]))
            if c == 0 and 261 <= T < 375:            # in step with the audio (a faster feed collapses queued calls)
                calls.append(bank.results(timeout=120))
                assert calls[-1][:2] == (0, T)
    while True:
        no, hop, ms = bank.results(timeout=120)
        calls.append((no, hop, ms))
        if (no, hop) == (1, 375):
            break
    bank.close()
    got = [[[] for _ in range(2)] for _ in range(B)]
    for no, hop, ms in calls:
        for m in ms:
            assert m["decode_hop"] <= (hop if hop < 375 else 377)
            got[m["receiver"]][no].append((" ".join(m["msg_tuple"]), m["decode_notes"], int(m["their_snr"]), m["tsec"], m["fHz"],
                                           m["decode_hop"]))
    assert got == [w[:2] for w in want]
    first = min(hop for no, hop, ms in calls if no == 0 and ms)
    assert first < 375
