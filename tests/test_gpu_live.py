"""Live mode (ft8_decode_cycles_live) over many streams and consecutive cycles, against a CPU model of the reference's ring.

A running reference Receiver keeps a 750-row waterfall ring (np.ones at start) and a 180000-sample audio buffer; each hop
writes the row of the window over the last 3840 samples.  For a cycle of parity p that is, per stream:

    ring[(375 p + h) mod 750] = oracle spectrogram row of the window ending at sample 480 h of concat(tail, audio), h = 1..375
    decode = ft8_oracle.decode_cycle(audio, odd_even=p, grid=ring)
    tail   = audio[-3840:]                          (zeros before a stream's first cycle)

The previous cycle is visible only through two things: payload rows (h0 + 4 + 4 s + 375 p) mod 750 that wrap into the
other half (h0 <= -32 in an even cycle, any h0 in an odd one) and the first hops' windows, which read the tail.  So the
streams here carry stations that start 1.30-1.48 s before every cycle boundary at SNRs near the decode threshold, and the
unmarked premise tests show that a ring-blind model (other half 1.0, tail zeros) decodes them differently.

The GPU tests check every stream-cycle against the model (payload sets exact; dt, df, SNR within tolerance; order and notes
differences counted and bounded), then that the batch layout, the chunked host-copy path, the audio dtype and the handle's
history (reset, growing B, isolated and stage calls in between) change nothing that a fresh receiver would not see.
"""
import ctypes as C
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, load_golden
from pyft8_b200 import _lib as L
from pyft8_b200 import synth

T_A, S_A, SEED_A = 5, 12, 100           # sequence A: 12 streams x 5 cycles, parities 0 1 0 1 0
T_B, S_B, SEED_B = 3, 6, 200            # sequence B: 6 streams x 3 cycles, parities 1 0 1
HALF = 375
EARLY_H0 = -32                          # h0 <= -32: a payload row of an even cycle wraps into the odd half


def synth_stream(seed, n_cycles, per=5, early=8):
    """Continuous int16 audio of n_cycles 15 s cycles: per cycle `per` stations starting 0.0-1.5 s after its boundary
    (SNR -16..0 dB) and, after the first, `early` stations starting 1.30-1.48 s BEFORE it (SNR -19..-8 dB), so that they
    straddle the boundary."""
    rng = np.random.default_rng(seed)
    x = rng.normal(0.0, 1000.0, 180000 * n_cycles)
    sig = []
    for k in range(n_cycles):
        sig += [(15.0 * k + float(rng.uniform(0.0, 1.5)), (-16, 0)) for _ in range(per)]
        if k:
            sig += [(15.0 * k - float(rng.uniform(1.30, 1.48)), (-19, -8)) for _ in range(early)]
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


def _synth_job(args):
    return synth_stream(*args)


def make_sequence(pool, seed, n_streams, n_cycles):
    """int16[n_streams, n_cycles, 180000]; stream s from seed + s"""
    return np.stack(pool.map(_synth_job, [(seed + s, n_cycles) for s in range(n_streams)], chunksize=1))


# ------------------------------------------------------------------------------------------------ CPU ring model
def _rows(tail, audio):
    """oracle.spectrogram rows 1..375 with the window reaching back into `tail` (3840 samples before the cycle)."""
    import ft8_oracle as o
    x = np.concatenate([tail.astype(np.float32), audio.astype(np.float32)])
    rows = np.empty((HALF, 976), np.float32)
    buf = np.empty(3840, np.float32)
    for h in range(1, HALF + 1):
        np.multiply(x[480 * h:480 * h + 3840], o._HANN, out=buf)
        rows[h - 1] = 20 * np.log10(np.abs(np.fft.rfft(buf)[:976]) + 1e-12)
    return rows


def _half(p):
    return (HALF * p + np.arange(1, HALF + 1)) % 750


def ring_model_cycle(pre, prev, audio, p, blind=False, knobs=None):
    """One stream-cycle of the ring model: `prev` is the stream's previous cycle (None for its first), `pre` the cycle before
    that.  The two halves of the ring together hold 750 rows, so after two cycles the ring holds exactly the rows of the
    last two: a stream-cycle can be rebuilt from its three latest cycles, which lets a pool run them independently.
    blind: the ring-blind variant (other half 1.0, tail zeros).  knobs: ft8_oracle keyword arguments of the search
    (score_min, max_cands, f0_range, h0_range) and of decode_cycle (llr_sd_min, osd_singleflips, osd_doubleflips).
    Returns ft8_oracle.decode_cycle's (records, cands)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ft8_oracle as o
    zeros = np.zeros(3840, np.float32)
    ring = np.ones((750, 976), np.float32)
    if prev is not None and not blind:
        ring[_half(1 - p)] = _rows(zeros if pre is None else pre[-3840:], prev)
    ring[_half(p)] = _rows(zeros if prev is None or blind else prev[-3840:], audio)
    if not knobs:
        return o.decode_cycle(audio, odd_even=p, grid=ring)
    kw = dict(knobs)
    search = [kw.pop(k, d) for k, d in (("score_min", 85), ("max_cands", 200), ("f0_range", None), ("h0_range", None))]
    cands = o.search(ring, search[0], search[1], odd_even=p, f0_range=search[2], h0_range=search[3])
    return o.decode_cycle(audio, odd_even=p, grid=ring, cands=cands, **kw)


def model_records(recs, cl):
    """[(bits77, notes, tsec, fHz, snr, h0)] in emission order"""
    return [(r["bits77"], r["notes"], r["tsec"], r["fHz"], r["snr"], int(cl[r["cand"]].h0)) for r in recs]


def _model_job(job):
    """One stream-cycle of the ring model.  job = (pre, prev, audio, p, blind[, knobs]) as ring_model_cycle takes them.
    Returns [(bits77, notes, tsec, fHz, snr, h0)] in emission order."""
    return model_records(*ring_model_cycle(*job))


def _jobs(seq, p0, blind=False, knobs=None):
    out = []
    for s in range(seq.shape[0]):
        for k in range(seq.shape[1]):
            out.append((seq[s, k - 2] if k >= 2 else None, seq[s, k - 1] if k >= 1 else None, seq[s, k], (p0 + k) % 2, blind,
                        knobs))
    return out


def run_model(pool, seq, p0, blind=False, knobs=None, job=_model_job):
    """model[s][k] = job's result for stream s, cycle k (by default its records)"""
    res = pool.map(job, _jobs(seq, p0, blind, knobs), chunksize=1)
    S, T = seq.shape[:2]
    return [res[s * T:(s + 1) * T] for s in range(S)]


@pytest.fixture(scope="module")
def pool():
    with mp.get_context("spawn").Pool(os.cpu_count() or 1) as p:
        yield p


@pytest.fixture(scope="module")
def seq_a(pool):
    return make_sequence(pool, SEED_A, S_A, T_A)


@pytest.fixture(scope="module")
def seq_b(pool):
    return make_sequence(pool, SEED_B, S_B, T_B)


@pytest.fixture(scope="module")
def model_a(pool, seq_a):
    return run_model(pool, seq_a, 0)


@pytest.fixture(scope="module")
def model_b(pool, seq_b):
    return run_model(pool, seq_b, 1)


# ------------------------------------------------------------------------------------------------ premises (CPU)
def test_ring_model_reproduces_reference_live_pairs(pool, golden_cycles):
    """The model equals the unmodified reference Receiver fed hop by hop (tests/golden/live_pairs.npz), with the criteria of
    the existing two-cycle live test."""
    import ft8_oracle as o
    import make_golden_live as mgl
    g = load_golden("live_pairs.npz")
    s = mgl.synth_stream(int(g["syn_seed"]))
    pairs = {"wav": (golden_cycles["test_08"][0], golden_cycles["test_09"][0]), "syn": (s[:180000], s[180000:])}
    for name, (a, b) in pairs.items():
        got = run_model(pool, np.stack([a, b])[None], 0)[0]
        for i in range(2):
            txt = [o.unpack77(r[0]) for r in got[i]]
            assert [" ".join(t) for t in txt if t] == list(g[f"{name}_text_{i}"]), (name, i)
            assert all(txt), (name, i)
            assert [r[1] for r in got[i]] == list(g[f"{name}_notes_{i}"]), (name, i)
            np.testing.assert_allclose([r[2] for r in got[i]], g[f"{name}_tsec_{i}"], atol=0.005 + 1e-9)
            np.testing.assert_allclose([r[3] for r in got[i]], g[f"{name}_fhz_{i}"], atol=0.5 + 1e-9)
            assert np.all(np.abs(np.array([r[4] for r in got[i]]) - g[f"{name}_snr_{i}"]) <= 1), (name, i)


MIN_RING_VISIBLE = 5      # stream-cycles per class whose output the ring changes


def test_workload_makes_the_ring_matter(pool, seq_a, model_a, seq_b, model_b):
    """The ring-blind model decodes differently (payload set, notes or order) from the ring model in at least
    MIN_RING_VISIBLE stream-cycles of each class: odd cycles, even cycles at index >= 2, and even cycles right after a
    first odd one.  With three or more such stream-cycles, a kernel that ignored the ring could not stay inside the GPU
    tests' bounds (no set difference, at most one order and one notes difference)."""
    blind_a, blind_b = run_model(pool, seq_a, 0, blind=True), run_model(pool, seq_b, 1, blind=True)
    changed = {"odd": 0, "even_index_ge_2": 0, "even_after_first_odd": 0}
    for model, blind, p0 in ((model_a, blind_a, 0), (model_b, blind_b, 1)):
        for s in range(len(model)):
            for k in range(len(model[s])):
                p = (p0 + k) % 2
                if k == 0:
                    continue                          # a stream's first cycle has no history in either model
                key = "odd" if p else ("even_index_ge_2" if k >= 2 else "even_after_first_odd")
                changed[key] += [(r[0], r[1]) for r in model[s][k]] != [(r[0], r[1]) for r in blind[s][k]]
    print(f"[live] stream-cycles the ring changes: {changed}")
    assert min(changed.values()) >= MIN_RING_VISIBLE, changed


def test_workload_decodes_early_stations(seq_a, model_a):
    """At least 20 decoded stations with h0 <= -32 in even cycles after the first, and at least 20 in odd cycles."""
    n = {0: 0, 1: 0}
    for s in range(S_A):
        for k in range(1, T_A):
            n[k % 2] += sum(r[5] <= EARLY_H0 for r in model_a[s][k])
    assert n[0] >= 20 and n[1] >= 20, n


# ------------------------------------------------------------------------------------------------ GPU
def _split(rec, n):
    out, off = [], 0
    for b in range(len(n)):
        out.append(np.array(rec[off:off + n[b]], copy=True))
        off += n[b]
    return out


def live_run(eng, seq, p0, dtype=np.int16):
    """got[s][k] = records of stream s, cycle k (one live call per cycle, stream s = row s)"""
    S, T = seq.shape[:2]
    got = [[None] * T for _ in range(S)]
    for k in range(T):
        rec, n = eng.decode_cycles_live(np.ascontiguousarray(seq[:, k]).astype(dtype), (p0 + k) % 2)
        for s, r in enumerate(_split(rec, n)):
            got[s][k] = r
    return got


def _same(a, b):
    """bit-identical records, every field except `cycle` (the stream's row in its call)"""
    a, b = a.copy(), b.copy()
    a["cycle"] = 0
    b["cycle"] = 0
    return len(a) == len(b) and a.tobytes() == b.tobytes()


def compare_with_model(got, model, p0, min_model_decodes=None):
    from pyft8_b200.engine import bits91_to_int
    from pyft8_b200.receiver import record_to_message
    set_diff, order_bad, notes_bad, tol_bad, n_model = [], [], [], [], 0
    for s in range(len(model)):
        for k in range(len(model[s])):
            em = got[s][k][got[s][k]["emitted"] == 1]
            pay = [bits91_to_int(x["bits91"]) >> 14 for x in em]
            want = model[s][k]
            n_model += len(want)
            assert len(pay) == len(set(pay)), (s, k, "duplicate payload flagged emitted")
            d = set(pay) ^ {w[0] for w in want}
            if d:
                set_diff.append((s, k, sorted("%x" % v for v in d)))
            elif pay != [w[0] for w in want]:
                order_bad.append((s, k))
            ref = {w[0]: w for w in want}
            for x, g in zip(em, pay):
                if g in ref:
                    m = record_to_message(x)
                    if m["decode_notes"] != ref[g][1]:
                        notes_bad.append((s, k, "%x" % g, m["decode_notes"], ref[g][1]))
                    if abs(m["tsec"] - ref[g][2]) > 0.005 + 1e-9 or abs(m["fHz"] - ref[g][3]) > 0.5 + 1e-9 \
                            or abs(int(m["their_snr"]) - ref[g][4]) > 1:
                        tol_bad.append((s, k, "%x" % g))
    rep = dict(first_parity=p0, model_decodes=n_model, set_differences=set_diff[:8], n_set_differences=len(set_diff),
               order_differs=order_bad, notes_differ=notes_bad[:8], n_notes_differ=len(notes_bad), out_of_tolerance=tol_bad[:8])
    print(f"[live] {rep}")
    assert n_model > (10 * len(model) if min_model_decodes is None else min_model_decodes), rep
    assert not set_diff, rep
    assert not tol_bad, rep
    # near-ties between the CUDA and numpy FFTs can swap two emissions or the pass that decodes one (as in the large
    # parity sweeps): counted and bounded
    assert len(order_bad) <= 1 and len(notes_bad) <= 1, rep


@pytest.fixture(scope="module")
def gpu_a(seq_a):
    from pyft8_b200.engine import Engine
    eng = Engine(max_cycles=S_A)
    got = live_run(eng, seq_a, 0)
    eng.close()
    return got


@pytest.mark.gpu
def test_live_sequence_matches_ring_model(gpu_a, model_a):
    """12 streams x 5 cycles (parities 0 1 0 1 0) on one B = 12 handle against the ring model, stream-cycle by stream-cycle."""
    compare_with_model(gpu_a, model_a, 0)


@pytest.mark.gpu
def test_live_sequence_starting_odd_matches_ring_model(seq_b, model_b):
    """6 streams x 3 cycles starting with an odd cycle (parities 1 0 1)."""
    from pyft8_b200.engine import Engine
    eng = Engine(max_cycles=S_B)
    got = live_run(eng, seq_b, 1)
    eng.close()
    compare_with_model(got, model_b, 1)


@pytest.mark.gpu
def test_streams_are_independent(seq_a, gpu_a):
    """Each stream alone on a B = 1 handle gives bit-identical records to its row of the B = 12 run."""
    from pyft8_b200.engine import Engine
    eng = Engine(max_cycles=1)
    bad = []
    for s in range(S_A):
        eng.live_reset()
        one = live_run(eng, seq_a[s:s + 1], 0)[0]
        bad += [(s, k) for k in range(T_A) if not _same(one[k], gpu_a[s][k])]
    eng.close()
    assert not bad, bad


CHECKED_AT = (0, 149, 150, 151, 299)     # B = 300 host audio: two chunks of 150 streams


@pytest.mark.gpu
def test_chunked_host_path_and_device_path(seq_a, gpu_a):
    """B = 300 host audio takes the chunked copy path (two chunks of 150).  Streams 0..4 of sequence A sit at both ends of
    both chunks, noise elsewhere; their records equal the B = 12 run, and the whole batch equals the same batch given as
    device memory (one launch per stage)."""
    import torch
    from pyft8_b200.engine import Engine, _ptr
    B, T = 300, 3
    rng = np.random.default_rng(7)
    batch = rng.integers(-3000, 3001, (B, T, 180000), dtype=np.int16)
    for i, b in enumerate(CHECKED_AT):
        batch[b] = seq_a[i, :T]
    eng = Engine(max_cycles=B)
    host = live_run(eng, batch, 0)
    eng.close()
    bad = [(b, k) for i, b in enumerate(CHECKED_AT) for k in range(T) if not _same(host[b][k], gpu_a[i][k])]
    assert not bad, bad
    eng = Engine(max_cycles=B)
    dev_bad = []
    for k in range(T):
        a = torch.from_numpy(np.ascontiguousarray(batch[:, k])).to("cuda:0")
        rec = np.zeros(B * eng.max_cands, L.RECORD_DTYPE)
        n = np.zeros(B, np.int32)
        eng._check(eng._lib.ft8_decode_cycles_live(eng._h, C.c_void_p(a.data_ptr()), L.AUDIO_I16, B, k % 2, _ptr(rec), len(rec),
                                                   _ptr(n), L.MEM_DEVICE))
        dev = _split(rec[:int(n.sum())], n)
        dev_bad += [(b, k) for b in range(B) if dev[b].tobytes() != host[b][k].tobytes()]
    eng.close()
    assert not dev_bad, dev_bad[:16]
    assert sum(len(host[b][k]) for b in range(B) for k in range(T)) > 0


@pytest.mark.gpu
def test_float32_audio_equals_int16(seq_a, gpu_a):
    """The same sample values as float32 give bit-identical records over the whole sequence."""
    from pyft8_b200.engine import Engine
    eng = Engine(max_cycles=S_A)
    got = live_run(eng, seq_a, 0, dtype=np.float32)
    eng.close()
    bad = [(s, k) for s in range(S_A) for k in range(T_A) if not _same(got[s][k], gpu_a[s][k])]
    assert not bad, bad


@pytest.mark.gpu
def test_dtype_switch_keeps_the_tail(seq_a, gpu_a):
    """int16, float32, int16, float32, int16 cycles decode exactly like five int16 cycles: the previous cycle's tail is
    kept across a change of dtype."""
    from pyft8_b200.engine import Engine
    eng = Engine(max_cycles=S_A)
    bad = []
    for k in range(T_A):
        dt = np.float32 if k % 2 else np.int16
        rec, n = eng.decode_cycles_live(seq_a[:, k].astype(dt), k % 2)
        bad += [(s, k) for s, r in enumerate(_split(rec, n)) if not _same(r, gpu_a[s][k])]
    eng.close()
    assert not bad, bad


def _joiners(seq_a, gpu_a):
    """Two streams that decode early stations in cycle 1 (their records read rows built from the tail) and two others."""
    early = [int(np.sum(gpu_a[s][1]["h0_idx"] <= -25)) for s in range(S_A)]
    order = sorted(range(S_A), key=lambda s: -early[s])
    join, first = order[:2], order[2:4]
    assert all(early[s] > 0 for s in join), early
    return first, join


def _fresh_odd(seq_a, streams):
    """records of `streams` whose first live call is cycle 1 (odd), on a fresh handle"""
    from pyft8_b200.engine import Engine
    eng = Engine(max_cycles=len(streams))
    rec, n = eng.decode_cycles_live(seq_a[streams, 1], 1)
    eng.close()
    return _split(rec, n)


@pytest.mark.gpu
def test_reset_then_growing_batch_reads_zero_tails(seq_a, gpu_a):
    """B = 4, live_reset, B = 2, B = 4: streams 2 and 3 of the last call have no history and must decode like a fresh
    stream whose first call is odd; streams 0 and 1 continue their history."""
    from pyft8_b200.engine import Engine
    first, join = _joiners(seq_a, gpu_a)
    four = first + join
    fresh = _fresh_odd(seq_a, join)
    eng = Engine(max_cycles=4)
    eng.decode_cycles_live(seq_a[four, 0], 0)
    eng.live_reset()
    eng.decode_cycles_live(seq_a[first, 0], 0)
    got = _split(*eng.decode_cycles_live(seq_a[four, 1], 1))
    eng.close()
    want = [gpu_a[first[0]][1], gpu_a[first[1]][1], fresh[0], fresh[1]]
    bad = [i for i in range(4) if not _same(got[i], want[i])]
    assert not bad, f"streams {bad} of the last call differ (0, 1: continuing history; 2, 3: joining)"


@pytest.mark.gpu
def test_growing_batch_on_new_handle_reads_zero_tails(seq_a, gpu_a):
    """B = 2 then B = 4 on a new handle: the two streams that join read zeros before their first sample."""
    from pyft8_b200.engine import Engine
    first, join = _joiners(seq_a, gpu_a)
    fresh = _fresh_odd(seq_a, join)
    eng = Engine(max_cycles=4)
    eng.decode_cycles_live(seq_a[first, 0], 0)
    got = _split(*eng.decode_cycles_live(seq_a[first + join, 1], 1))
    eng.close()
    want = [gpu_a[first[0]][1], gpu_a[first[1]][1], fresh[0], fresh[1]]
    bad = [i for i in range(4) if not _same(got[i], want[i])]
    assert not bad, f"streams {bad} of the last call differ (0, 1: continuing history; 2, 3: joining)"


@pytest.mark.gpu
def test_isolated_and_stage_calls_leave_live_state_alone(seq_a, gpu_a):
    """Isolated decode_cycles and the stage entry points between live calls change neither the live results nor their own."""
    from pyft8_b200.engine import Engine
    other = np.ascontiguousarray(seq_a[:, ::-1].reshape(-1, 180000)[:S_A])     # other cycles of the same streams
    ref = Engine(max_cycles=S_A)
    want_iso = ref.decode_cycles(other)
    ref.close()
    eng = Engine(max_cycles=S_A)
    bad = []
    for k in range(T_A):
        rec, n = eng.decode_cycles_live(seq_a[:, k], k % 2)
        bad += [(s, k) for s, r in enumerate(_split(rec, n)) if not _same(r, gpu_a[s][k])]
        iso = eng.decode_cycles(other)
        assert iso[0].tobytes() == want_iso[0].tobytes() and np.array_equal(iso[1], want_iso[1]), k
        grid = eng.spectrogram(other[:2])
        eng.sync(grid, odd_even=k % 2)
        eng.sync(np.ones((1, L.GRID_ROWS_LIVE, L.GRID_COLS), np.float32), odd_even=1, want_payload=False)
        eng.cycle_spectrum(other[:1])
        eng.hop_spectrum(other[0])
    eng.close()
    assert not bad, bad
