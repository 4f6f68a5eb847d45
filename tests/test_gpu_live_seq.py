"""Consecutive live cycles in one call (ft8_decode_cycles_live_seq) against C sequential ft8_decode_cycles_live calls.

The entry decodes C cycles of B streams as batches of whole cycle steps and is specified as bit-identical with the live
calls it replaces, records concatenated call after call with `cycle` = c*B + b, and with the same live state afterwards.
So every comparison here is exact: all record bytes after mapping `cycle`, and the per-cycle counts.  The audio is the
continuous multi-cycle workload of test_gpu_live.py (stations straddling every cycle boundary), so a wrong boundary row,
tail or ring half changes records.
"""
import ctypes as C
import multiprocessing as mp
import os

import numpy as np
import pytest

from conftest import load_golden
from pyft8_b200 import _lib as L
from test_gpu_dropin import _live_messages
from test_gpu_live import _same, _split, make_sequence

S_A, T_A, SEED_A = 12, 5, 100         # 12 streams x 5 cycles (the sequence of test_gpu_live.py)
S_B, T_B, SEED_B = 3, 7, 300          # 3 streams x 7 cycles


@pytest.fixture(scope="module")
def pool():
    with mp.get_context("spawn").Pool(os.cpu_count() or 1) as p:
        yield p


@pytest.fixture(scope="module")
def xa(pool):
    """int16 [T_A, S_A, 180000], time-major as the entry takes it"""
    return np.ascontiguousarray(make_sequence(pool, SEED_A, S_A, T_A).transpose(1, 0, 2))


@pytest.fixture(scope="module")
def xb(pool):
    return np.ascontiguousarray(make_sequence(pool, SEED_B, S_B, T_B).transpose(1, 0, 2))


def _engine(max_cycles):
    from pyft8_b200.engine import Engine
    return Engine(max_cycles=max_cycles)


def live_calls(eng, x, p0, c0=0):
    """one decode_cycles_live call per step of x [C, B, 180000] -> (records with cycle = (c0 + c)*B + b, n[C, B])"""
    B = x.shape[1]
    recs, ns = [], []
    for c in range(len(x)):
        r, n = eng.decode_cycles_live(x[c], (p0 + c) % 2)
        r = r.copy()
        r["cycle"] += (c0 + c) * B
        recs.append(r)
        ns.append(n.copy())
    return np.concatenate(recs), np.stack(ns)


def seq_call(eng, x, p0, c0=0):
    r, n = eng.decode_cycles_live_seq(x, p0)
    r = r.copy()
    r["cycle"] += c0 * x.shape[1]
    return r, n.copy()


def seq_device(eng, x, p0):
    """the same entry with the audio in torch device memory"""
    import torch
    from pyft8_b200.engine import _ptr
    Cs, B = x.shape[:2]
    a = torch.from_numpy(np.ascontiguousarray(x)).to("cuda:0")
    dt = L.AUDIO_I16 if x.dtype == np.int16 else L.AUDIO_F32
    rec = np.zeros(Cs * B * eng.max_cands, L.RECORD_DTYPE)
    n = np.zeros(Cs * B, np.int32)
    eng._check(eng._lib.ft8_decode_cycles_live_seq(eng._h, C.c_void_p(a.data_ptr()), dt, B, Cs, p0, _ptr(rec), len(rec), _ptr(n),
                                                   L.MEM_DEVICE))
    return rec[:int(n.sum())].copy(), n.reshape(Cs, B)


def _cells(run):
    """records of each (cycle, stream), cycle-major"""
    return _split(run[0], run[1].ravel())


def assert_equal_runs(got, want, what=""):
    (rec, n), (wrec, wn) = got, want
    assert n.shape == wn.shape and np.array_equal(n, wn), (what, np.argwhere(n != wn)[:8].tolist() if n.shape == wn.shape else n.shape)
    assert len(rec) == len(wrec), what
    bad = [i for i in range(len(rec)) if rec[i].tobytes() != wrec[i].tobytes()]
    assert not bad, (what, f"{len(bad)} records differ, first at {bad[0]}: cycle {int(wrec[bad[0]]['cycle'])}")
    assert len(rec) > 0, what


# ------------------------------------------------------------------------------------------------ equivalence
_REF = {}


def _reference(xa, p0, dtype):
    """five sequential live calls of 12 streams on a fresh handle"""
    if (p0, dtype) not in _REF:
        eng = _engine(S_A)
        _REF[p0, dtype] = live_calls(eng, xa.astype(dtype), p0)
        eng.close()
    return _REF[p0, dtype]


@pytest.mark.gpu
@pytest.mark.parametrize("mem", ["host", "device"])
@pytest.mark.parametrize("dtype", [np.int16, np.float32], ids=["int16", "float32"])
@pytest.mark.parametrize("p0", [0, 1])
def test_seq_equals_sequential_live_calls(xa, p0, dtype, mem):
    """12 streams x 5 cycles in one call equal five live calls: every record field, cycle = c*B + b, and n[C, B]."""
    x = xa.astype(dtype)
    eng = _engine(S_A * T_A)
    got = seq_call(eng, x, p0) if mem == "host" else seq_device(eng, x, p0)
    st = eng.stats()
    eng.close()
    want = _reference(xa, p0, dtype)
    assert_equal_runs(got, want, (p0, mem))
    assert st["cycles"] == S_A * T_A and st["decoded"] == len(want[0])


# ------------------------------------------------------------------------------------------------ pieces
@pytest.mark.gpu
def test_pieces_chain_through_the_live_state(xb):
    """max_cycles = 8, B = 3, C = 7 runs as pieces of 2, 2, 2, 1 steps; it equals seven live calls and the same input in one
    piece on a max_cycles = 21 handle."""
    ref = _engine(S_B)
    want = live_calls(ref, xb, 0)
    ref.close()
    for max_cycles in (8, 21):
        eng = _engine(max_cycles)
        assert_equal_runs(seq_call(eng, xb, 0), want, max_cycles)
        eng.close()


@pytest.mark.gpu
def test_long_recording_in_pieces(xa):
    """One stream of 40 cycles on a max_cycles = 16 handle (pieces of 16, 16, 8) equals 40 live calls of B = 1.  The
    stream is the 12 five-cycle streams one after the other."""
    x = np.ascontiguousarray(xa.transpose(1, 0, 2).reshape(-1, 180000)[:40])
    ref = _engine(1)
    want = live_calls(ref, x[:, None], 0)
    ref.close()
    eng = _engine(16)
    got = seq_call(eng, x, 0)
    eng.close()
    assert got[1].shape == (40, 1)
    assert_equal_runs(got, want)


# ------------------------------------------------------------------------------------------------ state hand-over
SCENARIOS = {
    "seq2_seq3": [("seq", 0, 2), ("seq", 2, 5)],
    "seq5": [("seq", 0, 5)],
    "live_live_seq3": [("live", 0, 1), ("live", 1, 2), ("seq", 2, 5)],
    "seq3_live_live": [("seq", 0, 3), ("live", 3, 4), ("live", 4, 5)],
}


def _run(eng, x, steps):
    recs, ns = [], []
    for kind, a, b in steps:
        r, n = (seq_call if kind == "seq" else live_calls)(eng, x[a:b], a % 2, a)
        recs.append(r)
        ns.append(n)
    return np.concatenate(recs), np.concatenate(ns)


def _next(eng, x, parity):
    r, n = eng.decode_cycles_live(x[5], parity)
    return r.copy(), n.copy()[None]


@pytest.fixture(scope="module")
def handover_ref(xb):
    """cycles 0..4 by five live calls, then cycle 5 as the next (odd) call or as a second even call in a row"""
    eng = _engine(15)
    out = {}
    for parity in (1, 0):
        eng.live_reset()
        out["run"] = _run(eng, xb, [("live", 0, 5)])
        out[parity] = _next(eng, xb, parity)
    eng.close()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(SCENARIOS))
def test_state_hand_over(xb, handover_ref, name):
    """Seq and live calls in any order leave the state C live calls leave: the same records, and the same records for one
    more call -- the next one (odd), and an even one, which reads the half of the second-to-last cycle."""
    eng = _engine(15)
    for parity in (1, 0):
        eng.live_reset()
        assert_equal_runs(_run(eng, xb, SCENARIOS[name]), handover_ref["run"], name)
        assert_equal_runs(_next(eng, xb, parity), handover_ref[parity], (name, "next call of parity", parity))
    eng.close()


# ------------------------------------------------------------------------------------------------ fresh streams
@pytest.mark.gpu
@pytest.mark.parametrize("reset", [False, True])
def test_fresh_streams(xb, reset):
    """Streams 0, 1 over cycles 0..1, then streams 0..2 over cycles 2..4: streams 0 and 1 continue, stream 2 (beyond the
    earlier B) reads a fresh ring and zero tails.  With reset, the handle first decodes two other cycles of all three
    streams and forgets them."""
    fresh = _engine(15)
    want01 = seq_call(fresh, xb[0:5, 0:2], 0)
    fresh.live_reset()
    want2 = seq_call(fresh, xb[2:5, 2:3], 0)
    fresh.close()
    w01 = _cells(want01)        # index c * 2 + b
    w2 = _cells(want2)          # index c - 2
    eng = _engine(8)
    if reset:
        eng.decode_cycles_live_seq(xb[5:7], 1)
        eng.live_reset()
    first = _cells(seq_call(eng, xb[0:2, 0:2], 0))
    second = _cells(seq_call(eng, xb[2:5], 0, 2))
    eng.close()
    bad = [("first", i) for i in range(4) if not _same(first[i], w01[i])]
    for c in range(3):
        bad += [("second", c + 2, b) for b in range(2) if not _same(second[3 * c + b], w01[2 * (c + 2) + b])]
        bad += [("joining", c + 2)] if not _same(second[3 * c + 2], w2[c]) else []
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ reference anchor
@pytest.mark.gpu
@pytest.mark.parametrize("pair", ["wav", "syn"])
def test_two_cycles_in_one_call_equal_reference(pair, golden_cycles):
    """Both golden live pairs (the unmodified reference fed the same 30 s hop by hop) through one call, C = 2, B = 1."""
    import make_golden_live as mgl
    from pyft8_b200 import messages
    g = load_golden("live_pairs.npz")
    if pair == "wav":
        a, b = golden_cycles["test_08"][0], golden_cycles["test_09"][0]
    else:
        s = mgl.synth_stream(int(g["syn_seed"]))
        a, b = s[:180000], s[180000:]
    eng = _engine(2)
    rec, n = eng.decode_cycles_live_seq(np.stack([a, b]), 0)
    eng.close()
    messages.call_hashes.clear()
    got = [_live_messages(r, None) for r in _split(rec, n[:, 0])]
    for i in range(2):
        assert [m[0] for m in got[i]] == list(g[f"{pair}_text_{i}"]), (pair, i)
        assert [m[1] for m in got[i]] == list(g[f"{pair}_notes_{i}"]), (pair, i)
        np.testing.assert_allclose([m[2] for m in got[i]], g[f"{pair}_tsec_{i}"], atol=0.005 + 1e-9)
        np.testing.assert_allclose([m[3] for m in got[i]], g[f"{pair}_fhz_{i}"], atol=0.5 + 1e-9)
        assert np.all(np.abs(np.array([m[4] for m in got[i]]) - g[f"{pair}_snr_{i}"]) <= 1)


# ------------------------------------------------------------------------------------------------ capacity and arguments
@pytest.mark.gpu
def test_record_overflow_trims_cycle_major_and_advances_the_state(xb):
    """A rec_capacity that ends inside the third cycle (in the second piece of a max_cycles = 2 handle): FT8_E_CAPACITY, the
    records that fit, n trimmed cycle-major, every cycle counted in the stats, and the next call as after five live calls."""
    x = np.ascontiguousarray(xb[:, 0])
    ref = _engine(1)
    wrec, wn = live_calls(ref, x[:5, None], 0)
    wnext = _next(ref, x[:, None], 1)
    ref.close()
    wn = wn[:, 0]
    assert wn[2] >= 2, wn
    cap = int(wn[0] + wn[1] + wn[2] // 2)
    eng = _engine(2)
    rec = np.zeros(cap, L.RECORD_DTYPE)
    n = np.zeros(5, np.int32)
    with pytest.raises(RuntimeError, match="rec_capacity too small"):
        eng.decode_cycles_live_seq(x[:5], 0, rec=rec, n=n)
    assert n.tolist() == [wn[0], wn[1], wn[2] // 2, 0, 0]
    assert rec.tobytes() == wrec[:cap].tobytes()
    st = eng.stats()
    assert st["cycles"] == 5 and st["decoded"] == int(wn.sum()), st
    assert eng.last_kernel_ms(0) > 0.0
    assert_equal_runs(_next(eng, x[:, None], 1), wnext)
    eng.close()


@pytest.mark.gpu
def test_bad_arguments_give_documented_codes():
    from pyft8_b200.engine import _ptr
    eng = _engine(2)
    audio = np.zeros((2, 2, 180000), np.int16)
    rec = np.zeros(4 * eng.max_cands, L.RECORD_DTYPE)
    n = np.zeros(4, np.int32)

    def call(a, dtype, B, Cs, odd_even):
        rc = eng._lib.ft8_decode_cycles_live_seq(eng._h, a, dtype, B, Cs, odd_even, _ptr(rec), len(rec), _ptr(n), L.MEM_HOST)
        return rc, eng._lib.last_error()

    a = _ptr(audio)
    cases = [((a, L.AUDIO_I16, 2, 0, 0), L.E_BADARG, "bad argument"),
             ((a, L.AUDIO_I16, 3, 1, 0), L.E_CAPACITY, "B exceeds cfg.max_cycles"),
             ((a, L.AUDIO_I16, 2, 2, 2), L.E_BADARG, "odd_even must be 0 or 1"),
             ((a, 7, 2, 2, 0), L.E_BADARG, "audio_dtype must be FT8_AUDIO_I16 or FT8_AUDIO_F32"),
             ((None, L.AUDIO_I16, 2, 2, 0), L.E_BADARG, "bad argument")]
    for args, code, msg in cases:
        rc, err = call(*args)
        assert rc == code and msg in err, (args[1:], rc, err)
    rc, err = call(a, L.AUDIO_I16, 2, 2, 0)                  # the handle still works
    eng.close()
    assert rc == L.OK, err


def test_python_shapes_and_dtypes_are_checked():
    """ValueError before anything reaches the library (no device needed: the checks run first)."""
    from pyft8_b200.engine import Engine
    eng = Engine.__new__(Engine)
    eng.max_cands = 200
    for bad in (np.zeros(180000, np.int16), np.zeros((1, 1, 1, 180000), np.int16), np.zeros((2, 1, 1000), np.int16),
                np.zeros((0, 1, 180000), np.int16), np.zeros((2, 0, 180000), np.int16),
                np.zeros((2, 180000), np.int32), np.zeros((2, 180000), np.float64)):
        with pytest.raises(ValueError):
            eng.decode_cycles_live_seq(bad, 0)
    with pytest.raises(ValueError):
        eng.decode_cycles_live_seq(np.zeros((2, 3, 180000), np.int16), 0, n=np.zeros(5, np.int32))
    with pytest.raises(ValueError):
        eng.decode_cycles_live_seq(np.zeros((2, 180000), np.int16), 0, rec=np.zeros(10, np.int64))


# ------------------------------------------------------------------------------------------------ WAV
def _decode_wav_live_per_cycle(path):
    """decode_wav(live=True) as it was: one B = 1 live call per cycle on a max_cycles = 1 engine"""
    from pyft8_b200.engine import Engine
    from pyft8_b200.receiver import Receiver, format_records
    from pyft8_b200.wav import read_wav
    audio = read_wav(path)
    rx = Receiver("", None)
    eng = Engine(device=rx._device, max_cycles=1, max_cands=rx.max_cands, sync_score_min=rx.sync_score_min)
    out = []
    for i in range(len(audio)):
        rec, _ = eng.decode_cycles_live(audio[i], i & 1)
        mb = format_records(rec)
        out.append([t for t, k in zip(mb.text.tolist(), mb.keep.tolist()) if k])
    eng.close()
    return out


@pytest.mark.gpu
def test_decode_wav_live_equals_per_cycle_loop(tmp_path, golden_cycles, xa):
    """test_08, test_09 and three cycles of a synthetic stream in one WAV: decode_wav(live=True) returns exactly what the
    per-cycle loop returned, message texts including hashed calls."""
    from pyft8_b200 import messages
    from pyft8_b200.wav import decode_wav, write_wav
    path = str(tmp_path / "five_cycles.wav")
    write_wav(path, np.concatenate([golden_cycles["test_08"][0], golden_cycles["test_09"][0], xa[0:3, 0].reshape(-1)]))
    messages.call_hashes.clear()
    want = _decode_wav_live_per_cycle(path)
    messages.call_hashes.clear()
    got = decode_wav(path, live=True)
    assert len(want) == 5 and all(want), [len(w) for w in want]
    assert got == want
