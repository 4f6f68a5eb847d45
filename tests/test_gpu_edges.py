"""Every stage at the edges of its search window, against the CPU oracle.

The other suites place every signal in the middle of the search window (dt in [-0.5, 1.0] s, 200..2950 Hz).  Here the
inputs are aimed at the boundary code instead:

A. the device generator ``k_synth`` for signals that start before the cycle or are cut off at its end, and at 128 signals;
B. painted dB grids: coarse search, payload gather (rows that wrap mod 750 or are not stored) and LLRs at the range ends,
   the 58-bin f0 tile edges and the h0 group / half boundaries, on 376-row grids and on the 750-row ring;
C. grids whose scores are exact integers in fp32 under any summation order: exact score ties (stable rank, cut by
   max_cands inside a tie group, earliest h0 across group and half merges) and the score threshold itself;
D. fine sync over its whole accepted input range (-100 <= h0 <= 200, 4 <= f0 <= 1880), both fine modes;
E. the whole path on a workload of early, late and band-edge signals.

Discrete decisions are asserted only where the unmarked CPU tests of this file show that the oracle's decision margin is
clear (the premises), so a near-tie fails at authoring time instead of flaking on the GPU.
"""
import ctypes as C
import functools
import math
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

import ft8_oracle as o
from conftest import ROOT
from pyft8_b200 import _lib as L
from pyft8_b200 import synth
from pyft8_b200.engine import Engine, bits91_to_int

NOISE_SIGMA = 1000.0


def _amp(snr_db, sigma=NOISE_SIGMA):
    """Signal amplitude for an SNR in 2500 Hz (synth.make_cycle's convention)."""
    return sigma * np.sqrt(2.0 * (2500.0 / 6000.0) * 10.0 ** (np.asarray(snr_db, np.float64) / 10.0))


def _symbols(seed, n):
    rng = np.random.default_rng(seed)
    return np.array([synth.symbols_from_bits77(synth.pack77(*synth.random_message(rng))) for _ in range(n)], np.uint8)


def _place(x, sym, f_hz, s0, amp):
    """Add amp * Im(waveform) starting at sample s0, clipped to the cycle (workload.host_cycle's placement)."""
    wf = np.imag(synth.shift_carrier(synth.gfsk_baseband(list(sym)), float(f_hz)))
    lo, hi = max(s0, 0), min(s0 + len(wf), 180000)
    if lo < hi:
        x[lo:hi] += float(amp) * wf[lo - s0:hi - s0]


def _start_sample(dt):
    return int((0.5 + float(dt)) * 12000)


@pytest.fixture(scope="module")
def eng():
    e = Engine(device=0, max_cycles=32)
    yield e
    e.close()


# ================================================================== A. generator at the edges
SYN_DT = (-2.0, -1.51, -0.5, 1.0, 2.0, 2.96)
SYN_F = (100.0, 101.7, 1500.3, 2994.9)


def _host_clean(sym, f, dt, amp):
    x = np.zeros(180000)
    for s in range(len(f)):
        _place(x, sym[s], f[s], _start_sample(dt[s]), amp[s])
    return np.clip(np.round(x), -32768, 32767)


def test_generator_premise_edge_placements():
    """The dt values start before the cycle (truncation toward zero differs from floor for -1.51), at it, and cut the
    waveform off at its end."""
    s0 = [_start_sample(np.float32(d)) for d in SYN_DT]
    assert s0[0] == -18000 and s0[1] < 0 and s0[2] == 0
    assert math.floor((0.5 + float(np.float32(-1.51))) * 12000) != s0[1]          # int() and floor() disagree here
    assert s0[-1] + 79 * 1920 > 180000 and s0[-2] + 79 * 1920 > 180000


@pytest.mark.gpu
def test_generator_single_signals_at_edges_equal_host_modulator(eng):
    cases = [(d, f) for d in SYN_DT for f in SYN_F]
    B = len(cases)
    sym = _symbols(61, B)[:, None, :]
    f = np.array([[c[1]] for c in cases], np.float32)
    dt = np.array([[c[0]] for c in cases], np.float32)
    amp = np.full((B, 1), 8000.0, np.float32)
    got = eng.synth_cycles(sym, f, dt, amp, 0.0, seed=3).astype(np.float64)
    for b in range(B):
        ref = _host_clean(sym[b], f[b], dt[b], amp[b])
        err = np.max(np.abs(got[b] - ref))
        assert err <= 2.0, (cases[b], err)
        assert np.count_nonzero(ref) > 50000, cases[b]                              # the signal is really in the cycle


@pytest.mark.gpu
def test_generator_128_signals_and_the_limit(eng):
    n = 128
    rng = np.random.default_rng(62)
    sym = _symbols(62, n)[None]
    f = rng.uniform(100.0, 2995.0, (1, n)).astype(np.float32)
    f[0, :len(SYN_F)] = SYN_F
    dt = rng.uniform(-2.0, 2.96, (1, n)).astype(np.float32)
    dt[0, :len(SYN_DT)] = SYN_DT
    amp = rng.uniform(50.0, 250.0, (1, n)).astype(np.float32)                      # sum stays inside int16
    got = eng.synth_cycles(sym, f, dt, amp, 0.0, seed=4)[0].astype(np.float64)
    ref = _host_clean(sym[0], f[0], dt[0], amp[0])
    assert np.max(np.abs(got - ref)) <= 2.0
    assert np.max(np.abs(ref)) < 32767
    with pytest.raises(RuntimeError, match=f"error {L.E_BADARG}: ft8_synth_cycles"):
        eng.synth_cycles(_symbols(63, 129)[None], np.full((1, 129), 1000.0, np.float32), np.zeros((1, 129), np.float32),
                         np.full((1, 129), 100.0, np.float32), 0.0)


# ================================================================== B. painted grids at boundary positions
B_H0 = (-37, -36, -34, -33, -32, -21, -5, 11, 24, 25, 41, 57, 73, 85, 86)
B_F0 = ((32, 89, 147, 901, 958), (33, 90, 148, 902, 959))      # range ends and both sides of the 58-bin tile edges


def _paint(g, f0, h0, value, row0=0):
    """Costas pattern of the middle block (the rows the coarse search scores) on both bins of each tone."""
    for k, tone in enumerate(o.COSTAS):
        g[row0 + h0 + 148 + 4 * k, f0 + 2 * tone:f0 + 2 * tone + 2] = value


@functools.lru_cache(maxsize=None)
def _painted_grid(fam, gi):
    """376-row grid: background N(10, 3) dB, five integer-valued patterns; pattern j sits at (B_F0[fam][j], h0) with the
    h0 rotated over B_H0 so that the 15 grids of a family place every h0 at every f0 of the family."""
    rng = np.random.default_rng(7000 + 100 * fam + gi)
    g = rng.normal(10.0, 3.0, (376, 976)).astype(np.float32)
    g[0] = 1.0
    painted = []
    for j, f0 in enumerate(B_F0[fam]):
        h0 = B_H0[(gi + 3 * j) % len(B_H0)]
        _paint(g, f0, h0, 30.0 + j)
        painted.append((f0, h0))
    return g, tuple(painted)


def _painted_grids():
    return [_painted_grid(fam, gi) for fam in range(2) for gi in range(len(B_H0))]


@functools.lru_cache(maxsize=None)
def _painted_ring(r):
    """750-row ring: the even half (rows 0..374) and the odd half (375..749) hold different backgrounds and patterns;
    over the three rings every h0 of B_H0 is painted in each half."""
    rng = np.random.default_rng(7500 + r)
    g = np.empty((750, 976), np.float32)
    g[:375] = rng.normal(10.0, 3.0, (375, 976))
    g[375:] = rng.normal(14.0, 4.0, (375, 976))
    even, odd = [], []
    for j in range(5):
        fe, he = B_F0[r % 2][j], B_H0[(5 * r + j) % 15]
        fo, ho = B_F0[(r + 1) % 2][j], B_H0[(5 * r + j + 7) % 15]
        _paint(g, fe, he, 30.0 + j)
        _paint(g, fo, ho, 36.0 + j, row0=375)
        even.append((fe, he))
        odd.append((fo, ho))
    return g, (tuple(even), tuple(odd))


@functools.lru_cache(maxsize=None)
def _search(key, odd_even=0):
    grid = _painted_grid(*key[1:])[0] if key[0] == "grid" else _painted_ring(key[1])[0]
    return o.search(grid, odd_even=odd_even), o.search_scores(grid, odd_even)


def _assert_clear_margins(res, scores, score_min=85.0, gap=1e-2):
    """Oracle decisions with a margin far above fp32 rounding (~1e-4 on these scores): per candidate f0 the best h0 beats
    the runner-up, candidate scores are pairwise apart, and none is near the threshold."""
    f0s, h0s, sc, _ = res
    rows = scores[np.asarray(f0s) - o.F0_LO]
    top2 = np.sort(rows, axis=1)[:, -2:]
    assert np.all(top2[:, 1] - top2[:, 0] >= gap)
    assert np.all(np.diff(np.sort(sc)) >= gap)
    assert np.all(sc - score_min >= gap)
    near = np.abs(scores.max(axis=1) - score_min) < gap
    assert not np.any(near)


def test_painted_grids_premise():
    for fam in range(2):
        for gi in range(len(B_H0)):
            res, scores = _search(("grid", fam, gi))
            _, painted = _painted_grid(fam, gi)
            got = set(zip(res[0].tolist(), res[1].tolist()))
            assert set(painted) <= got, (fam, gi)                          # every painted position is a candidate
            _assert_clear_margins(res, scores)
    wrapped = 0
    for r in range(3):
        g, halves = _painted_ring(r)
        for oe in (0, 1):
            res, scores = _search(("ring", r), oe)
            assert set(halves[oe]) <= set(zip(res[0].tolist(), res[1].tolist())), (r, oe)
            _assert_clear_margins(res, scores)
            wrapped += int(np.sum(res[1] <= -33))
    assert wrapped >= 6


def _check_sync_against_oracle(f0, h0, sc, n, pay, res, tag):
    fo, ho, so, po = res
    assert n == len(fo), tag
    assert np.array_equal(f0[:n], fo) and np.array_equal(h0[:n], ho), tag
    np.testing.assert_allclose(sc[:n], so, atol=2e-3, err_msg=str(tag))
    assert np.array_equal(pay[:n], po), tag                                        # every payload, bit-exact


def _check_llr_against_oracle(eng, pay, tag):
    llr, sd, snr = eng.llr(pay)
    for i in range(len(pay)):
        rl, rsd, rsnr = o.db_to_llr(pay[i])
        np.testing.assert_allclose(llr[i], rl, rtol=1e-5, atol=2e-5, err_msg=str((tag, i)))
        np.testing.assert_allclose(sd[i], rsd, rtol=1e-5, err_msg=str((tag, i)))
        assert snr[i] == rsnr, (tag, i)


@pytest.mark.gpu
def test_painted_grids_search_payload_llr(eng):
    grids = _painted_grids()
    f0, h0, sc, n, pay = eng.sync(np.stack([g for g, _ in grids]))
    keys = [(fam, gi) for fam in range(2) for gi in range(len(B_H0))]
    n_wrap = 0
    for b, key in enumerate(keys):
        res, _ = _search(("grid",) + key)
        nb = int(n[b])
        _check_sync_against_oracle(f0[b], h0[b], sc[b], nb, pay[b], res, key)
        wrap = h0[b, :nb] <= -33                         # first payload rows are not stored: the implicit 1.0 rows
        assert np.all(pay[b, :nb][wrap][:, 0, :] == 1.0)
        n_wrap += int(wrap.sum())
        _check_llr_against_oracle(eng, pay[b, :nb], key)
    assert n_wrap >= 20


def _sync_device(eng, grid, odd_even):
    """ft8_sync on a device-resident grid (a host 750-row ring cannot return payloads)."""
    import torch
    dev = torch.device("cuda", eng.device)
    K = eng.max_cands
    g = torch.from_numpy(np.ascontiguousarray(grid, np.float32)).to(dev)
    f0 = torch.zeros(K, dtype=torch.int16, device=dev)
    h0 = torch.zeros(K, dtype=torch.int16, device=dev)
    sc = torch.zeros(K, dtype=torch.float32, device=dev)
    n = torch.zeros(1, dtype=torch.int32, device=dev)
    pay = torch.zeros((K, 58, 8), dtype=torch.float32, device=dev)
    torch.cuda.synchronize(dev)
    P = lambda t: C.c_void_p(t.data_ptr())
    eng._check(eng._lib.ft8_sync(eng._h, P(g), grid.shape[0], 1, int(odd_even), P(f0), P(h0), P(sc), P(n), P(pay),
                                 L.MEM_DEVICE))
    torch.cuda.synchronize(dev)
    return f0.cpu().numpy(), h0.cpu().numpy(), sc.cpu().numpy(), int(n.cpu()[0]), pay.cpu().numpy()


@pytest.mark.gpu
def test_painted_ring_both_halves_search_payload_llr(eng):
    for r in range(3):
        ring, _ = _painted_ring(r)
        for oe in (0, 1):
            res, _ = _search(("ring", r), oe)
            f0, h0, sc, n, pay = _sync_device(eng, ring, oe)
            _check_sync_against_oracle(f0, h0, sc, n, pay, res, (r, oe))
            for i in np.nonzero(h0[:n] <= -33)[0]:
                # even cycle: rows 718..749 of the odd half; odd cycle: the last rows of the even half
                rows = [(375 * oe + h0[i] + 4 + 4 * s) % 750 for s in o.PAYLOAD_SYMS]
                assert (rows[0] >= 718) if oe == 0 else (rows[0] < 375)
                assert np.array_equal(pay[i], ring[rows][:, f0[i] + 1:f0[i] + 17:2])
            _check_llr_against_oracle(eng, pay[:n], (r, oe))


@pytest.mark.gpu
def test_painted_grids_batch_equals_single_calls(eng):
    grids = [_painted_grid(0, 0)[0], _painted_grid(1, 4)[0], _painted_grid(0, 9)[0], _painted_grid(1, 13)[0]]
    batch = eng.sync(np.stack(grids))
    for b, g in enumerate(grids):
        one = eng.sync(g)
        for x, y in zip(batch, one):
            assert np.array_equal(x[b], y[0]), b


# ================================================================== C. exact ties and the threshold
CENTRE_COLS = 64 + 27 * np.arange(32)          # the samples of row 185 k_sync_scores centres the dB values on


def _tone_values(score):
    """14 small integers (two bins per Costas tone x 7 rows) summing to `score`."""
    v = np.full(14, score // 14, np.float32)
    v[:score % 14] += 1
    return v.reshape(7, 2)


def _paint_values(g, f0, h0, vals):
    for k, tone in enumerate(o.COSTAS):
        g[h0 + 148 + 4 * k, f0 + 2 * tone:f0 + 2 * tone + 2] = vals[k]


def _tie_grid(patterns):
    """Zero-dB grid with integer patterns: every score of a painted (f0, h0) is the integer sum of its tone values, exact in
    fp32 whatever the summation order, because every off-tone bin of the box is 0 and the centring row stays 0."""
    g = np.zeros((376, 976), np.float32)
    for f0, h0, score in patterns:
        _paint_values(g, f0, h0, _tone_values(score))
    return g


# tie groups: scores 150 / 120 / 100 at interleaved f0, edge-ish h0; ranks 0-3, 4-8, 9-12
TIE_GROUPS = [(40, -37, 150), (70, 86, 120), (110, -33, 100), (200, 24, 150), (260, 25, 120), (330, 57, 100),
              (420, -5, 150), (500, 11, 120), (600, 41, 100), (700, 73, 150), (760, -21, 120), (830, 85, 100),
              (900, -36, 120)]
TIE_CUTS = (2, 6, 11)                           # max_cands cutting inside the first, second and third tie group
# the same pattern at two h0 of one f0 (rows do not overlap): across the half split, across 16-groups, inside a group
TIE_H0_PAIRS = [(50, 24, 25, 130), (150, -22, -21, 125), (300, 40, 41, 120), (450, 3, 4, 115)]
# threshold: exactly score_min is not a candidate, score_min + 1 is
THRESHOLD_PATTERNS = [(100, 0, 85), (300, 10, 86), (500, -30, 60), (700, 60, 61)]
THRESHOLDS = (85.0, 60.0)


def _pair_grid():
    return _tie_grid([(f0, ha, s) for f0, ha, hb, s in TIE_H0_PAIRS] + [(f0, hb, s) for f0, ha, hb, s in TIE_H0_PAIRS])


def _tie_cases():
    return [("groups", _tie_grid(TIE_GROUPS), 85.0, TIE_CUTS + (200,)),
            ("pairs", _pair_grid(), 85.0, (200,)),
            ("threshold", _tie_grid(THRESHOLD_PATTERNS), THRESHOLDS[0], (200,)),
            ("threshold", _tie_grid(THRESHOLD_PATTERNS), THRESHOLDS[1], (200,))]


def test_exact_tie_grids_premise():
    """The oracle's float64 scores are the intended integers, nothing else comes near a threshold, and the centring samples
    are 0; the expected lists follow from them."""
    for name, g, score_min, _ in _tie_cases():
        assert np.all(g[185, CENTRE_COLS] == 0.0), name
        s = o.search_scores(g)
        best = s.max(axis=1)
        near = best > score_min - 10             # everything within reach of the threshold is an exact integer
        assert np.all(best[near] == np.round(best[near])), name
    s = o.search_scores(_tie_grid(TIE_GROUPS))
    for f0, h0, score in TIE_GROUPS:
        assert s[f0 - o.F0_LO, h0 - o.H0_LO] == score
        assert np.sum(s[f0 - o.F0_LO] == score) == 1
    s = o.search_scores(_pair_grid())
    for f0, ha, hb, score in TIE_H0_PAIRS:
        row = s[f0 - o.F0_LO]
        assert row[ha - o.H0_LO] == row[hb - o.H0_LO] == score == row.max()
        assert np.count_nonzero(row == score) == 2
    s = o.search_scores(_tie_grid(THRESHOLD_PATTERNS))
    for f0, h0, score in THRESHOLD_PATTERNS:
        assert s[f0 - o.F0_LO].max() == s[f0 - o.F0_LO, h0 - o.H0_LO] == score
    # the float32 dot products of o.search give the same integers
    f0s, h0s, sc, _ = o.search(_tie_grid(TIE_GROUPS))
    assert [(int(a), int(b), float(c)) for a, b, c in zip(f0s, h0s, sc)] == \
        [(f, h, float(x)) for f, h, x in sorted(TIE_GROUPS, key=lambda t: -t[2])]
    for cut in TIE_CUTS:                                                           # each cut falls inside a tie group
        assert sc[cut - 1] == sc[cut]
    f0s, h0s, _, _ = o.search(_pair_grid())
    assert dict(zip(f0s.tolist(), h0s.tolist())) == {f0: ha for f0, ha, hb, s in TIE_H0_PAIRS}
    for score_min in THRESHOLDS:
        f0s, _, sc, _ = o.search(_tie_grid(THRESHOLD_PATTERNS), score_min)
        assert sorted(sc.tolist()) == sorted(s for _, _, s in THRESHOLD_PATTERNS if s > score_min)
        assert score_min in [p[2] for p in THRESHOLD_PATTERNS] and score_min + 1 in [p[2] for p in THRESHOLD_PATTERNS]


@pytest.mark.gpu
def test_exact_ties_and_threshold_candidate_lists(eng):
    for name, g, score_min, cuts in _tie_cases():
        for K in cuts:
            e = Engine(max_cycles=1, max_cands=K, sync_score_min=score_min)
            f0, h0, sc, n, pay = e.sync(g)
            e.close()
            res = o.search(g, score_min, K)
            n = int(n[0])
            tag = (name, score_min, K)
            assert n == len(res[0]), tag
            assert np.array_equal(f0[0, :n], res[0]) and np.array_equal(h0[0, :n], res[1]), (tag, f0[0, :n], h0[0, :n])
            assert np.array_equal(sc[0, :n], res[2].astype(np.float32)), tag      # exact: the scores are integers
            assert np.array_equal(pay[0, :n], res[3]), tag


# ================================================================== D. fine sync over its whole accepted range
D_H0 = (-100, -60, -37, -1, 0, 1, 83, 84, 86, 120, 200)
D_F0 = (4, 32, 959, 1880)
D_TT = (-8, -2, 2, 6)                  # intended time tweak (the signal sits exactly there)
D_FF = (-32, -8, 8, 32)                # intended frequency tweak in 1/16 Hz


def _fine_case_targets(i, j):
    return D_TT[(i + j) % 4], D_FF[(i + 2 * j) % 4]


@functools.lru_cache(maxsize=None)
def _fine_cycles():
    """One cycle per h0 with four +20 dB signals (one per f0 of D_F0) on low noise.  Signal j starts at sample
    60 * (tb0 + tt) -- baseband sample tb0 + tt, tb0 = int(0.5 + 200 * h0/25) -- and sits at 3.125 * f0 + ff/16 Hz,
    so the oracle's time and frequency scans peak at the intended (tt, ff) with a clear margin."""
    sym = _symbols(64, len(D_H0) * len(D_F0))
    rng = np.random.default_rng(65)
    spec = []
    for i, h0 in enumerate(D_H0):
        x = rng.normal(0.0, 300.0, 180000)
        tb0 = int(0.5 + (h0 / 25) / 0.005)
        for j, f0 in enumerate(D_F0):
            tt, ff = _fine_case_targets(i, j)
            _place(x, sym[4 * i + j], 3.125 * f0 + ff / 16, 60 * (tb0 + tt), _amp(20.0, 300.0))
        spec.append(o.cycle_spectrum(np.clip(np.round(x), -32768, 32767).astype(np.int16)))
    return np.stack(spec)


@functools.lru_cache(maxsize=None)
def _fine_oracle(i, j):
    spec = _fine_cycles()[i]
    return o.llr_fine(spec, 3.125 * D_F0[j], D_H0[i] / 25)


def _fine_scan_scores(spec, f0, h0):
    """The oracle's time-scan and frequency-scan scores (o.llr_fine's two arg-max inputs)."""
    fb0, tb0 = int(0.5 + 3.125 * f0 * o.NFFT_CYCLE / o.SAMP_RATE), int(0.5 + (h0 / 25) / 0.005)
    z = o.fine_baseband(spec, fb0)
    ts = np.array([o.fine_score(o.fine_grid_from_baseband(z, tb0 + t)) for t in range(-8, 8, 2)])
    tt = -8 + 2 * int(np.argmax(ts))
    fs = np.array([o.signal_grid_fine(spec, fb0 + f, tb0 + tt)[1] for f in range(-32, 33, 8)])
    return ts, fs


def _rel_gap(s):
    top = np.sort(s)[-2:]
    return (top[1] - top[0]) / abs(top[1])


def test_fine_time_origin_rule():
    """The kernels' tb0 = 8*h0 (h0 >= 0) / 8*h0 + 1 (h0 < 0) is int(0.5 + tsec/0.005) with tsec = h0/25 over the accepted range."""
    for h0 in range(-100, 201):
        assert int(0.5 + (h0 / 25) / 0.005) == (8 * h0 if h0 >= 0 else 8 * h0 + 1), h0


def test_fine_cases_premise():
    """Per case: the oracle's top-two time-scan and frequency-scan scores differ by >= 1e-3 relative; the Costas-row arg-max
    behind nsync and the snr's integer part are clear of fp32 noise.  The set reaches the clipping of the first symbols,
    of the last Costas symbol and of payload symbols."""
    spec = _fine_cycles()
    n_pass, tts, ffs = 0, set(), set()
    for i, h0 in enumerate(D_H0):
        for j, f0 in enumerate(D_F0):
            ts, fs = _fine_scan_scores(spec[i], f0, h0)
            assert _rel_gap(ts) >= 1e-3 and _rel_gap(fs) >= 1e-3, (h0, f0, _rel_gap(ts), _rel_gap(fs))
            r = _fine_oracle(i, j)
            tts.add(r["tt"])
            ffs.add(r["ff"])
            g = r["grid"]
            top = np.sort(g[list(o.COSTAS_SYMS)], axis=1)[:, -2:]
            assert np.all(top[:, 1] - top[:, 0] >= 1e-4 * g.max()), (h0, f0)
            if r["nsync"] > 6:
                n_pass += 1
                p = 20 * np.log10(g[list(o.PAYLOAD_SYMS)])
                d = float(np.max(p) - np.min(p) - 58)
                assert abs(d) > 25 or abs(d - round(d)) > 1e-3, (h0, f0, d)
    assert n_pass >= 30
    assert {-8, 6} <= tts and {-32, 32} <= ffs                                  # both ends of both scans are chosen
    tb = [int(0.5 + (h / 25) / 0.005) for h in D_H0]
    assert min(tb) - 8 < 0                                                      # first symbols clipped to 0
    assert any(t + 6 + 32 * 78 > o.NFFT_FINE - 32 and t + 32 * 71 + 6 <= o.NFFT_FINE - 32 for t in tb)   # last Costas only
    assert max(tb) + 32 * 71 > o.NFFT_FINE - 32                                # payload symbols clipped


@pytest.mark.gpu
@pytest.mark.parametrize("fine_mode", [0, 1])
def test_fine_sync_whole_input_range(fine_mode):
    spec = _fine_cycles()
    co = np.repeat(np.arange(len(D_H0), dtype=np.int32), len(D_F0))
    h0 = np.repeat(np.array(D_H0, np.int16), len(D_F0))
    f0 = np.tile(np.array(D_F0, np.int16), len(D_H0))
    e = Engine(max_cycles=len(D_H0), fine_mode=fine_mode)
    r = e.fine(spec, co, f0, h0)
    e.close()
    for k in range(len(co)):
        i, j = k // len(D_F0), k % len(D_F0)
        ref = _fine_oracle(i, j)
        tag = (fine_mode, int(h0[k]), int(f0[k]))
        assert (r["tt"][k], r["ff"][k], r["nsync"][k]) == (ref["tt"], ref["ff"], ref["nsync"]), (tag, r["tt"][k], r["ff"][k], r["nsync"][k], ref)
        if ref["nsync"] > 6:
            g = ref["grid"]
            np.testing.assert_allclose(r["grid"][k], g, rtol=2e-5, atol=2e-6 * g.max(), err_msg=str(tag))
            with np.errstate(all="ignore"):
                llr, sd, snr = o.db_to_llr(20 * np.log10(g[list(o.PAYLOAD_SYMS)]))
            np.testing.assert_allclose(r["llr"][k], llr, rtol=1e-3, atol=1e-3, err_msg=str(tag))
            np.testing.assert_allclose(r["sd"][k], sd, rtol=1e-4, err_msg=str(tag))
            assert r["snr"][k] == snr, tag


# ================================================================== E. whole path on an edge workload
E_CYCLES, E_SIGNALS, E_SEED = 32, 20, 2026
E_MIN_PER_CLASS = 20                   # oracle decodes per edge class, at least (measured: 30..207 per class)
E_CLASSES = {"h0<-12": lambda f0, h0: h0 < -12, "h0>37": lambda f0, h0: h0 > 37,
             "f0<64": lambda f0, h0: f0 < 64, "f0>944": lambda f0, h0: f0 > 944}


@functools.lru_cache(maxsize=None)
def _edge_params():
    """dt from [-2.0, -0.6] u [1.1, 2.9] s; half the signals at 100..200 Hz or 2950..2995 Hz, the rest in the usual band."""
    rng = np.random.default_rng(E_SEED)
    shape = (E_CYCLES, E_SIGNALS)
    sym = _symbols(E_SEED, 256)[rng.integers(0, 256, shape)]
    dt = np.where(rng.random(shape) < 0.5, rng.uniform(-2.0, -0.6, shape), rng.uniform(1.1, 2.9, shape))
    f_edge = np.where(rng.random(shape) < 0.5, rng.uniform(100.0, 200.0, shape), 2995.0 - rng.uniform(0.0, 45.0, shape))
    f = np.where(np.arange(E_SIGNALS) % 2 == 0, f_edge, rng.uniform(200.0, 2950.0, shape))
    amp = _amp(rng.uniform(-16.0, 5.0, shape))
    return dict(symbols=sym, f_hz=f.astype(np.float32), dt_s=dt.astype(np.float32), amp=amp.astype(np.float32))


def _edge_host_cycle(b):
    p = _edge_params()
    x = np.random.default_rng(E_SEED * 1000 + b).normal(0.0, NOISE_SIGMA, 180000)
    for s in range(E_SIGNALS):
        _place(x, p["symbols"][b, s], p["f_hz"][b, s], _start_sample(p["dt_s"][b, s]), p["amp"][b, s])
    return np.clip(np.round(x), -32768, 32767).astype(np.int16)


def _oracle_cycle(a):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ft8_oracle as orc
    recs, cl = orc.decode_cycle(a)
    return [(r["bits77"], r["notes"], r["tsec"], r["fHz"], r["snr"], cl[r["cand"]].f0, cl[r["cand"]].h0) for r in recs]


@pytest.fixture(scope="module")
def pool():
    with mp.get_context("spawn").Pool(os.cpu_count() or 1) as p:
        yield p


def _class_counts(ref):
    return {k: sum(fn(x[5], x[6]) for cyc in ref for x in cyc) for k, fn in E_CLASSES.items()}


def test_edge_workload_premise(pool):
    """The oracle really decodes early, late and band-edge stations of this workload (host-modulated copy of it)."""
    ref = pool.map(_oracle_cycle, [_edge_host_cycle(b) for b in range(E_CYCLES)], chunksize=1)
    counts = _class_counts(ref)
    print("[edge_workload] host-modulated oracle decodes per class:", counts, "total", sum(map(len, ref)))
    assert all(v >= E_MIN_PER_CLASS for v in counts.values()), counts


@pytest.mark.gpu
def test_edge_workload_gpu_vs_oracle(pool):
    p = _edge_params()
    e = Engine(max_cycles=E_CYCLES)
    audio = e.synth_cycles(p["symbols"], p["f_hz"], p["dt_s"], p["amp"], NOISE_SIGMA, seed=E_SEED)
    rec, n = e.decode_cycles(audio)
    e.close()
    ref = pool.map(_oracle_cycle, [audio[b] for b in range(E_CYCLES)], chunksize=1)
    from pyft8_b200.receiver import record_to_message
    set_diff, order_bad, notes_bad, tol_bad = [], [], [], []
    off = 0
    for b in range(E_CYCLES):
        r = rec[off:off + n[b]]
        off += n[b]
        em = r[r["emitted"] == 1]
        got = [bits91_to_int(x["bits91"]) >> 14 for x in em]
        want = [x[0] for x in ref[b]]
        assert len(got) == len(set(got)), b
        if set(got) != set(want):
            set_diff.append((b, sorted("%x" % v for v in set(got) ^ set(want))))
        elif got != want:
            order_bad.append(b)
        refmap = {x[0]: x for x in ref[b]}
        for x, g in zip(em, got):
            if g in refmap:
                m = record_to_message(x)
                if m["decode_notes"] != refmap[g][1]:
                    notes_bad.append((b, "%x" % g, m["decode_notes"], refmap[g][1]))
                if abs(m["tsec"] - refmap[g][2]) > 0.005 + 1e-9 or abs(m["fHz"] - refmap[g][3]) > 0.5 + 1e-9 \
                        or abs(int(m["their_snr"]) - refmap[g][4]) > 1:
                    tol_bad.append((b, "%x" % g))
    counts = _class_counts(ref)
    rep = dict(ref_decodes=sum(map(len, ref)), class_counts=counts, set_differences=set_diff[:8], order_differs=order_bad,
               notes_differ=notes_bad[:8], dt_df_snr_out_of_tolerance=tol_bad[:8])
    print("[edge_workload]", rep)
    assert all(v >= E_MIN_PER_CLASS for v in counts.values()), rep
    assert not set_diff, rep
    assert not tol_bad, rep
    assert len(order_bad) <= 1 and len(notes_bad) <= 1, rep
