"""Every decode knob of ft8_cfg through every decode entry point, against the CPU oracle with the same knobs.

The knobs mirror the reference's keyword arguments, and each is read at one place of the device path:

    search_h0_lo/hi            k_sync_scores (relative to the cycle's hop 0: 0, 375 or 5 by mode)
    search_f0_lo/hi, sync_score_min, max_cands                              k_topk
    llr_sd_min                 the sd gates of k_pass0 and k_pass234
    osd_singleflips / osd_doubleflips                                       k_osd_items
    fine_mode                  which fine-sync kernels run (no effect on results)

Three workloads aim them:

A. isolated low-SNR cycles in the style of cfg4_120sig, which decode in every pass including OSD (ipass 5 and 6), through
   decode_cycles from host and device memory, one cycle per call so that the work counters of ft8_stats can be compared
   with the oracle's cycle by cycle (ft8_oracle.work_counters);
B. continuous streams with stations that straddle every cycle boundary (test_gpu_live.py's), through decode_cycles_live
   against the ring model and through decode_cycles_live_seq against sequential live calls, where the h0 window decides
   whether a station that reads the other ring half is a candidate at all;
C. the Python front ends (Receiver, decode_wav), which must hand the receiver's ranges to every engine they create.

The unmarked tests are the premises: each knob value changes the oracle's output on its workload, and no candidate's sd
lies within 1e-3 (relative) of a chosen threshold, so that a kernel that ignores a knob fails and a correct one cannot flake.
"""
import multiprocessing as mp
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from pyft8_b200 import _lib as L
from test_gpu_live import _split, compare_with_model, make_sequence, model_records, ring_model_cycle, run_model
from test_gpu_live_seq import assert_equal_runs, live_calls, seq_call

COUNTERS = ("candidates", "stopped_sd", "fine_evals", "fine_pass", "ldpc_calls", "osd_calls")
SD_GAP = 1e-3                         # least relative distance of any candidate sd from a chosen llr_sd_min

# ------------------------------------------------------------------------------------------------ knob sets (Engine kwargs)
ISO_N, ISO_SEED = 4, 41               # cfg4_120sig-style cycles
ISO_ROWS = {
    "default": {},
    "sd3": dict(llr_sd_min=3.0),
    "sd6.865": dict(llr_sd_min=6.865),
    "sd7.9": dict(llr_sd_min=7.9),
    "osd0_0": dict(osd_singleflips=0, osd_doubleflips=0),
    "osd10_0": dict(osd_singleflips=10, osd_doubleflips=0),
    "osd30_25": dict(osd_singleflips=30, osd_doubleflips=25),
    "osd91_2": dict(osd_singleflips=91, osd_doubleflips=2),
    "combined": dict(sync_score_min=70.0, max_cands=150, llr_sd_min=6.865, osd_singleflips=10, osd_doubleflips=1,
                     search_f0_range=(90, 902), search_h0_range=(-31, 60), fine_mode=1),
}
SD_ROWS = ("sd3", "sd6.865", "sd7.9")
OSD_ROWS = ("osd0_0", "osd10_0", "osd30_25", "osd91_2")

# live streams: 3 x 4 cycles starting even, 3 x 3 starting odd
LIVE_SEQS = {"even": (500, 3, 4, 0), "odd": (600, 3, 3, 1)}
LIVE_ROWS = {
    "default": {},
    "h0_other_half": dict(search_h0_range=(-37, -31), search_f0_range=(90, 902)),   # only stations that read the other half
    "h0_own_half": dict(search_h0_range=(-31, 87), search_f0_range=(160, 480)),     # excludes them; 500-1500 Hz
    "h0_0_40": dict(search_h0_range=(0, 40), search_f0_range=(90, 902)),
    "score70_k40": dict(sync_score_min=70.0, max_cands=40),
    "score100_k928": dict(sync_score_min=100.0, max_cands=928),
    "sd2.9": dict(llr_sd_min=2.9),
    "osd10_0": dict(osd_singleflips=10, osd_doubleflips=0),
}
WINDOW_ROWS = ("h0_other_half", "h0_own_half", "h0_0_40")
EARLY_H0 = -32                        # h0 <= -32: a payload row of an even cycle wraps into the odd half
# decode_cycles_live_seq: every knob non-default, fine_mode 1, C * B = 12 > max_cycles = 7 (pieces of 2 + 2 steps)
SEQ_KNOBS = dict(sync_score_min=75.0, max_cands=120, llr_sd_min=2.9, osd_singleflips=10, osd_doubleflips=1,
                 search_f0_range=(90, 902), search_h0_range=(-37, 60), fine_mode=1)
SEQ_MAX_CYCLES = 7


def oracle_kw(knobs):
    """Engine keyword arguments -> ft8_oracle search / decode_cycle keyword arguments (fine_mode has no oracle side)"""
    return dict(score_min=knobs.get("sync_score_min", 85), max_cands=knobs.get("max_cands", 200),
                f0_range=knobs.get("search_f0_range"), h0_range=knobs.get("search_h0_range"),
                llr_sd_min=knobs.get("llr_sd_min", 5), osd_singleflips=knobs.get("osd_singleflips", 30),
                osd_doubleflips=knobs.get("osd_doubleflips", 2))


def _summary(recs, cl):
    """(records as the ring model gives them, work counters, every sd the sd gates compared)"""
    import ft8_oracle as o
    sds = [c.grid_sd for c in cl] + [c.fine_sd for c in cl if not np.isnan(c.fine_sd)]
    return model_records(recs, cl), o.work_counters(cl), sds


# ------------------------------------------------------------------------------------------------ pool jobs
def _iso_audio_job(b):
    from pyft8_b200 import workload
    return workload.host_cycle(workload.make_params("cfg4_120sig", ISO_N, seed=ISO_SEED), b)


def _iso_oracle_job(job):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ft8_oracle as o
    audio, knobs = job
    kw = oracle_kw(knobs)
    grid = o.spectrogram(audio)
    cands = o.search(grid, kw.pop("score_min"), kw.pop("max_cands"), 0, kw.pop("f0_range"), kw.pop("h0_range"))
    return _summary(*o.decode_cycle(audio, grid=grid, cands=cands, **kw))


def _live_model_job(job):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    return _summary(*ring_model_cycle(*job))


# ------------------------------------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def pool():
    with mp.get_context("spawn").Pool(os.cpu_count() or 1) as p:
        yield p


@pytest.fixture(scope="module")
def iso_audio(pool):
    return np.stack(pool.map(_iso_audio_job, range(ISO_N), chunksize=1))


@pytest.fixture(scope="module")
def iso_oracle(pool, iso_audio):
    """iso_oracle[row][b] = (records, counters, sds) of cycle b"""
    jobs = [(iso_audio[b], ISO_ROWS[r]) for r in ISO_ROWS for b in range(ISO_N)]
    res = pool.map(_iso_oracle_job, jobs, chunksize=1)
    return {r: res[i * ISO_N:(i + 1) * ISO_N] for i, r in enumerate(ISO_ROWS)}


@pytest.fixture(scope="module")
def live_seqs(pool):
    return {k: make_sequence(pool, seed, S, T) for k, (seed, S, T, p0) in LIVE_SEQS.items()}


@pytest.fixture(scope="module")
def live_oracle(pool, live_seqs):
    """live_oracle[row][seq][s][k] = (records, counters, sds) of the ring model with the row's knobs"""
    out = {}
    for r, knobs in list(LIVE_ROWS.items()) + [("seq", SEQ_KNOBS)]:
        kw = oracle_kw(knobs) if knobs else None
        out[r] = {k: run_model(pool, live_seqs[k], LIVE_SEQS[k][3], knobs=kw, job=_live_model_job)
                  for k in (LIVE_SEQS if r != "seq" else ("even",))}
    return out


def _cells(model):
    """(seq, stream, cycle, summary) of every stream-cycle of one row"""
    return [(q, s, k, x) for q in model for s, row in enumerate(model[q]) for k, x in enumerate(row)]


def _sd_margin(sds, thr):
    return float(np.min(np.abs(np.asarray(sds, np.float64) - thr))) / thr


# ------------------------------------------------------------------------------------------------ premises (CPU)
def test_sd_thresholds_clear_every_candidate_sd(iso_oracle, live_oracle):
    """No grid_sd or fine_sd of any candidate, in any run of either workload, lies within SD_GAP (relative) of the chosen
    llr_sd_min values (the device sds agree with the oracle's to about 1e-4)."""
    iso = [v for row in iso_oracle.values() for x in row for v in x[2]]
    live = [v for row in live_oracle.values() for (_, _, _, x) in _cells(row) for v in x[2]]
    margins = {}
    for thr in sorted({ISO_ROWS[r]["llr_sd_min"] for r in SD_ROWS + ("combined",)}):
        margins[f"iso {thr}"] = _sd_margin(iso, thr)
    for thr in sorted({LIVE_ROWS["sd2.9"]["llr_sd_min"], SEQ_KNOBS["llr_sd_min"]}):
        margins[f"live {thr}"] = _sd_margin(live, thr)
    print(f"[knobs] relative sd margins: { {k: round(v, 5) for k, v in margins.items()} } over {len(iso)} + {len(live)} sds")
    assert min(margins.values()) > SD_GAP, margins


def _changed(a, b):
    """cycles whose emitted (payload, notes) list or counters differ"""
    return sum([r[:2] for r in x[0]] != [r[:2] for r in y[0]] or x[1] != y[1] for x, y in zip(a, b))


def test_workload_decodes_in_every_pass(iso_oracle):
    """The isolated workload decodes in ipass 0, fine passes and OSD: ipass-5/6 decodes are what S and D decide."""
    ipass = {}
    for x in iso_oracle["default"]:
        for r in x[0]:
            ip = {"grid": 0}.get(r[1].split("_")[0], 2)
            ipass[ip] = ipass.get(ip, 0) + 1
    osd = sum(r[1].split("_")[-1].startswith("OSD") for x in iso_oracle["default"] for r in x[0])
    print(f"[knobs] isolated default decodes: grid {ipass.get(0, 0)}, fine {ipass.get(2, 0)} of which OSD {osd}")
    assert ipass.get(0, 0) > 20 * ISO_N and osd >= 2 * ISO_N, (ipass, osd)


def test_each_knob_value_changes_the_oracle(iso_oracle):
    """Each llr_sd_min changes the decodes or counters of some cycle compared with 5; each (S, D) pair changes the decodes or
    the OSD successes compared with (30, 2)."""
    base = iso_oracle["default"]
    rep = {}
    for r in SD_ROWS + ("combined",):
        rep[r] = _changed(iso_oracle[r], base)
    for r in OSD_ROWS:
        osd = lambda rows: [sorted((x[0], x[1]) for x in c[0] if "OSD" in x[1]) for c in rows]
        rep[r] = sum(a != b for a, b in zip(osd(iso_oracle[r]), osd(base)))
    print(f"[knobs] cycles whose oracle output each knob value changes (of {ISO_N}): {rep}")
    assert min(rep.values()) >= 1, rep


def test_live_knobs_change_the_ring_model(live_oracle):
    """Each live row changes the ring model's output; the h0 windows select the boundary stations as intended: (-37, -31)
    decodes only stations that read the other ring half, (-31, 87) none of them, (0, 40) only h0 in [0, 40)."""
    base = {(q, s, k): x for q, s, k, x in _cells(live_oracle["default"])}
    rep, early = {}, {}
    for r in LIVE_ROWS:
        if r == "default":
            continue
        cells = _cells(live_oracle[r])
        rep[r] = sum([y[:2] for y in x[0]] != [y[:2] for y in base[q, s, k][0]] or x[1] != base[q, s, k][1]
                     for q, s, k, x in cells)
        early[r] = sum(y[5] <= EARLY_H0 for _, _, _, x in cells for y in x[0])
    early["default"] = sum(y[5] <= EARLY_H0 for x in base.values() for y in x[0])
    h0 = {r: [y[5] for _, _, _, x in _cells(live_oracle[r]) for y in x[0]] for r in WINDOW_ROWS}
    print(f"[knobs] live stream-cycles each row changes: {rep}; decodes with h0 <= {EARLY_H0}: {early}")
    assert min(rep.values()) >= 2, rep
    assert early["h0_other_half"] >= 4 and all(v <= EARLY_H0 for v in h0["h0_other_half"]), h0["h0_other_half"]
    assert early["h0_own_half"] == 0 and early["default"] >= 4, early
    assert h0["h0_0_40"] and all(0 <= v < 40 for v in h0["h0_0_40"]), h0["h0_0_40"]


# ------------------------------------------------------------------------------------------------ GPU: isolated cycles
def _counter_diff(st, want):
    return {k: (int(st[k]), want[k]) for k in COUNTERS if st[k] != want[k]}


@pytest.mark.gpu
@pytest.mark.parametrize("row", list(ISO_ROWS))
def test_isolated_decode_with_knobs_matches_oracle(iso_audio, iso_oracle, row):
    """decode_cycles on a B = 1 handle with the row's cfg, cycle by cycle: emitted payload sets exact, dt / df / SNR within
    tolerance, order and notes differences bounded (test_gpu_live.compare_with_model), and the work counters of ft8_stats
    equal the oracle's exactly.  The same audio from device memory gives the same records and counters."""
    import torch
    from pyft8_b200.engine import Engine
    eng = Engine(max_cycles=1, **ISO_ROWS[row])
    got, bad = [], []
    for b in range(ISO_N):
        rec, _ = eng.decode_cycles(iso_audio[b:b + 1])
        rec, st = rec.copy(), eng.stats()
        got.append(rec)
        d = _counter_diff(st, iso_oracle[row][b][1])
        if d:
            bad.append((b, d))
        dev = torch.from_numpy(iso_audio[b:b + 1]).to("cuda:0")
        drec, _ = eng.decode_cycles_dev(dev.data_ptr(), L.AUDIO_I16, 1)
        assert drec.tobytes() == rec.tobytes() and eng.stats() == st, (row, b, "device audio differs from host audio")
    eng.close()
    compare_with_model([got], [[x[0] for x in iso_oracle[row]]], 0)
    assert not bad, (row, "work counters differ from the oracle (gpu, oracle)", bad)


# ------------------------------------------------------------------------------------------------ GPU: live and consecutive live
@pytest.mark.gpu
@pytest.mark.parametrize("row", list(LIVE_ROWS))
def test_live_decode_with_knobs_matches_ring_model(live_seqs, live_oracle, row):
    """decode_cycles_live with the row's cfg, a sequence starting with each parity: every stream-cycle against the ring model
    with the same knobs (the criteria of test_live_sequence_matches_ring_model), and each call's work counters equal the sum
    of its streams' oracle counters."""
    from pyft8_b200.engine import Engine
    bad = []
    for q, (_, S, T, p0) in LIVE_SEQS.items():
        model = live_oracle[row][q]
        eng = Engine(max_cycles=S, **LIVE_ROWS[row])
        got = [[None] * T for _ in range(S)]
        for k in range(T):
            rec, n = eng.decode_cycles_live(np.ascontiguousarray(live_seqs[q][:, k]), (p0 + k) % 2)
            for s, r in enumerate(_split(rec, n)):
                got[s][k] = r
            d = _counter_diff(eng.stats(), {c: sum(model[s][k][1][c] for s in range(S)) for c in COUNTERS})
            if d:
                bad.append((q, k, d))
        eng.close()
        compare_with_model(got, [[x[0] for x in m] for m in model], p0, min_model_decodes=S)
    assert not bad, (row, "work counters differ from the ring model (gpu, oracle)", bad)


@pytest.mark.gpu
def test_live_seq_with_every_knob_equals_live_calls_and_ring_model(live_seqs, live_oracle):
    """decode_cycles_live_seq with every knob non-default (fine_mode 1 included) and C * B > max_cycles, so that the call
    runs in two pieces: records and counts bit-identical with sequential live calls on a handle with the same cfg, the
    records against the ring model, and the call's work counters equal the oracle's over all its stream-cycles."""
    from pyft8_b200.engine import Engine
    _, S, T, p0 = LIVE_SEQS["even"]
    x = np.ascontiguousarray(live_seqs["even"].transpose(1, 0, 2))          # [T, S, 180000]
    assert S * T > SEQ_MAX_CYCLES and SEQ_MAX_CYCLES >= 2 * S
    ref = Engine(max_cycles=S, **SEQ_KNOBS)
    want = live_calls(ref, x, p0)
    ref.close()
    eng = Engine(max_cycles=SEQ_MAX_CYCLES, **SEQ_KNOBS)
    got = seq_call(eng, x, p0)
    st = eng.stats()
    eng.close()
    assert_equal_runs(got, want, "seq vs live calls")
    model = live_oracle["seq"]["even"]
    cells = _split(got[0], got[1].ravel())                                    # index c * S + s
    compare_with_model([[cells[k * S + s] for k in range(T)] for s in range(S)], [[x_[0] for x_ in m] for m in model], p0,
                       min_model_decodes=S)
    d = _counter_diff(st, {c: sum(m[k][1][c] for m in model for k in range(T)) for c in COUNTERS})
    assert not d, d


# ------------------------------------------------------------------------------------------------ GPU: Python front ends
RX_KW = dict(search_freq_range=[500, 1500], search_time_range=[-1.0, 1.0], sync_score_min=80, max_cands=60)
RX_RANGES = [[160, 480], [-12, 37]]     # int(f / 3.125), int((t + 0.5) * 25): receiver.py:232, 319
BAND = (160, 480)                       # search_freq_range=[500, 1500] alone


def _texts(rec):
    """kept message texts of one cycle's records, as decode_wav(live=True) formats them"""
    from pyft8_b200.receiver import format_records
    mb = format_records(rec)
    return [t for t, k in zip(mb.text.tolist(), mb.keep.tolist()) if k]


def _live_loop(eng, audio):
    """records of one B = 1 live call per cycle, the first even"""
    return [eng.decode_cycles_live(audio[i], i & 1)[0].copy() for i in range(len(audio))]


def _msg_key(m):
    return (" ".join(m["msg_tuple"]), m["tsec"], m["fHz"], m["their_snr"], m["decode_notes"])


@pytest.fixture(scope="module")
def wav_audio(live_seqs, tmp_path_factory):
    """stream 0 of the even live sequence: int16 [4, 180000] and the same as a WAV file"""
    from pyft8_b200.wav import write_wav
    a = np.ascontiguousarray(live_seqs["even"][0])
    path = str(tmp_path_factory.mktemp("knobs") / "stream0.wav")
    write_wav(path, a)
    return a, path


@pytest.mark.gpu
def test_receiver_forwards_knobs_to_isolated_decodes(wav_audio):
    """Receiver(search_freq_range, search_time_range, sync_score_min, max_cands) derives the reference's index ranges, and
    decode_cycles, decode_cycles_columnar and decode_wav(live=False) each equal a direct Engine call with those knobs."""
    from pyft8_b200 import messages
    from pyft8_b200.engine import Engine
    from pyft8_b200.receiver import Receiver, format_records
    from pyft8_b200.wav import decode_wav
    a, path = wav_audio
    rx = Receiver("", None, **RX_KW)
    assert [list(r) for r in rx._search_ranges] == RX_RANGES
    eng = Engine(max_cycles=len(a), max_cands=RX_KW["max_cands"], sync_score_min=RX_KW["sync_score_min"],
                 search_f0_range=RX_RANGES[0], search_h0_range=RX_RANGES[1])
    rec = eng.decode_cycles(a)[0].copy()
    eng.close()
    assert len(rec) > 0 and np.all((rec["f0_idx"] >= RX_RANGES[0][0]) & (rec["f0_idx"] < RX_RANGES[0][1]))
    assert np.all((rec["h0_idx"] >= RX_RANGES[1][0]) & (rec["h0_idx"] < RX_RANGES[1][1]))
    messages.call_hashes.clear()
    mb = format_records(rec)
    want = [[] for _ in range(len(a))]
    for i in np.flatnonzero(mb.keep):
        want[int(mb.cycle[i])].append(" ".join(mb.msg_tuple[i]))
    messages.call_hashes.clear()
    got = rx.decode_cycles(a, emit=False)
    assert [[" ".join(m["msg_tuple"]) for m in c] for c in got] == want
    messages.call_hashes.clear()
    assert rx.decode_cycles_columnar(a).rec.tobytes() == rec.tobytes()
    messages.call_hashes.clear()
    assert [[_msg_key(m) for m in c] for c in decode_wav(path, receiver=rx)] == [[_msg_key(m) for m in c] for c in got]


@pytest.mark.gpu
def test_decode_wav_live_honours_search_ranges(wav_audio):
    """decode_wav(live=True) hands the receiver's ranges to its engine: with search_freq_range=[500, 1500] it returns what a
    per-cycle live loop on an engine with f0 in [160, 480) returns, and none of the messages the full band adds outside it;
    with receiver=rx it honours rx's narrow ranges and thresholds."""
    from pyft8_b200 import messages
    from pyft8_b200.engine import Engine
    from pyft8_b200.receiver import Receiver
    from pyft8_b200.wav import decode_wav
    a, path = wav_audio
    full_eng = Engine(max_cycles=1)
    full = _live_loop(full_eng, a)
    full_eng.close()
    band_eng = Engine(max_cycles=1, search_f0_range=BAND)
    band = _live_loop(band_eng, a)
    band_eng.close()
    messages.call_hashes.clear()
    want = [_texts(r) for r in band]
    messages.call_hashes.clear()
    outside = [set(_texts(r[(r["f0_idx"] < BAND[0]) | (r["f0_idx"] >= BAND[1])])) - set(w) for r, w in zip(full, want)]
    assert sum(map(len, outside)) >= 5 and sum(map(len, want)) >= 5, (outside, want)
    messages.call_hashes.clear()
    got = decode_wav(path, live=True, search_freq_range=[500, 1500])
    assert not [t for g, o_ in zip(got, outside) for t in g if t in o_], "messages from outside the band"
    assert got == want
    rx_eng = Engine(max_cycles=1, max_cands=RX_KW["max_cands"], sync_score_min=RX_KW["sync_score_min"],
                    search_f0_range=RX_RANGES[0], search_h0_range=RX_RANGES[1])
    narrow = _live_loop(rx_eng, a)
    rx_eng.close()
    messages.call_hashes.clear()
    want_rx = [_texts(r) for r in narrow]
    rx = Receiver("", None, **RX_KW)
    messages.call_hashes.clear()
    assert decode_wav(path, receiver=rx, live=True) == want_rx
