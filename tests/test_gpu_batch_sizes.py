"""Decodes at the benchmark's batch sizes: every cycle of bench.py's 4096-cycle cfg2 batch and 8192-cycle cfg4 batch.

Some host and kernel code only runs when one call holds more than 1024 cycles, or more than 256 host cycles:
* F1 (`launch_cycle_spectrum`) works in scratch chunks of 1024 cycles, and from the second chunk on it offsets the audio and
  spectrum pointers by the chunk start.  Device-resident or prefetched audio with B > 1024 reaches that loop, and so does
  ft8_cycle_spectrum with B > 1024.  Host audio is copied and decoded in chunks of at most 256 cycles and never does.
* `k_rec_scan` carries the record base from one block of 1024 cycles to the next.
* host audio is copied in min(16, ceil(B / 256)) chunks, the last one shorter when B is not a multiple of the chunk.
* the streaming entry's prefetch and the cycle-major capacity cut of the records, past the first 1024 cycles.

The reference for every cycle is the same audio decoded in slices of 1000 cycles on a max_cycles = 1000 handle, at device
pointer offsets into the same tensor.  A slice takes one scratch chunk and one scan block, and its boundaries fall at other
cycles than the large batch's.  Cycles are decoded independently, so each cycle's records must be byte-identical in both,
once `cycle` is shifted by the slice start; so must the per-cycle counts and the work counters.  The CPU oracle anchors a
sample of cycles on both sides of every internal boundary.

Device scratch, staged audio and records are never cleared between calls, so a handle that had decoded the same batch
before could pass on its leftovers: every path under test runs on a fresh handle, and only one large handle is alive at a
time.  Each test prints what it measured (sizes, record counts, device memory in use) as a `[batch_sizes]` line.
"""
import ctypes as C
import json
import multiprocessing as mp
import os

import numpy as np
import pytest

from pyft8_b200 import _lib as L
from pyft8_b200 import workload
from test_gpu_large import _oracle_cycle
from test_gpu_live_seq import assert_equal_runs, live_calls, seq_call, seq_device

pytestmark = pytest.mark.gpu

CYCLE_BYTES = 180000 * 2                      # one int16 cycle
SLICE = 1000                                  # reference batch: under 1024, not a multiple of 256 or 1024
CFG2 = ("cfg2_50sig", 4096, 2000)             # bench.py's headline batch: rank 0 at the default --seed
CFG4 = ("cfg4_120sig", 8192, 2004)            # bench.py's configs[3]: --cfg4-cycles at --seed + 4
ORACLE_CFG2 = [0, 1, 255, 256, 999, 1000, 1023, 1024, 1025, 2047, 2048, 3071, 3072, 4095]
ORACLE_CFG4 = [1023, 1024, 4095, 4096, 5119, 5120, 6143, 6144, 7167, 7168, 8191]
STAT_KEYS = ("candidates", "stopped_sd", "fine_evals", "fine_pass", "ldpc_calls", "ldpc_iters", "osd_calls", "decoded",
             "emitted", "fine_rechecked")


def _report(name, d):
    print(f"[batch_sizes] {name}: {json.dumps(d)}")


def _engine(max_cycles):
    from pyft8_b200.engine import Engine
    return Engine(max_cycles=max_cycles)


def _free_device_cache():
    import torch
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def generate(config, B, seed):
    """int16 [B, 180000] torch tensor on cuda:0 holding bench.py's workload, made on a handle of its own"""
    import torch
    params = workload.make_params(config, B, seed=seed)
    audio = torch.empty((B, 180000), dtype=torch.int16, device="cuda:0")
    gen = _engine(1)
    try:
        workload.device_cycles(gen, params, audio.data_ptr())
        gen.synchronize()
    finally:
        gen.close()
    return audio


def decode_slices(audio, B):
    """The reference: cycles [s0, s0 + 1000) one call each on a fresh max_cycles = 1000 handle, `cycle` shifted by s0.
    Returns (records, n[B], the work counters summed over the calls)."""
    eng = _engine(SLICE)
    recs, ns, st = [], [], dict.fromkeys(STAT_KEYS, 0)
    try:
        for s0 in range(0, B, SLICE):
            r, n = eng.decode_cycles_dev(audio.data_ptr() + s0 * CYCLE_BYTES, L.AUDIO_I16, min(SLICE, B - s0))
            r = r.copy()
            r["cycle"] += s0
            recs.append(r)
            ns.append(n.copy())
            s = eng.stats()
            for k in STAT_KEYS:
                st[k] += s[k]
    finally:
        eng.close()
    return np.concatenate(recs), np.concatenate(ns), st


def decode_whole(audio, B):
    """All B cycles in one device-resident call on a fresh max_cycles = B handle -> ((records, n, stats), device memory)"""
    import torch
    free0, total = torch.cuda.mem_get_info()
    eng = _engine(B)
    try:
        r, n = eng.decode_cycles_dev(audio.data_ptr(), L.AUDIO_I16, B)
        out = (r.copy(), n.copy(), eng.stats())
        free1, _ = torch.cuda.mem_get_info()
    finally:
        eng.close()
    return out, dict(device_total_gb=round(total / 1e9, 2), in_use_before_handle_gb=round((total - free0) / 1e9, 2),
                     in_use_after_decode_gb=round((total - free1) / 1e9, 2))


def assert_same_records(got, want, what):
    """n equal per cycle, records byte-identical (NaN fine_sd included) and cycle-major and contiguous"""
    (rec, n), (wrec, wn) = got, want
    assert len(n) == len(wn), what
    assert np.array_equal(n, wn), (what, "n differs in cycles", np.flatnonzero(n != wn)[:8].tolist())
    assert len(rec) == len(wrec) == int(wn.sum()), (what, len(rec), len(wrec))
    bad = np.flatnonzero(np.any(rec.view(np.uint8).reshape(-1, 64) != wrec.view(np.uint8).reshape(-1, 64), axis=1))
    assert not len(bad), (what, f"{len(bad)} records differ, in cycles", np.unique(wrec["cycle"][bad])[:8].tolist())
    assert np.array_equal(np.bincount(rec["cycle"], minlength=len(n)), n), what


def assert_same_stats(st, want, B, what):
    assert {k: st[k] for k in STAT_KEYS} == want, (what, st, want)
    assert st["cycles"] == B, (what, st)


def emitted_per_cycle(rec, B):
    return np.bincount(rec["cycle"], weights=rec["emitted"], minlength=B)


def oracle_deviations(rec, n, cycles, ref):
    """Emitted records of the sampled cycles against ft8_oracle.decode_cycle (ref[i] for cycles[i], as _oracle_cycle
    returns it): payload-set differences, order, notes and dt/df/SNR out of tolerance, each listed by cycle."""
    from pyft8_b200.engine import bits91_to_int
    from pyft8_b200.receiver import record_to_message
    off = np.concatenate([[0], np.cumsum(n)])
    d = dict(set_diff=[], order=[], notes=[], tol=[], dup=[], oracle_decodes=0, gpu_decodes=0)
    for b, want in zip(cycles, ref):
        r = rec[off[b]:off[b + 1]]
        em = r[r["emitted"] == 1]
        got = [bits91_to_int(x["bits91"]) >> 14 for x in em]
        d["oracle_decodes"] += len(want)
        d["gpu_decodes"] += len(got)
        if len(got) != len(set(got)):
            d["dup"].append(b)
        diff = set(got) ^ {w[0] for w in want}
        if diff:
            d["set_diff"].append((b, sorted("%x" % v for v in diff)))
        elif got != [w[0] for w in want]:
            d["order"].append(b)
        wmap = {w[0]: w for w in want}
        for x, g in zip(em, got):
            if g in wmap:
                m = record_to_message(x)
                if m["decode_notes"] != wmap[g][1]:
                    d["notes"].append((b, "%x" % g, m["decode_notes"], wmap[g][1]))
                # dt +-5 ms, df +-0.5 Hz, SNR +-1 dB
                if abs(m["tsec"] - wmap[g][2]) > 0.005 + 1e-9 or abs(m["fHz"] - wmap[g][3]) > 0.5 + 1e-9 \
                        or abs(int(m["their_snr"]) - wmap[g][4]) > 1:
                    d["tol"].append((b, "%x" % g))
    return d


def assert_oracle_bars(dev, n_cycles, what):
    assert dev["oracle_decodes"] > 5 * n_cycles, (what, dev)          # the sampled cycles really decode
    assert not dev["dup"] and not dev["set_diff"] and not dev["tol"], (what, dev)
    # an fp32 near-tie between the CUDA FFTs and numpy's can swap two emissions or the pass that decodes a message
    # (test_gpu_large.py): counted and bounded
    assert len(dev["order"]) <= 1 and len(dev["notes"]) <= 1, (what, dev)


@pytest.fixture(scope="module")
def pool():
    with mp.get_context("spawn").Pool(os.cpu_count() or 1) as p:
        yield p


# ------------------------------------------------------------------------------------------------ cfg2, 4096 cycles
@pytest.fixture(scope="module")
def cfg2():
    """bench.py's headline batch: its audio in page-locked host memory (as bench.py streams it), the 1000-cycle slices and
    the whole batch in one device-resident call.  The device audio and both handles are gone when this returns."""
    import torch
    from pyft8_b200.engine import PinnedArray
    config, B, seed = CFG2
    audio = generate(config, B, seed)
    slices = decode_slices(audio, B)
    whole, mem = decode_whole(audio, B)
    pinned = PinnedArray((B, 180000), np.int16)
    torch.from_numpy(pinned.array).copy_(audio)
    del audio
    _free_device_cache()
    yield dict(pinned=pinned, host=pinned.array, slices=slices, whole=whole, mem=mem)
    pinned.close()


def test_cfg2_4096_device_resident_equals_1000_cycle_slices(cfg2):
    """The headline call (4096 cycles: four F1 scratch chunks, four scan blocks) against five reference calls (1000, 1000,
    1000, 1000, 96 cycles): every record byte, n per cycle and the work counters; cycles >= 1024 decode like the others."""
    B = CFG2[1]
    (rec, n, st), (wrec, wn, wst) = cfg2["whole"], cfg2["slices"]
    assert_same_records((rec, n), (wrec, wn), "cfg2 4096 vs slices of 1000")
    assert_same_stats(st, wst, B, "cfg2 4096 vs slices of 1000")
    em = emitted_per_cycle(rec, B)
    lo, hi = float(em[:1024].mean()), float(em[1024:].mean())
    _report("cfg2_4096_device", dict(cycles=B, records=len(rec), emitted_per_cycle_below_1024=lo,
                                     emitted_per_cycle_from_1024=hi, device_memory=cfg2["mem"]))
    # a cycle decoded from another cycle's spectrum keeps its grid decodes (passes 0, 1) but loses most fine-stage ones
    assert lo > 10 and abs(hi - lo) <= 0.05 * lo, (lo, hi)


def test_cfg2_boundary_cycles_vs_oracle(cfg2, pool):
    """14 cycles on both sides of the 256-cycle copy chunks, the 1000-cycle slices and the 1024-cycle scratch chunks and scan
    blocks, against the oracle; the 1000-cycle slices deviate from it exactly as the 4096-cycle call does."""
    ref = pool.map(_oracle_cycle, [cfg2["host"][b] for b in ORACLE_CFG2], chunksize=1)
    dev = oracle_deviations(*cfg2["whole"][:2], ORACLE_CFG2, ref)
    _report("cfg2_oracle", dict(cycles=ORACLE_CFG2, **dev))
    assert dev == oracle_deviations(*cfg2["slices"][:2], ORACLE_CFG2, ref)
    assert_oracle_bars(dev, len(ORACLE_CFG2), "cfg2")


def test_cfg2_host_audio_in_16_copy_chunks(cfg2):
    """decode_cycles(pinned host audio): 16 copy chunks of 256 cycles, each with its own front end"""
    B = CFG2[1]
    eng = _engine(B)
    try:
        rec, n = eng.decode_cycles(cfg2["host"])
        got, st = (rec.copy(), n.copy()), eng.stats()
    finally:
        eng.close()
    assert_same_records(got, cfg2["whole"][:2], "cfg2 host, 16 chunks")
    assert_same_stats(st, {k: cfg2["whole"][2][k] for k in STAT_KEYS}, B, "cfg2 host, 16 chunks")


def test_cfg2_host_streaming_pair(cfg2):
    """bench.py's end-to-end pair: decode_cycles(host, next_audio=host) queues the prefetch, and decode_cycles(host)
    consumes it (one device-resident front end of 4096 cycles); both calls give the device-resident records."""
    B = CFG2[1]
    host = cfg2["host"]
    eng = _engine(B)
    try:
        r1, n1 = eng.decode_cycles(host, next_audio=host)
        first = (r1.copy(), n1.copy())
        assert eng._pf_ref is not None and eng._pf_ref.ctypes.data == host.ctypes.data      # the next call consumes the copy
        r2, n2 = eng.decode_cycles(host)
        second, st = (r2.copy(), n2.copy()), eng.stats()
    finally:
        eng.close()
    assert_same_records(first, cfg2["whole"][:2], "cfg2 stream, first call")
    assert_same_records(second, cfg2["whole"][:2], "cfg2 stream, prefetched call")
    assert_same_stats(st, {k: cfg2["whole"][2][k] for k in STAT_KEYS}, B, "cfg2 stream, prefetched call")


def test_cfg2_host_3001_cycles_short_last_chunk(cfg2):
    """B = 3001 host cycles: 12 copy chunks, eleven of 251 and a last one of 240; equal to cycles 0..3000 of the batch"""
    B = 3001
    eng = _engine(B)
    try:
        rec, n = eng.decode_cycles(cfg2["host"][:B])
        got = (rec.copy(), n.copy())
    finally:
        eng.close()
    wrec, wn = cfg2["whole"][:2]
    assert_same_records(got, (wrec[:int(wn[:B].sum())], wn[:B]), "cfg2 host, 3001 cycles")


def test_cfg2_record_capacity_cut_past_first_scan_block(cfg2):
    """ft8_decode_cycles of the device-resident batch with rec_capacity = records of cycles < 1500, plus 3: FT8_E_CAPACITY,
    the counts trimmed cycle-major (cycle 1500 keeps 3), the records a prefix of the whole batch's, every cycle counted."""
    import torch
    from pyft8_b200.engine import _ptr
    B = CFG2[1]
    wrec, wn, wst = cfg2["whole"]
    assert wn[1500] > 3
    cap = int(wn[:1500].sum()) + 3
    audio = torch.from_numpy(cfg2["host"]).to("cuda:0")
    rec = np.zeros(cap, L.RECORD_DTYPE)
    n = np.zeros(B, np.int32)
    eng = _engine(B)
    try:
        rc = eng._lib.ft8_decode_cycles(eng._h, C.c_void_p(audio.data_ptr()), L.AUDIO_I16, B, 0, _ptr(rec), cap, _ptr(n),
                                        L.MEM_DEVICE)
        err, st = eng._lib.last_error(), eng.stats()
    finally:
        eng.close()
        del audio
        _free_device_cache()
    assert rc == L.E_CAPACITY and "rec_capacity too small" in err, (rc, err)
    want_n = np.concatenate([wn[:1500], [3], np.zeros(B - 1501, np.int32)])
    assert np.array_equal(n, want_n), np.flatnonzero(n != want_n)[:8].tolist()
    assert rec.tobytes() == wrec[:cap].tobytes()
    assert st["cycles"] == B and st["decoded"] == len(wrec) == wst["decoded"], st


# ------------------------------------------------------------------------------------------------ cfg4, 8192 cycles
def test_cfg4_8192_device_resident_equals_slices_and_oracle(pool):
    """bench.py's configs[3] (8192 cycles x 120 signals: eight scratch chunks and scan blocks) in one device-resident call
    against nine reference calls of up to 1000 cycles, then eleven cycles at the 1024-cycle boundaries against the oracle.
    The cfg2 fixture has closed its handles and freed its device audio before this runs."""
    config, B, seed = CFG4
    audio = generate(config, B, seed)
    try:
        wrec, wn, wst = decode_slices(audio, B)
        (rec, n, st), mem = decode_whole(audio, B)
        sample = audio[ORACLE_CFG4].cpu().numpy()
    finally:
        del audio
        _free_device_cache()
    assert_same_records((rec, n), (wrec, wn), "cfg4 8192 vs slices of 1000")
    assert_same_stats(st, wst, B, "cfg4 8192 vs slices of 1000")
    em = emitted_per_cycle(rec, B)
    lo, hi = float(em[:1024].mean()), float(em[1024:].mean())
    ref = pool.map(_oracle_cycle, list(sample), chunksize=1)
    dev = oracle_deviations(rec, n, ORACLE_CFG4, ref)
    _report("cfg4_8192_device", dict(cycles=B, records=len(rec), emitted_per_cycle_below_1024=lo,
                                     emitted_per_cycle_from_1024=hi, device_memory=mem))
    _report("cfg4_oracle", dict(cycles=ORACLE_CFG4, **dev))
    assert lo > 20 and abs(hi - lo) <= 0.05 * lo, (lo, hi)
    assert dev == oracle_deviations(wrec, wn, ORACLE_CFG4, ref)
    assert_oracle_bars(dev, len(ORACLE_CFG4), "cfg4")


# ------------------------------------------------------------------------------------------------ consecutive live cycles
LIVE_STREAMS, LIVE_STEPS = 512, 3


@pytest.fixture(scope="module")
def live_1536():
    """1536 distinct cfg1 cycles as 3 steps x 512 streams (step c, stream b = cycle 512 c + b), and the reference: three
    decode_cycles_live calls of 512 streams on a fresh handle"""
    audio = generate("cfg1_20sig", LIVE_STEPS * LIVE_STREAMS, 2001)
    x = audio.cpu().numpy().reshape(LIVE_STEPS, LIVE_STREAMS, 180000)
    del audio
    _free_device_cache()
    eng = _engine(LIVE_STREAMS)
    try:
        want = live_calls(eng, x, 0)
    finally:
        eng.close()
    return x, want


@pytest.mark.parametrize("mem", ["host", "device"])
def test_live_seq_one_piece_of_1536_cycles(live_1536, mem):
    """decode_cycles_live_seq of 3 x 512 on a max_cycles = 1536 handle is one piece of 1536 cycles (two scan blocks; device
    audio also takes two F1 scratch chunks, host audio six copy chunks of 256): bit-identical with the three live calls."""
    x, want = live_1536
    eng = _engine(LIVE_STEPS * LIVE_STREAMS)
    try:
        got = seq_call(eng, x, 0) if mem == "host" else seq_device(eng, x, 0)
        st = eng.stats()
    finally:
        eng.close()
        _free_device_cache()
    assert_equal_runs(got, want, mem)
    assert st["cycles"] == LIVE_STEPS * LIVE_STREAMS and st["decoded"] == len(want[0]), st
    assert got[1][2].sum() > 5 * LIVE_STREAMS                 # the last step, whose cycles sit in the second scan block


# ------------------------------------------------------------------------------------------------ stand-alone F1
@pytest.mark.parametrize("dtype", ["int16", "float32"])
def test_cycle_spectrum_across_scratch_chunks(dtype):
    """ft8_cycle_spectrum of 1030 cycles (scratch chunks of 1024 and 6) tiled from 7 distinct ones, so that cycle 1024 + j
    and cycle j hold different audio: every cycle bit-identical to a B = 7 call, and cycles 0, 1023, 1024, 1029 within 2e-6
    of the largest magnitude of a float64 rfft.  float32 audio (int16 / 7, not integers) checks the 4-byte chunk offsets."""
    import torch
    B, P = 1030, 7
    small = _engine(8)
    try:
        a = torch.empty((P, 180000), dtype=torch.int16, device="cuda:0")
        workload.device_cycles(small, workload.make_params("cfg2_50sig", P, seed=2002), a.data_ptr())
        small.synchronize()
        base = a.cpu().numpy()
        del a
        if dtype == "float32":
            base = (base / 7.0).astype(np.float32)
        want = small.cycle_spectrum(base)
    finally:
        small.close()
    tile = np.arange(B) % P
    eng = _engine(B)
    try:
        spec = eng.cycle_spectrum(base[tile])
    finally:
        eng.close()
        _free_device_cache()
    assert spec.shape == (B, L.SPEC_BINS)
    err = {}
    for b in (0, 1023, 1024, 1029):
        x = np.zeros(192000)
        x[:180000] = base[tile[b]]
        ref = np.fft.rfft(x)
        err[b] = float(np.abs(spec[b] - ref).max() / np.abs(ref).max())
    bits, wbits = spec.view(np.uint64), want.view(np.uint64)
    differ = [b for b in range(B) if not np.array_equal(bits[b], wbits[tile[b]])]
    _report(f"cycle_spectrum_{dtype}", dict(cycles=B, max_err_rel_to_max=err, cycles_differing_from_b7=differ[:8]))
    assert not differ, (len(differ), differ[:8])
    assert all(e <= 2e-6 for e in err.values()), err
