"""Throughput of consecutive live cycles: for B streams x C cycles, cycles/s of
  (1) C sequential decode_cycles_live calls of B streams (ft8_decode_cycles_live),
  (2) one decode_cycles_live_seq call (ft8_decode_cycles_live_seq),
  (3) one isolated decode_cycles call on the same B*C cycles (ft8_decode_cycles),
and a check that (1) and (2) give identical records.

Audio is device-resident, made by the library's generator (ft8_synth_cycles) with bench.py's workload (cfg2_50sig: 50
signals per cycle), so no host copy is timed.  Its cycles are independent rather than continuous; the decode does the same
work either way.  Every mode runs once at the timed shape before it is timed; times are CUDA events on the handle's stream
around work that ends in a synchronise, the best of --reps runs.  The per-stage times (ft8_last_kernel_ms 1-8: spectrogram,
sync, cycle spectrum, pass 0, fine, passes 2-4, OSD, records) are those of the last timed run of (2) and (3).  One handle of max_cycles = max(B*C) serves all modes, so
(2) runs as one piece.  Prints the card's name and power limit with the numbers.

    python tools/live_seq_bench.py [--shapes 1x4096,64x64] [--reps 3] [--json out.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        return out or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown (nvidia-smi unavailable)"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--shapes", default="1x4096,64x64", help="comma-separated BxC (streams x consecutive cycles)")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--json", default=None, help="also write the results here")
    args = ap.parse_args()
    shapes = [tuple(int(v) for v in s.split("x")) for s in args.shapes.split(",")]

    import torch
    from pyft8_b200 import _lib as L, workload
    from pyft8_b200.engine import Engine, _ptr
    if not torch.cuda.is_available():
        raise SystemExit("live_seq_bench: no CUDA device")
    n_max = max(B * Cn for B, Cn in shapes)
    eng = Engine(max_cycles=n_max)
    lib, h, K = eng._lib, eng._h, eng.max_cands
    stream = torch.cuda.ExternalStream(lib.ft8_stream(h))
    esz = 180000 * 2

    def timed(fn, before=None):
        best = None
        for _ in range(args.reps):
            if before:
                before()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = ms if best is None else min(best, ms)
        return best

    rows = []
    for B, Cn in shapes:
        N = B * Cn
        params = workload.make_params("cfg2_50sig", N, seed=args.seed)
        audio = torch.empty((Cn, B, 180000), dtype=torch.int16, device="cuda:0")
        workload.device_cycles(eng, params, audio.data_ptr())
        torch.cuda.synchronize()
        base = audio.data_ptr()
        rec_all = np.zeros(N * K, L.RECORD_DTYPE)
        n_all = np.zeros(N, np.int32)
        rec_step = [np.zeros(B * K, L.RECORD_DTYPE) for _ in range(Cn)]
        n_step = np.zeros((Cn, B), np.int32)

        def sequential():
            for c in range(Cn):
                eng._check(lib.ft8_decode_cycles_live(h, C.c_void_p(base + c * B * esz), L.AUDIO_I16, B, c & 1, _ptr(rec_step[c]),
                                                      B * K, _ptr(n_step[c]), L.MEM_DEVICE))

        def seq():
            eng._check(lib.ft8_decode_cycles_live_seq(h, C.c_void_p(base), L.AUDIO_I16, B, Cn, 0, _ptr(rec_all), len(rec_all),
                                                      _ptr(n_all), L.MEM_DEVICE))

        def isolated():
            eng._check(lib.ft8_decode_cycles(h, C.c_void_p(base), L.AUDIO_I16, N, 0, _ptr(rec_all), len(rec_all), _ptr(n_all),
                                             L.MEM_DEVICE))

        # warm-up at the timed shape, and the equality of (1) and (2); both start from a fresh live state
        eng.live_reset()
        sequential()
        want = []
        for c in range(Cn):
            r = rec_step[c][:int(n_step[c].sum())].copy()
            r["cycle"] += c * B
            want.append(r)
        want = np.concatenate(want)
        want_n = n_step.copy()
        eng.live_reset()
        seq()
        got = rec_all[:int(n_all.sum())]
        assert np.array_equal(n_all.reshape(Cn, B), want_n), f"{B}x{Cn}: per-cycle counts differ"
        assert got.tobytes() == want.tobytes(), f"{B}x{Cn}: records differ"
        isolated()

        t_seqn = timed(sequential, eng.live_reset)
        t_seq = timed(seq, eng.live_reset)
        seq_stats, seq_ms = eng.stats(), eng.last_kernel_ms(0)
        seq_stages = [round(eng.last_kernel_ms(i), 3) for i in range(1, 9)]
        t_iso = timed(isolated)
        iso_stages = [round(eng.last_kernel_ms(i), 3) for i in range(1, 9)]
        row = dict(B=B, C=Cn, cycles=N, records=len(want),
                   sequential_live_cps=round(N / t_seqn * 1e3, 1), live_seq_cps=round(N / t_seq * 1e3, 1),
                   isolated_cps=round(N / t_iso * 1e3, 1), live_seq_vs_isolated=round(t_iso / t_seq, 3),
                   live_seq_vs_sequential=round(t_seqn / t_seq, 2), live_seq_launches=int(seq_stats["kernel_launches"]),
                   live_seq_library_ms=round(seq_ms, 2), stage_ms_live_seq=seq_stages, stage_ms_isolated=iso_stages)
        rows.append(row)
        print(f"[live_seq] B={B} C={Cn}: sequential live {row['sequential_live_cps']:.0f} cycles/s, live_seq "
              f"{row['live_seq_cps']:.0f}, isolated {row['isolated_cps']:.0f} (live_seq/isolated {row['live_seq_vs_isolated']:.3f}, "
              f"live_seq/sequential {row['live_seq_vs_sequential']:.1f}x); records identical ({len(want)})", flush=True)
        del audio
        torch.cuda.empty_cache()
    eng.close()
    out = dict(card=card(), workload="cfg2_50sig", reps=args.reps, results=rows)
    print(json.dumps(out))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
