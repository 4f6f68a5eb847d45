"""Cost of progressive live decoding (ft8_decode_cycles_live_progress) against the end-of-cycle live decode.

For R streams, two consecutive cycles each (device-resident audio from the library's generator with bench.py's cfg2_50sig
workload: 50 signals per cycle), the progressive schedule a receiver bank runs with progress_hops = 1: one rows-only call
for hops 1..S-1, then one call per hop S..375.  Reported per R, for the second cycle (the first warms up every shape and
leaves a full ring and previous cycle behind): the time of each call (median, max, and which hop the max was at; host
clock around the call, which ends in a synchronise), the sum over the cycle, one ft8_decode_cycles_live call of the same R
cycles on the same ring state, and the messages released per hop.  The bar: at R = 1024 every one-hop call under the
40 ms hop period.  Prints the card's name and power limit with the numbers.

    python tools/progressive_bench.py [--streams 64,1024,4096] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

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
    ap.add_argument("--streams", default="64,1024,4096")
    ap.add_argument("--json", default=None)
    args = ap.parse_args()
    import torch
    from pyft8_b200 import _lib as L
    from pyft8_b200 import workload
    from pyft8_b200.engine import Engine
    print("card:", card(), flush=True)
    results = []
    for R in [int(x) for x in args.streams.split(",")]:
        eng = Engine(max_cycles=R)
        S = eng.search_hop
        audio = torch.empty((2, R, 180000), dtype=torch.int16, device="cuda")
        for c in range(2):
            workload.device_cycles(eng, workload.make_params("cfg2_50sig", R, 9000 + c), audio[c].data_ptr())
        torch.cuda.synchronize()
        rec = np.zeros(R * eng.max_cands, L.RECORD_DTYPE)
        n = np.zeros(R, np.int32)
        eh = np.zeros(len(rec), np.uint16)
        schedule = [S - 1] + list(range(S, 376))

        def progressive(c):
            times, released = [], {}
            for hop in schedule:
                t = time.perf_counter()
                r, _, e = eng.decode_cycles_live_progress_dev(audio[c].data_ptr(), L.AUDIO_I16, R, c & 1, hop, rec, n, eh)
                times.append((time.perf_counter() - t) * 1e3)
                for x in e[r["emitted"] == 1].tolist():
                    released[x] = released.get(x, 0) + 1
            return times, released

        progressive(0)                                   # warm-up: every shape, and a full ring + previous cycle
        eng.synchronize()
        times, released = progressive(1)
        # the end-of-cycle live decode of the same cycle on the same ring state (cycle 0 decoded live again first)
        eng.live_reset()
        eng._check(eng._lib.ft8_decode_cycles_live(eng._h, audio[0].data_ptr(), L.AUDIO_I16, R, 0, rec.ctypes.data, len(rec),
                                                   n.ctypes.data, L.MEM_DEVICE))
        eng.synchronize()
        t = time.perf_counter()
        eng._check(eng._lib.ft8_decode_cycles_live(eng._h, audio[1].data_ptr(), L.AUDIO_I16, R, 1, rec.ctypes.data, len(rec),
                                                   n.ctypes.data, L.MEM_DEVICE))
        live_ms = (time.perf_counter() - t) * 1e3
        live_emitted = eng.stats()["emitted"]
        one_hop = times[1:]
        worst = int(np.argmax(one_hop))
        res = dict(streams=R, search_hop=S, rows_call_ms=round(times[0], 3), call_ms_median=round(float(np.median(one_hop)), 3),
                   call_ms_max=round(float(max(one_hop)), 3), call_max_at_hop=schedule[1 + worst],
                   cycle_sum_ms=round(float(sum(times)), 2), live_call_ms=round(live_ms, 2),
                   released=sum(released.values()), live_emitted=int(live_emitted),
                   released_per_hop={int(k): v for k, v in sorted(released.items())})
        print(json.dumps({k: v for k, v in res.items() if k != "released_per_hop"}), flush=True)
        hops = sorted(released)
        print("  released per hop (hop:count):", " ".join(f"{h}:{released[h]}" for h in hops), flush=True)
        results.append(res)
        del audio
        eng.close()
        torch.cuda.empty_cache()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(card=card(), results=results), f, indent=1)


if __name__ == "__main__":
    main()
