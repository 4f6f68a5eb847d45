#!/usr/bin/env python
"""bench.py -- decoded 15-s FT8 cycles/s of the receive hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one process per GPU under torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  the reference's own CPU implementation on the host cores

A step = one pass of the whole path (audio -> records) over one batch of synthetic cycles (BASELINE configs[1]:
4096 cycles x 50 GFSK signals, SNR -24..+10 dB, 200-2950 Hz).  `value` is timed with the batch resident in HBM;
`e2e` is the same through Engine.decode_cycles with pinned HOST buffers (H2D of the audio and D2H of the records inside
the timed region; at N > 1 the host-side gather of every rank's records on rank 0 as well).  Prints ONE JSON line on
rank 0.  The default N = 1 run also measures BASELINE configs[2] (LDPC/OSD codewords/s) and configs[3] (dense band) in
the same process, outside the headline timed region (`configs`).

Roofline block: nothing is typed in here.  Algorithmic bytes are SURVEY 8d's (ALG_BYTES below, derivation in DESIGN.md
section 4); the ncu-derived quantities (DRAM traffic, pipe utilisation per kernel) are loaded from
profiles/ncu_current.json (tools/ncu_extract.py output, tagged with the commit it was captured at and printed as
`ncu_capture_commit`); on-chip peaks come from profiles/peaks_b200.json (tools/micro/peaks.cu run on the box) and the HBM
peak from MEASURED_PEAKS.json.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "decoded 15-s FT8 cycles/sec"
UNIT = "cycles/s"
WORKLOAD = "cfg2_50sig"          # BASELINE configs[1]; --workload selects configs[0] / configs[3] shapes for extra data points
REF_DIR = os.path.join(ROOT, "oracle", "_ref")     # unmodified reference, pip-installed by __graft_entry__.build()
# algorithmic bytes per unit (SURVEY.md 8d; DESIGN.md section 4); int16 audio in
ALG_BYTES = {
    "spectrogram": 360000 + 375 * 976 * 4,          # per cycle: audio once + grid once
    "sync": 375 * 976 * 4 + 200 * (16 + 58 * 8 * 4),  # per cycle: grid once + candidates/payloads
    "cycle_spectrum": 360000 + 47415 * 8,           # per cycle: audio once + the bins the fine stage reads
    "pass0_ldpc5": 58 * 8 * 4 + 696 + 24,           # per candidate
    "fine_tscan": 8000 + 224 * 8,                   # per candidate: the 1000-bin band once + the 224 samples it hands on
    "fine_fscan_mma": 328 * 8 + 224 * 8,            # per candidate: the 328 edge bins + the 224 samples
    "fine_final": 8000 + 174 * 4,                   # per candidate: the band once more + the LLRs
    "pass234_ldpc": 696 + 696 + 24,                 # per LDPC call
    "osd": 696 + 64,                                # per OSD call
}
# index = `which` of ft8_last_kernel_ms; "fine" (5) is the sum of the three kernels 9..11, listed separately in roofline_stages
STAGES = ["all", "spectrogram", "sync", "cycle_spectrum", "pass0_ldpc5", "fine", "pass234_ldpc", "osd", "collect",
          "fine_tscan", "fine_fscan_mma", "fine_final"]
# kernels of each stage (names as tools/ncu_extract.py shortens them) and the work unit its per-unit figures refer to
STAGE_KERNELS = {"spectrogram": ["k_spectrogram"], "sync": ["k_sync_scores", "k_topk"], "cycle_spectrum": ["k_cs_cols", "k_cs_rows"],
                 "pass0_ldpc5": ["k_pass0"], "fine_tscan": ["k_fine_tscan"], "fine_fscan_mma": ["k_fscan_mma"], "fine_final": ["k_fine_final"],
                 "pass234_ldpc": ["k_pass234"], "osd": ["k_osd_items", "k_osd_resolve"]}
STAGE_UNIT = {"spectrogram": "cycles", "sync": "cycles", "cycle_spectrum": "cycles", "pass0_ldpc5": "candidates", "fine_tscan": "fine_evals",
              "fine_fscan_mma": "fine_evals", "fine_final": "fine_evals",
              "pass234_ldpc": "ldpc_calls", "osd": "osd_calls"}
# what bounds a stage when the committed capture has no counters for its kernels (stated, frac left null -- never "hbm")
DECLARED_BOUND = {"pass0_ldpc5": "issue", "fine_tscan": "l1_data_pipe", "fine_fscan_mma": "tensor", "fine_final": "l1_data_pipe",
                  "pass234_ldpc": "issue", "osd": "int_alu"}
HBM_STAGES = ("spectrogram", "sync", "cycle_spectrum")          # the stages the north star holds against the HBM roofline
# on-chip roofs: name -> (ncu utilisation key in the capture, peak key in profiles/peaks_b200.json, unit)
ONCHIP = {"l1_data_pipe": ("l1_data_pipe_pct", "l1_wavefronts_per_s_lds64", "wavefronts/s"),
          "fp32": ("fma_pipe_pct", "fma_warp_inst_per_s", "warp-inst/s"),
          "int_alu": ("alu_pipe_pct", "int_alu_warp_inst_per_s", "warp-inst/s"),
          "issue": ("issue_active_pct", "issue_warp_inst_per_s_peak", "warp-inst/s"),
          "tensor": ("tensor_pipe_pct", "tf32_dense_tflops", "TFLOP/s")}


def _load_json(path):
    try:
        return json.load(open(path))
    except Exception:
        return None


def _peaks():
    p = _load_json(os.path.join(ROOT, "MEASURED_PEAKS.json"))
    if p and "hbm_gbs" in p:
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def roofline_block(stage_ms, units, cycles):
    """Per-stage roofline entries from live CUDA-event times + the committed capture / peak files (see module docstring)."""
    hbm_peak, hbm_src = _peaks()
    cap = _load_json(os.path.join(ROOT, "profiles", "ncu_current.json")) or {}
    onchip_peaks = _load_json(os.path.join(ROOT, "profiles", "peaks_b200.json")) or {}
    kern = cap.get("kernels", {})
    cap_units = dict(cap.get("work_per_step") or {})
    cap_units["cycles"] = cap.get("cycles_per_launch")
    stages = []
    for i, name in enumerate(STAGES):
        if name not in ALG_BYTES:
            continue
        ms = float(stage_ms[i])
        n_units = units[STAGE_UNIT[name]]
        ent = {"kernel": name, "ms": round(ms, 4), "share": round(ms / float(stage_ms[0]), 4) if stage_ms[0] > 0 else None,
               "unit_of_work": STAGE_UNIT[name], "units": int(n_units)}
        ks = [k for k in STAGE_KERNELS[name] if k in kern]
        # per-step totals of the captured kernels of this stage (average launch x launches per step)
        t_cap = sum(kern[k]["time_ms"] * kern[k].get("launches_per_step", 1) for k in ks)
        cu = cap_units.get(STAGE_UNIT[name])
        scale = (n_units / cu) if (cu and ks) else None            # live units / captured units
        traffic = int(sum(kern[k]["dram_bytes"] * kern[k].get("launches_per_step", 1) for k in ks) * scale) if scale else None
        util = {}
        for roof, (key, _, _) in ONCHIP.items():
            if ks and t_cap > 0 and all(key in kern[k] for k in ks):
                util[roof] = sum(kern[k][key] * kern[k]["time_ms"] * kern[k].get("launches_per_step", 1) for k in ks) / t_cap
        # the same pipe work per unit in the live time: utilisation scales with captured time per unit / live time per unit
        live = {r: u * (t_cap * scale / ms) for r, u in util.items()} if (scale and ms > 0) else {}
        alg = ALG_BYTES[name] * n_units
        hbm_ach = alg / (ms / 1e3) / 1e9 if ms > 0 else 0.0
        onchip_best = max(live, key=live.get) if live else None
        if name not in HBM_STAGES and onchip_best is None:
            ent.update({"bound": DECLARED_BOUND[name], "achieved": None, "peak": None, "unit": ONCHIP[DECLARED_BOUND[name]][2], "frac": None,
                        "note": "no ncu counters for this stage in the committed capture"})
        elif name in HBM_STAGES:
            ent.update({"bound": "hbm", "achieved": round(hbm_ach, 2), "peak": hbm_peak, "unit": "GB/s", "frac": round(hbm_ach / hbm_peak, 5)})
        else:
            _, pkey, punit = ONCHIP[onchip_best]
            peak = onchip_peaks.get(pkey)
            frac = live[onchip_best] / 100.0
            ent.update({"bound": onchip_best, "achieved": (frac * peak) if peak else None, "peak": peak, "unit": punit, "frac": round(frac, 5)})
        if onchip_best is not None:
            _, pkey, punit = ONCHIP[onchip_best]
            ent["on_chip"] = {"bound": onchip_best, "frac": round(live[onchip_best] / 100.0, 5), "peak": onchip_peaks.get(pkey), "unit": punit}
        ent["hbm_frac"] = round(hbm_ach / hbm_peak, 5)
        ent["alg_bytes"] = int(alg)
        ent["traffic"] = traffic
        ent["ncu_pct_of_peak_at_capture"] = {k: round(v, 1) for k, v in util.items()} or None
        stages.append(ent)
    dom = max(stages, key=lambda s: s["ms"])
    roofline = {k: dom.get(k) for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic")}
    roofline.update({"hbm_peak_source": hbm_src, "ncu_capture": cap.get("capture"), "ncu_capture_commit": cap.get("commit"),
                     "onchip_peaks": "profiles/peaks_b200.json" if onchip_peaks else None,
                     "note": "dominant kernel by device time; per stage: bound = hbm for S1/S2/F1 (north star) with the on-chip roof "
                             "beside it, else the most utilised on-chip pipe of the committed ncu capture rescaled to the live time"})
    s12 = [s for s in stages if s["kernel"] in ("spectrogram", "sync")]
    s12_ms = sum(s["ms"] for s in s12)
    roofline["s1_s2"] = {"ms": round(s12_ms, 4), "alg_bytes": int(sum(s["alg_bytes"] for s in s12)),
                         "hbm_frac": round(sum(s["alg_bytes"] for s in s12) / (s12_ms / 1e3) / 1e9 / hbm_peak, 5) if s12_ms > 0 else None}
    return roofline, stages


DUMP_BUDGET = 64 << 20           # bytes --dump-outputs may write in all


def dump_outputs(out_dir, rec, counts, max_cands):
    """Write what one device-resident step returned: counts.npy (records per cycle) and rec_<field>.npy for every field of
    the records, float64 for the integer fields (exact) and float32 for the float ones.  Every value written is finite: fine_sd,
    NaN ("not computed") in records decoded before the fine stage (ipass < 2), is written as 0 there; rec_ipass tells those
    records apart.  When the records of the whole batch could exceed DUMP_BUDGET (max_cands records per cycle), only the
    records of a fixed seeded sample of cycles are written; cycles.npy lists the cycles written.  The sample depends on the
    batch size and max_cands alone, so two builds run with the same arguments write the same cycles."""
    fields = [f for f in rec.dtype.names if f != "reserved"]
    out_dtype = {f: np.float32 if rec.dtype[f].base.kind == "f" else np.float64 for f in fields}
    rec_bytes = sum(np.dtype(out_dtype[f]).itemsize * int(np.prod(rec.dtype[f].shape)) for f in fields)
    B = len(counts)
    k = min(B, (DUMP_BUDGET - 16 * B) // (max_cands * rec_bytes))
    cycles = np.arange(B) if k == B else np.sort(np.random.default_rng(0).choice(B, k, replace=False))
    sel = rec[np.isin(rec["cycle"], cycles)]
    sel["fine_sd"][sel["ipass"] < 2] = 0
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "counts.npy"), counts.astype(np.float64))
    np.save(os.path.join(out_dir, "cycles.npy"), cycles.astype(np.float64))
    for f in fields:
        np.save(os.path.join(out_dir, f"rec_{f}.npy"), sel[f].astype(out_dtype[f]))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def _dist_init():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # no data-path collective exists (cycles are independent); gloo carries the barrier, the max-over-ranks and the
        # host-side record gather
        dist_mod.init_process_group("gloo", rank=rank, world_size=world)
        dist = dist_mod
    return dist, rank, local, world


# ---------------------------------------------------------------------------------------------- CPU arms
def ref_available():
    return os.path.isdir(os.path.join(REF_DIR, "PyFT8"))


def _cpu_decode_one(a):
    """One cycle on one host core: the UNMODIFIED reference (oracle/_ref, driven through its own Receiver / AudioIn /
    Candidate API by oracle/ref_harness.py) when it travelled to this box, else the numpy port (oracle/ft8_oracle.py).
    Returns (texts of the emitted messages, n candidates, n ldpc calls | None, seconds)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    t = time.time()
    if ref_available():
        os.environ["PYFT8_REF_ROOT"] = REF_DIR
        import ref_harness as rh
        with tempfile.TemporaryDirectory() as d:
            out = rh.decode_cycle(a, workdir=d)
        return [" ".join(m["msg_tuple"]) for m in out["messages"]], out["n_cands"], None, time.time() - t
    import ft8_oracle as o
    recs, cl = o.decode_cycle(a)
    return [" ".join(o.unpack77(r["bits77"]) or ()) for r in recs], len(cl), sum(c.n_ldpc for c in cl), time.time() - t


_POOL = None


def _cpu_warm(_):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    if ref_available():
        os.environ["PYFT8_REF_ROOT"] = REF_DIR
        import ref_harness as rh
        rh.load_reference()
    else:
        import ft8_oracle  # noqa: F401
    return os.getpid()


def cpu_pool(cores):
    """Worker processes (one per host core) with the CPU implementation imported, so that timing excludes start-up."""
    global _POOL
    if _POOL is None:
        import multiprocessing as mp
        _POOL = mp.get_context("spawn").Pool(cores)
        _POOL.map(_cpu_warm, range(4 * cores), chunksize=1)
    return _POOL


def _host_cycle0(p):
    sys.path.insert(0, ROOT)
    from pyft8_b200 import workload
    p = dict(p)
    p["seed"] = (p["seed"] << 8) ^ int(p["pick"][0, 0]) ^ (int(p["pick"][0, 1]) << 10)     # distinct noise per cycle
    return workload.host_cycle(p, 0)


def cpu_rate(cycles, cores):
    """The CPU implementation on `cores` worker processes, one cycle at a time each: (cycles/s, ldpc calls/s | None, detail)."""
    pool = cpu_pool(cores)
    t = time.time()
    res = pool.map(_cpu_decode_one, list(cycles), chunksize=1)
    wall = time.time() - t
    ldpc = None if any(r[2] is None for r in res) else sum(r[2] for r in res) / wall
    return len(cycles) / wall, ldpc, dict(wall_s=wall, decodes=sum(len(r[0]) for r in res), texts=[r[0] for r in res],
                                          per_cycle_s=float(np.mean([r[3] for r in res])))


def cpu_kind():
    return ("reference", "unmodified G1OJS/PyFT8 v3.9.0 (oracle/_ref) through Receiver/AudioIn/Candidate, import stubs for "
            "pyaudio/paho + fake clock (oracle/ref_harness.py)") if ref_available() else ("port", "numpy port oracle/ft8_oracle.py")


def run_reference(args, dist, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on all host cores (one process per core),
    bounded sample of the same workload per step."""
    if rank != 0:
        return
    from pyft8_b200 import workload
    cores = os.cpu_count() or 1
    per_step = cores * args.ref_cycles_per_core
    n_cyc = per_step * (args.steps + args.warmup)
    params = workload.make_params(WORKLOAD, n_cyc, seed=args.seed)
    # the numpy modulator needs ~0.8 s per 50-signal cycle: build the inputs on the worker pool too (outside the timed region)
    small = [{k: (v[b:b + 1] if isinstance(v, np.ndarray) else v) for k, v in params.items() if k != "pool_bits77"} for b in range(n_cyc)]
    cyc = cpu_pool(cores).map(_host_cycle0, small, chunksize=1)
    for w in range(args.warmup):
        cpu_rate(cyc[w * per_step:(w + 1) * per_step], cores)
    t0 = time.time()
    ldpc, decodes = 0.0, 0
    for s in range(args.warmup, args.warmup + args.steps):
        r, l, det = cpu_rate(cyc[s * per_step:(s + 1) * per_step], cores)
        ldpc = None if (l is None or ldpc is None) else ldpc + l
        decodes += det["decodes"]
    wall = time.time() - t0
    value = per_step * args.steps / wall
    kind, how = cpu_kind()
    sample = f"{per_step} cycles per step ({args.ref_cycles_per_core} per core) of {WORKLOAD}, numpy-generated from the same parameters; {how}"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "cycles_per_step": per_step, "signals_per_cycle": workload.CONFIGS[WORKLOAD][0], "host": "cpu"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "decodes_per_cycle": decodes / (per_step * args.steps),
        "ldpc_codewords_per_sec": (ldpc / args.steps) if ldpc is not None else None,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


# ---------------------------------------------------------------------------------------------- extra BASELINE configs
def _oracle_ldpc(x):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ft8_oracle as o
    z = x.copy()
    st, n, _ = o.ldpc_decode(z, 90, 20)
    return st, n


def _oracle_osd(x):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ft8_oracle as o
    b = o.osd(x.copy())
    return b if b else 0


def config_cfg3_fec(device, n_total, check):
    """BASELINE configs[2]: noisy 174-bit LLR codewords at Eb/N0 0..4 dB through ft8_ldpc(., 90, 20), ft8_osd on the failures
    (decoders.py:153-171, 223-272).  Kernel times from the library's CUDA events; `check` vectors per point are re-decoded
    by the CPU oracle (decision-level identity)."""
    from pyft8_b200 import synth, _lib as L
    from pyft8_b200.engine import Engine, bits91_to_int
    eng = Engine(device=device, max_cycles=1)
    rng = np.random.default_rng(3)
    msgs = [synth.pack77(*synth.random_message(rng)) for _ in range(1024)]
    cws = np.array([synth.codeword_bits(b) for b in msgs], np.float32) * 2 - 1
    per = n_total // 5
    t_ldpc = t_osd = 0.0
    n_osd = mism = osd_mism = checked = osd_checked = 0
    bp_ok, fallback, rescued = [], [], []
    pool = cpu_pool(os.cpu_count() or 1) if check else None
    for e in range(5):
        idx = rng.integers(0, 1024, per)
        sigma = np.sqrt(1.0 / (2.0 * (91.0 / 174.0) * 10 ** (e / 10)))
        y = cws[idx] + rng.standard_normal((per, 174), np.float32) * np.float32(sigma)
        llr = (2.83 * y / y.std(axis=1, keepdims=True)).astype(np.float32)
        x = llr.copy()
        st, ni, bits = eng.ldpc(x, 90, 20)
        t_ldpc += eng.last_kernel_ms(0)
        ok = st == L.LDPC_OK
        fail = np.flatnonzero(~ok)
        if len(fail):
            found, ob = eng.osd(llr[fail])
            t_osd += eng.last_kernel_ms(0)
        else:
            found, ob = np.zeros(0, np.int32), np.zeros((0, 3), np.uint32)
        n_osd += len(fail)
        bp_ok.append(round(float(ok.mean()), 5))
        fallback.append(round(len(fail) / per, 5))
        rescued.append(round(float((found > 0).sum()) / max(len(fail), 1), 5))
        if check:
            ref = pool.map(_oracle_ldpc, [llr[i] for i in range(check)], chunksize=16)
            mism += sum((s_ != (st[i] if st[i] != L.LDPC_STALL else L.LDPC_FAIL)) or (n_ != ni[i]) for i, (s_, n_) in enumerate(ref))
            checked += check
            k = min(check // 8, len(fail))
            ref_o = pool.map(_oracle_osd, [llr[fail[j]] for j in range(k)], chunksize=2)
            osd_mism += sum((bits91_to_int(ob[j]) if found[j] else 0) != ref_o[j] for j in range(k))
            osd_checked += k
    eng.close()
    return {"config": "BASELINE configs[2]: noisy LLR codewords, Eb/N0 0..4 dB, ldpc_decode(.,90,20) then osd_012 on the failures",
            "codewords": 5 * per, "ldpc_codewords_per_sec": 5 * per / (t_ldpc / 1e3), "ldpc_kernel_ms": round(t_ldpc, 3),
            "osd_calls": int(n_osd), "osd_per_sec": n_osd / (t_osd / 1e3) if t_osd > 0 else None, "osd_kernel_ms": round(t_osd, 3),
            "bp_ok": bp_ok, "osd_fallback_rate": fallback, "osd_rescued": rescued,
            "oracle_checked": {"ldpc": checked, "osd": osd_checked}, "oracle_mismatch": int(mism + osd_mism),
            "timing": "device time of the LDPC / OSD kernels (CUDA events inside the library), codewords resident in HBM"}


def config_cycles(device, workload_name, B, steps, seed):
    """Another cycle-shaped BASELINE config (e.g. configs[3]: 8192 x 120 signals) measured like the headline: device-resident
    value and host-buffer e2e (streaming entry, every step's H2D and record D2H inside the timed region)."""
    import torch
    from pyft8_b200 import workload, _lib as L
    from pyft8_b200.engine import Engine
    eng = Engine(device=device, max_cycles=B)
    params = workload.make_params(workload_name, B, seed=seed)
    audio = torch.empty((B, 180000), dtype=torch.int16, device=f"cuda:{device}")
    workload.device_cycles(eng, params, audio.data_ptr())
    torch.cuda.synchronize()
    host = torch.empty((B, 180000), dtype=torch.int16, pin_memory=True)
    host.copy_(audio)
    host_np = host.numpy()
    rec_pin = torch.zeros((B * eng.max_cands, L.RECORD_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
    n_pin = torch.zeros(B, dtype=torch.int32).pin_memory()
    rec_np, n_np = rec_pin.numpy().view(L.RECORD_DTYPE).reshape(-1), n_pin.numpy()
    stream = torch.cuda.ExternalStream(L.load().ft8_stream(eng._h), device=f"cuda:{device}")
    for _ in range(2):
        eng.decode_cycles_dev(audio.data_ptr(), L.AUDIO_I16, B, rec=rec_np, n=n_np)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(steps):
        eng.decode_cycles_dev(audio.data_ptr(), L.AUDIO_I16, B, rec=rec_np, n=n_np)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    st = eng.stats()
    eng.decode_cycles(host_np, next_audio=host_np, rec=rec_np, n=n_np)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = None
    for i in range(steps):
        r, _ = eng.decode_cycles(host_np, next_audio=host_np if i + 1 < steps else None, rec=rec_np, n=n_np)
    torch.cuda.synchronize()
    ms_e2e = 1e3 * (time.perf_counter() - t0)
    out = {"config": f"{workload_name}: {B} cycles x {workload.CONFIGS[workload_name][0]} signals per step", "steps": steps,
           "cycles_per_sec": B * steps / (ms / 1e3), "ms_per_step": ms / steps,
           "e2e": {"value": B * steps / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": int(B * 360000),
                   "d2h_bytes_per_step": int(len(r) * 64 + 4 * B + 96)},
           "candidates_per_cycle": st["candidates"] / B, "at_max_cands": None, "decodes_per_cycle": st["decoded"] / B,
           "emitted_per_cycle": st["emitted"] / B, "ldpc_codewords_per_sec": st["ldpc_calls"] / (ms / steps / 1e3),
           "osd_calls_per_cycle": st["osd_calls"] / B}
    eng.close()
    del audio, host, rec_pin
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------- our arm
def run_gpu(args, dist, rank, local, world):
    import torch
    from pyft8_b200 import workload
    from pyft8_b200 import _lib as L
    from pyft8_b200.engine import Engine
    from pyft8_b200.sharding import ShmRecordGather
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the CUDA path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    B = args.cycles
    eng = Engine(device=local, max_cycles=B)
    params = workload.make_params(WORKLOAD, B, seed=args.seed + 7919 * rank)
    audio = torch.empty((B, 180000), dtype=torch.int16, device=f"cuda:{local}")
    workload.device_cycles(eng, params, audio.data_ptr())
    torch.cuda.synchronize()
    # the input staging buffer: page-locked memory from the library's allocator (ft8_host_alloc).  FT8_BENCH_HOSTMEM=wc asks
    # for write-combined memory instead (measured: no difference, 1 GPU 64.6 vs 65.1 k cycles/s, 8 GPUs 357.0 vs 357.6 k --
    # at 8 GPUs the copies of all ranks together run at the platform's 129 GB/s host-to-device ceiling either way)
    from pyft8_b200.engine import PinnedArray
    hostmem = os.environ.get("FT8_BENCH_HOSTMEM", "pinned")
    host_pin = PinnedArray((B, 180000), np.int16, write_combined=(hostmem == "wc"))
    host_np = host_pin.array
    torch.from_numpy(host_np).copy_(audio)
    stream = torch.cuda.ExternalStream(L.load().ft8_stream(eng._h), device=f"cuda:{local}")
    rec = np.zeros(B * eng.max_cands, L.RECORD_DTYPE)
    nrec = np.zeros(B, np.int32)

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()

    def max_over_ranks(x):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def sum_over_ranks(x):
        if not dist:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    # ---- device-resident timing
    for _ in range(args.warmup):
        eng.decode_cycles_dev(audio.data_ptr(), L.AUDIO_I16, B, rec=rec, n=nrec)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stage_ms = np.zeros(len(STAGES))
    launches = 0
    stats = None
    e0.record(stream)
    for _ in range(args.steps):
        r, n = eng.decode_cycles_dev(audio.data_ptr(), L.AUDIO_I16, B, rec=rec, n=nrec)
        stage_ms += [eng.last_kernel_ms(i) for i in range(len(STAGES))]
        stats = eng.stats()
        launches += stats["kernel_launches"]
    e1.record(stream)
    barrier()
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    n_decoded, n_emitted = stats["decoded"], stats["emitted"]
    dev_records = np.array(r, copy=True)                  # last device-resident step's records (parity spot check below)
    dev_counts = np.array(n, copy=True)
    total_cycles = sum_over_ranks(B)
    value = total_cycles * args.steps / (ms_dev / 1e3)
    stage_ms /= args.steps
    ldpc_rate = sum_over_ranks(stats["ldpc_calls"]) / (ms_dev / args.steps / 1e3)
    e2e_out = host_text = None
    if not args.device_only:
        # ---- end to end: pinned host audio in, records out, every step, through Engine.decode_cycles (C ABI, host buffers).
        # Batches are streamed the way a skimmer would: each call names the next batch (ft8_decode_cycles_stream), whose PCIe
        # copy then runs on a second CUDA stream underneath this batch's kernels.  Every step's H2D copy and record D2H are
        # inside the timed region, and so is -- at N > 1 -- the host-side gather of all ranks' records on rank 0
        # (sharding.ShmRecordGather: the path's only cross-GPU step).
        rec_pin = torch.zeros((B * eng.max_cands, L.RECORD_DTYPE.itemsize), dtype=torch.uint8).pin_memory()
        n_pin = torch.zeros(B, dtype=torch.int32).pin_memory()
        rec_np, n_np = rec_pin.numpy().view(L.RECORD_DTYPE).reshape(-1), n_pin.numpy()
        gathered = [0, 0]
        shm = ShmRecordGather(dist, B * eng.max_cands, L.RECORD_DTYPE, tag=os.environ.get("MASTER_PORT", "0")) if dist else None
        shm_pinned = shm.pin() if shm else None

        step_wall = []

        def e2e_steps(k):
            r_i = None
            del step_wall[:]
            # step 0 is not prefetched: its copy runs in chunks with the front-end kernels starting as chunks land (and is
            # inside the timed region like every other step's); from step 1 on the copy hides under the previous step
            for i in range(k):
                t_i = time.perf_counter()
                # N > 1: the records are copied back straight into this rank's shared-memory slot (pinned with cudaHostRegister)
                out = shm.slot_array() if shm else rec_np
                r_i, _ = eng.decode_cycles(host_np, next_audio=host_np if i + 1 < k else None, rec=out, n=n_np)
                if shm:
                    shm.publish_inplace(len(r_i), rank * B)
                    parts = shm.collect()                 # barrier; rank 0 now sees every rank's records of this step
                    if rank == 0:
                        gathered[0], gathered[1] = sum(len(p) for p in parts), sum(p.nbytes for p in parts)
                step_wall.append(1e3 * (time.perf_counter() - t_i))
            return r_i

        e2e_steps(min(args.warmup, 2))
        barrier()
        t0 = time.perf_counter()
        rec_last = e2e_steps(args.steps)
        barrier()
        ms_e2e = max_over_ranks(1e3 * (time.perf_counter() - t0))
        n_e2e_decoded = len(rec_last)
        e2e = total_cycles * args.steps / (ms_e2e / 1e3)
        e2e_out = {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(B * 360000), "d2h_bytes_per_step": int(n_e2e_decoded * 64 + 4 * B + 96),
                   "ms_per_step": ms_e2e / args.steps,
                   # the timed region starts cold: step 0's input copy cannot hide under a previous step (it runs in chunks
                   # with the front-end kernels); the steps after it are the steady state of a stream (rank 0's wall clock)
                   "first_step_ms": round(step_wall[0], 3) if step_wall else None,
                   "steady_state_ms_per_step": round(float(np.median(step_wall[1:])), 3) if len(step_wall) > 1 else None,
                   # all ranks' input copies together: at 8 GPUs this reaches the box's host-to-device ceiling (134 GB/s measured),
                   # which then bounds e2e (372 k cycles/s) below the kernels (563 k)
                   "h2d_gb_per_s_all_ranks": round(world * B * 360000 * args.steps / (ms_e2e / 1e3) / 1e9, 2),
                   "gather": {"records_on_rank0_per_step": gathered[0], "bytes_on_rank0_per_step": gathered[1], "segments_pinned": shm_pinned,
                              "how": "sharding.ShmRecordGather: per-rank shared-memory segments + one gloo barrier per step, inside the timed region"} if dist else None,
                   "host_memory": "write-combined page-locked (ft8_host_alloc)" if hostmem == "wc" else "page-locked (ft8_host_alloc)",
                   "api": "Engine.decode_cycles(pinned host int16, next_audio=...) -> ft8_decode_cycles_stream: one handle, next batch copied under the kernels"}
        # host text formatting of one step's records (outside every timed region; SURVEY 8f rank 2): vectorised unpack + de-dup
        from pyft8_b200.receiver import format_records
        format_records(rec_last[:1000])
        t0 = time.perf_counter()
        mb = format_records(rec_last)
        host_text = {"records_per_sec": len(rec_last) / max(time.perf_counter() - t0, 1e-9), "records": int(len(rec_last)),
                     "messages": int(len(mb)), "note": "format_records on one step's records, one host thread, not in any timed region"}
        del rec_pin
        if shm:
            shm.close()
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dev_records, dev_counts, eng.max_cands)
    units = {"cycles": B, "candidates": stats["candidates"], "fine_evals": stats["fine_evals"],
             "ldpc_calls": max(stats["ldpc_calls"], 1), "osd_calls": max(stats["osd_calls"], 1)}
    roofline, stages = roofline_block(stage_ms, units, B)
    cpu = None
    if world == 1 and not args.no_cpu_baseline and not args.device_only:
        cores = os.cpu_count() or 1
        n_s = cores * args.cpu_cycles_per_core
        sample = [host_np[i].copy() for i in range(n_s)]
        v, l, det = cpu_rate(sample, cores)
        kind, how = cpu_kind()
        # parity spot check on the same cycles: emitted message texts of the CUDA path vs the CPU arm (reported, not asserted
        # here -- the assertions live in tests/)
        from pyft8_b200.receiver import format_records
        from pyft8_b200 import messages
        same, diffs = 0, []
        off = np.concatenate([[0], np.cumsum(dev_counts)])
        for i in range(n_s):
            messages.call_hashes.clear()
            mb = format_records(dev_records[off[i]:off[i + 1]])
            ours = sorted(t for t, k in zip(mb.text.tolist(), mb.keep.tolist()) if k)
            ok = ours == sorted(det["texts"][i])
            same += ok
            if not ok and len(diffs) < 4:
                diffs.append({"cycle": i, "only_cuda": sorted(set(ours) - set(det["texts"][i])), "only_cpu": sorted(set(det["texts"][i]) - set(ours)),
                              "n_cuda": len(ours), "n_cpu": len(det["texts"][i])})
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": f"first {n_s} cycles of this run's batch ({args.cpu_cycles_per_core} per core), {how}, {det['wall_s']:.1f} s wall",
               "ldpc_codewords_per_sec": l, "sample_parity": {"cycles": n_s, "identical_message_sets": int(same), "differences": diffs}}
    configs = None
    if world == 1 and not args.no_configs and not args.device_only:
        eng.close()
        del audio, host_np
        host_pin.close()
        torch.cuda.empty_cache()
        configs = {"cfg3_fec": config_cfg3_fec(local, args.fec_codewords, args.fec_check),
                   "cfg4_120sig": config_cycles(local, "cfg4_120sig", args.cfg4_cycles, args.steps, args.seed + 4)}
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "cycles_per_gpu_per_step": B, "signals_per_cycle": workload.CONFIGS[WORKLOAD][0],
                   "snr_db": list(workload.CONFIGS[WORKLOAD][1]),
                   "audio": "int16 12 kHz 15 s", "l2": "inputs_larger_than_l2 (%.2f GB per step per GPU)" % (B * 360000 / 1e9),
                   "parallelism": f"cycles sharded over {world} GPU(s), no collective; records gathered on rank 0 host-side"},
        "ldpc_codewords_per_sec": ldpc_rate,
        "decodes_per_cycle": n_decoded / B, "emitted_per_cycle": n_emitted / B,
        "work_per_step": {k: stats[k] for k in ("candidates", "stopped_sd", "fine_evals", "fine_pass", "ldpc_calls", "ldpc_iters", "osd_calls")},
        "e2e": e2e_out, "host_text": host_text, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "roofline_stages": stages, "cpu_baseline": cpu, "configs": configs,
    }
    print(json.dumps(out), flush=True)


def main():
    global WORKLOAD
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cycles", type=int, default=4096, help="cycles per GPU per step (BASELINE configs[1]: 4096)")
    ap.add_argument("--seed", type=int, default=2000)
    ap.add_argument("--workload", default=WORKLOAD, choices=["cfg1_20sig", "cfg2_50sig", "cfg4_120sig"],
                    help="cfg2_50sig is the headline configuration (BASELINE configs[1])")
    ap.add_argument("--ref-cycles-per-core", type=int, default=1)
    ap.add_argument("--cpu-cycles-per-core", type=int, default=1, help="cycles per host core of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the configs[2] / configs[3] measurements of the default N=1 run")
    ap.add_argument("--device-only", action="store_true", help="only the device-resident timed steps (used under ncu)")
    ap.add_argument("--fec-codewords", type=int, default=1000000)
    ap.add_argument("--fec-check", type=int, default=64, help="LDPC vectors per Eb/N0 point re-decoded by the oracle (configs.cfg3_fec)")
    ap.add_argument("--cfg4-cycles", type=int, default=8192)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the records and per-cycle counts of the "
                    "last device-resident step (rank 0's batch) to DIR/<name>.npy, at most 64 MB in all")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the CUDA path's outputs (--impl b200)")
    WORKLOAD = args.workload
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    dist, rank, local, world = _dist_init()
    try:
        if args.impl == "reference":
            run_reference(args, dist, rank, world)
        else:
            run_gpu(args, dist, rank, local, world)
    finally:
        if _POOL is not None:
            _POOL.terminate()
        if dist:
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
