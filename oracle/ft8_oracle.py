"""CPU oracle for the FT8 receive hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A numpy restatement of what G1OJS/PyFT8 v3.9.0 computes on the path
audio -> waterfall -> Costas search -> LLR -> fine sync -> LDPC -> OSD -> CRC-14.
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this module; ``pyft8_b200`` never does.

Parity pin: PINNED.  ``tests/test_oracle_golden.py`` checks every function here
against dumps produced by running the *unmodified* reference in the authoring
container (``oracle/ref_harness.py`` + ``oracle/make_golden.py`` ->
``tests/golden/*.npz``) on the reference's two shipped WAVs
(tests/pipeline/test_08.wav, test_09.wav) and on seeded synthetic cycles.
The reference has no automated tests of its own for this path (SURVEY.md section 4).

Each function cites the reference lines it restates (paths relative to the
reference root, ``PyFT8/...``).  numpy 2.x semantics are assumed (single
precision FFTs on float32/complex64 input), as in the image the reference was
probed in.
"""
import math

import numpy as np

from ft8_tables import CHECK_VARS, GEN_MASK91, PREFIX2

# --------------------------------------------------------------------------- geometry
SAMP_RATE = 12000
SAMPLES_PER_CYCLE = 180000
NFFT_SEARCH = 3840          # receiver.py:230  (2 bins per tone)
HOP = 480                   # receiver.py:232  (4 hops per symbol)
HOPS_PER_CYCLE = 375        # receiver.py:237
GRID_ROWS = 750             # receiver.py:238
GRID_COLS = 976             # receiver.py:240  (960 + 8*2)
F0_LO, F0_HI = 32, 960      # receiver.py:234-235 with [100, 3000] Hz
H0_LO, H0_HI = -37, 87      # receiver.py:319 with [-2.0, 3.0] s
NFFT_CYCLE = 192000         # receiver.py:249
NFFT_FINE = 3200            # receiver.py:46
COSTAS = (3, 1, 4, 0, 6, 5, 2)                       # receiver.py:13
PAYLOAD_SYMS = tuple(range(7, 36)) + tuple(range(43, 72))   # receiver.py:14
COSTAS_SYMS = tuple(range(7)) + tuple(range(36, 43)) + tuple(range(72, 79))  # receiver.py:15

# a-priori patterns: (name, first llr index, bits)    receiver.py:21-27
AP_PATTERNS = (
    ("NoAP", 0, ()),
    ("CQ", 0, (0,) * 26 + (1, 0, 0)),
    ("RR73", 58, (0, 1, 1, 1, 1, 1, 1, 0, 0, 1, 1, 1, 0, 1, 0, 1, 0, 0, 1)),
    ("73", 58, (0, 1, 1, 1, 1, 1, 1, 0, 1, 0, 0, 1, 0, 1, 0, 0, 0, 0, 1)),
    ("RRR", 58, (0, 1, 1, 1, 1, 1, 1, 0, 1, 0, 0, 1, 0, 0, 1, 0, 0, 0, 1)),
)

_CV = np.array(CHECK_VARS, dtype=np.int16)
CV6 = np.ascontiguousarray(_CV[:59, :6])             # decoders.py:134
CV7 = np.ascontiguousarray(_CV[59:, :7])             # decoders.py:135
_HANN = np.hanning(NFFT_SEARCH).astype(np.float32)   # receiver.py:236


def _costas_kernel(bins_per_tone):
    k = np.full((7, 7 * bins_per_tone), -1.0 / 6.0, np.float32)
    for s, tone in enumerate(COSTAS):
        k[s, tone * bins_per_tone:(tone + 1) * bins_per_tone] = 1.0
    return k.ravel()


CSYNC_SEARCH = _costas_kernel(2)     # receiver.py:323-327
CSYNC_FINE = _costas_kernel(1)       # receiver.py:198-201


# --------------------------------------------------------------------------- S1 spectrogram
def spectrogram(audio_i16):
    """Isolated-cycle waterfall, rows 0..375 (row 0 and every row > 375 are 1.0).

    Row h is the window over samples [480h-3840, 480h), zero before the cycle start:
    receiver.py:288-293 driven by receiver.py:295-306 under the SURVEY 8c recipe.
    Returns float32[376, 976] in dB.
    """
    x = np.zeros(NFFT_SEARCH + SAMPLES_PER_CYCLE, np.float32)
    x[NFFT_SEARCH:] = np.asarray(audio_i16).astype(np.float32)
    grid = np.ones((HOPS_PER_CYCLE + 1, GRID_COLS), np.float32)
    buf = np.empty(NFFT_SEARCH, np.float32)
    for h in range(1, HOPS_PER_CYCLE + 1):
        np.multiply(x[HOP * h:HOP * h + NFFT_SEARCH], _HANN, out=buf)
        z = np.fft.rfft(buf)[:GRID_COLS]
        grid[h] = 20 * np.log10(np.abs(z) + 1e-12)
    return grid


def grid_row(grid, r):
    """Row r (mod 750) of the two-cycle grid whose rows >= len(grid) still hold 1.0 (receiver.py:240)."""
    r %= GRID_ROWS
    if r < grid.shape[0]:
        return grid[r]
    return np.ones(GRID_COLS, np.float32)


def full_grid(grid):
    g = np.ones((GRID_ROWS, GRID_COLS), np.float32)
    g[:grid.shape[0]] = grid
    return g


# --------------------------------------------------------------------------- S2 Costas search
def search(grid, score_min=85, max_cands=200, odd_even=0, f0_range=None, h0_range=None):
    """Coarse sync over (f0, h0); one candidate per f0 bin.  receiver.py:338-367.

    f0_range / h0_range: [lo, hi) index ranges as Receiver derives them from search_freq_range / search_time_range
    (receiver.py:232, 319); None = the defaults [32, 960) and [-37, 87).

    Scores only the middle Costas block (rows h0+148+4k); strict '>' from 0;
    keeps score > score_min; stable sort by score descending; first max_cands.
    Returns (f0[n], h0[n], score[n] float64, payload_dB[n,58,8] float32).
    """
    g = full_grid(grid)
    cycle_h0 = odd_even * HOPS_PER_CYCLE
    base = 148 + 4 * np.arange(7)                       # receiver.py:322 + :347
    found = []
    f_lo, f_hi = f0_range if f0_range is not None else (F0_LO, F0_HI)
    h_lo, h_hi = h0_range if h0_range is not None else (H0_LO, H0_HI)
    for f0 in range(f_lo, f_hi):
        strip = g[:, f0:f0 + 14]
        best, best_h0 = 0.0, None
        for h0 in range(h_lo, h_hi):
            s = float(np.dot(strip[h0 + cycle_h0 + base, :].ravel(), CSYNC_SEARCH))
            if s > best:
                best, best_h0 = s, h0
        if best > score_min:
            found.append((f0, best_h0, best))
    found.sort(key=lambda c: c[2], reverse=True)         # stable (receiver.py:366)
    found = found[:max_cands]
    n = len(found)
    f0s = np.array([c[0] for c in found], np.int32).reshape(n)
    h0s = np.array([c[1] for c in found], np.int32).reshape(n)
    sc = np.array([c[2] for c in found], np.float64).reshape(n)
    pay = np.empty((n, 58, 8), np.float32)
    for i in range(n):
        pay[i] = payload_from_grid(g, f0s[i], h0s[i], cycle_h0)
    return f0s, h0s, sc, pay


def search_scores(grid, odd_even=0):
    """All 928 x 124 scores in float64 (used by tests to reason about near-ties)."""
    g = full_grid(grid).astype(np.float64)
    cycle_h0 = odd_even * HOPS_PER_CYCLE
    k = CSYNC_SEARCH.astype(np.float64).reshape(7, 14)
    out = np.zeros((F0_HI - F0_LO, H0_HI - H0_LO))
    for i, h0 in enumerate(range(H0_LO, H0_HI)):
        rows = g[h0 + cycle_h0 + 148 + 4 * np.arange(7)]          # 7 x 976
        for j in range(14):
            out[:, i] += (rows[:, F0_LO + j:F0_HI + j] * k[:, j:j + 1]).sum(axis=0)
    return out


def payload_from_grid(g750, f0, h0, cycle_h0=0):
    """58x8 dB payload: upper bin of each 2-bin tone, rows wrap mod 750.  receiver.py:358-362."""
    rows = [(cycle_h0 + h0 + 4 + 4 * s) % GRID_ROWS for s in PAYLOAD_SYMS]
    cols = [f0 + 1 + 2 * t for t in range(8)]
    return g750[rows, :][:, cols]


# --------------------------------------------------------------------------- L0 dB -> LLR
def db_to_llr(p):
    """Max-log 8-FSK LLRs with the reference's Gray map and scaling.  receiver.py:208-222.

    Returns (llr float32[174], sd float32, snr int).  llr > 0 means bit 1.
    """
    p = np.asarray(p)
    snr = int(np.clip(int(np.max(p) - np.min(p) - 58), -24, 24))
    a = np.max(p[:, [4, 5, 6, 7]], axis=1) - np.max(p[:, [0, 1, 2, 3]], axis=1)
    b = np.max(p[:, [2, 3, 4, 7]], axis=1) - np.max(p[:, [0, 1, 5, 6]], axis=1)
    c = np.max(p[:, [1, 2, 6, 7]], axis=1) - np.max(p[:, [0, 3, 4, 5]], axis=1)
    l = np.column_stack((a, b, c)).ravel()
    m = np.mean(l)
    sd = np.sqrt(np.mean(l * l) - m * m)
    with np.errstate(all="ignore"):
        llr = 2.83 * l / sd
    return llr, sd, snr


def set_ap(llr0, ap):
    """A-priori mask: known bits forced to +-5.  receiver.py:109-117."""
    name, b0, bits = AP_PATTERNS[ap]
    llr = llr0.copy()
    for i, b in enumerate(bits):
        llr[b0 + i] = (2 * b - 1) * 5
    if name == "CQ":
        llr[74:76] = -5
        llr[76] = 5
        llr[57:59] = -5
    return llr


# --------------------------------------------------------------------------- F1..F3 fine sync
def cycle_spectrum(audio_i16):
    """rfft of the cycle zero-padded to 192000 (0.0625 Hz bins).  receiver.py:280-286 (roll == identity)."""
    buf = np.zeros(NFFT_CYCLE, np.float32)
    buf[:SAMPLES_PER_CYCLE] = np.asarray(audio_i16).astype(np.float32)
    return np.fft.rfft(buf)


_TAPER_HI = 0.5 * (1 + np.cos(np.linspace(np.pi, 0, 100)))     # receiver.py:183 (rises 0 -> 1, sic)
_TAPER_LO = 0.5 * (1 + np.cos(np.linspace(-np.pi, 0, 100)))    # receiver.py:184


def fine_baseband(spec, fb):
    """1000 bins around fb -> 3200 samples at 200 Hz.  receiver.py:180-186."""
    a = np.zeros(NFFT_FINE, np.complex64)
    a[150:1000] = spec[fb:fb + 850]
    a[:150] = spec[fb - 150:fb]
    a[900:1000] *= _TAPER_HI
    a[:100] *= _TAPER_LO
    a = np.roll(a, -150)
    return np.fft.ifft(a)


def fine_grid_from_baseband(z, tb):
    """79 symbols x 8 tone magnitudes from 32-sample windows at clip(tb+32j).  receiver.py:189-195."""
    idx = np.clip(tb + 32 * np.arange(79), 0, NFFT_FINE - 32)
    sym = np.empty((79, 32), np.complex64)
    for j, i0 in enumerate(idx):
        sym[j] = z[i0:i0 + 32]
    return np.abs(np.fft.fft(sym, axis=1)[:, :8])


def fine_score(g):
    """Middle Costas block only, linear magnitudes.  receiver.py:203-206."""
    return float(np.dot(g[36:43, :7].ravel(), CSYNC_FINE))


def signal_grid_fine(spec, fb, tb):
    g = fine_grid_from_baseband(fine_baseband(spec, fb), tb)
    return g, fine_score(g)


def llr_fine(spec, fHz, tsec):
    """Fine time then frequency refinement + Costas gate.  receiver.py:140-173.

    Returns dict(tt, ff, nsync, grid[79,8]); tsec/fHz updates and the LLR step are
    applied by the caller when nsync > 6.
    """
    fb0 = int(0.5 + fHz * NFFT_CYCLE / SAMP_RATE)
    tb0 = int(0.5 + tsec / 0.005)
    z = fine_baseband(spec, fb0)
    tts = list(range(-8, 8, 2))
    sc = [fine_score(fine_grid_from_baseband(z, tb0 + t)) for t in tts]
    tt = tts[int(np.argmax(sc))]
    ffs = list(range(-32, 33, 8))
    sc = [signal_grid_fine(spec, fb0 + f, tb0 + tt)[1] for f in ffs]
    ff = ffs[int(np.argmax(sc))]
    g, _ = signal_grid_fine(spec, fb0 + ff, tb0 + tt)
    hits = np.argmax(g[list(COSTAS_SYMS), :], axis=1) - np.array(COSTAS * 3)
    nsync = int(np.sum(hits == 0))
    return dict(tt=tt, ff=ff, nsync=nsync, grid=g)


# --------------------------------------------------------------------------- K1 CRC-14 + validity
def crc14(bits77):
    """CRC-14 (poly 0x2757) of the 77 message bits zero-extended to 82, MSB first.  decoders.py:123-129."""
    r = 0
    for i in range(96):
        bit = (bits77 >> (76 - i)) & 1 if i < 77 else 0
        top = (r >> 13) & 1
        r = ((r << 1) & 0x3FFF) | bit
        if top:
            r ^= 0x2757
    return r


def bits_to_int(bits):
    v = 0
    for b in np.asarray(bits).astype(int).tolist():
        v = (v << 1) | (b & 1)
    return v


def crc_ok91(bits91):
    """decoders.py:117-130 minus the unpack: non-zero payload and matching CRC."""
    b77 = bits91 >> 14
    return b77 > 0 and crc14(b77) == (bits91 & 0x3FFF)


_A1 = " 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ"
_A2 = "0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ"
_A3 = "0123456789" + " " * 17
_A4 = " ABCDEFGHIJKLMNOPQRSTUVWXYZ"
NTOKENS, MAX22 = 2063592, 4194304


def _call_text(n28):
    """Standard 28-bit callsign -> text (None when not representable).  decoders.py:95-105."""
    nn = n28 - (NTOKENS + MAX22)
    ch = []
    for alphabet, div in ((_A1, 36 * 10 * 27 ** 3), (_A2, 10 * 27 ** 3), (_A3, 27 ** 3),
                          (_A4, 27 ** 2), (_A4, 27), (_A4, 1)):
        i, nn = divmod(nn, div)
        ch.append(alphabet[i])          # nn == -1 (n28 = 6257895) indexes from the end, like the reference
    return "".join(ch).strip()


def _call_shape_ok(c):
    """decoders.py:107-113: the two accepted callsign shapes."""
    if " " in c or len(c) < 3:
        return False
    if c[0] in "ABCDEFGHIJKLMNOPRSTUVWXYZ" and c[1].isdigit():
        if not (c[0] in "BFGIKMNRW" and c[2].isdigit()):
            return True
    return c[1] in PREFIX2.get(c[0], "") and c[2].isdigit()


def _c29_ok(c29, i3):
    n28, p = c29 >> 1, c29 & 1
    if n28 < NTOKENS + MAX22 - 1:            # decoders.py:73-84 (tokens, CQ nnn, CQ abcd, hashes)
        return True
    c = _call_text(n28)
    if not _call_shape_ok(c):
        return False
    if p and i3 == 1 and c[0] not in "AKNW":  # '/R' only on A/K/N/W calls, decoders.py:88-91
        return False
    return True


def valid77(b):
    """True iff the reference's unpack() returns a message for payload b.  decoders.py:16-68 as a predicate."""
    if b == 0:
        return False
    i3, b74 = b & 7, b >> 3
    if i3 in (1, 2):
        g15 = b74 & 0x7FFF
        if g15 == 0 or g15 in (32400, 32401):
            return False
        return _c29_ok((b74 >> 45) & 0x1FFFFFFF, i3) and _c29_ok((b74 >> 16) & 0x1FFFFFFF, i3)
    if i3 == 4:
        cq, rrr = b74 & 1, (b74 >> 1) & 3
        return (cq != 0) != (rrr != 0)
    return False


def good91(llr):
    """GOOD91 test on the hard decisions of llr[:91].  receiver.py:119-122 + decoders.py:117-131."""
    bits91 = bits_to_int(np.asarray(llr[:91]) > 0)
    if crc_ok91(bits91) and valid77(bits91 >> 14):
        return bits91
    return None


# --------------------------------------------------------------------------- L1/L2 LDPC
ST_REJECT, ST_OK, ST_FAIL = 0, 1, 2


def _pass_messages(llr, idx, prev, delta):
    """One flooding half-step over a group of checks.  decoders.py:140-151."""
    v2c = llr[idx] - prev
    t = np.tanh(-v2c)
    prod = np.prod(t, axis=1, keepdims=True)
    with np.errstate(all="ignore"):
        e = np.divide(prod, t)
        new = e / ((e - 1.18) * (1.18 + e))
    np.add.at(delta, idx, new - prev)
    return new


def ldpc_decode(llr, max_ncheck0, max_iters):
    """Sum-product decoder with the reference's schedule.  decoders.py:153-171.

    ``llr`` (float32[174]) is updated IN PLACE.  Returns (status, n_its, bits91):
    ST_REJECT (iteration-0 syndrome weight > max_ncheck0; llr untouched),
    ST_OK (syndrome 0, CRC ok, payload valid at iteration n_its) or ST_FAIL.
    """
    prev6 = np.zeros(CV6.shape, np.float32)
    prev7 = np.zeros(CV7.shape, np.float32)
    with np.errstate(all="ignore"):
        for it in range(max_iters):
            par6 = np.sum(llr[CV6] > 0, axis=1) & 1
            par7 = np.sum(llr[CV7] > 0, axis=1) & 1
            ncheck = int(par6.sum() + par7.sum())
            if it == 0 and ncheck > max_ncheck0:
                return ST_REJECT, -1, None
            if ncheck == 0:
                b = good91(llr)
                if b is not None:
                    return ST_OK, it, b
            else:
                delta = np.zeros_like(llr)
                prev6 = _pass_messages(llr, CV6, prev6, delta)
                prev7 = _pass_messages(llr, CV7, prev7, delta)
                llr += delta
    return ST_FAIL, -1, None


# --------------------------------------------------------------------------- O1 OSD
def _g0():
    a = np.zeros((83, 91), np.uint8)
    for i, m in enumerate(GEN_MASK91):
        for j in range(91):
            a[i, 90 - j] = (m >> j) & 1
    return np.concatenate([np.eye(91, dtype=np.uint8), a.T], axis=1)     # decoders.py:176-180


G0 = _g0()


def osd_order(llr):
    """Reliability order: |llr| descending, ties by ascending index, NaN last (SURVEY H6)."""
    return np.argsort(-np.abs(llr), kind="stable")


def osd_candidates(llr, singleflips=30, doubleflips=2):
    """All OSD trial words (91-bit ints) in the reference's enumeration order.  decoders.py:223-272."""
    g = G0.copy()
    rows = np.arange(91)
    cols = osd_order(llr)
    cr = 0
    for cc in range(174):
        hit = np.where(g[rows[cr:], cols[cc]] == 1)[0]
        if hit.size:
            sw = cr + hit[0]
            rows[[cr, sw]] = rows[[sw, cr]]
            piv = rows[cr]
            col = g[:, cols[cc]].copy()
            col[piv] = 0
            g[np.where(col == 1)[0], :] ^= g[piv, :]
            cols[[cr, cc]] = cols[[cc, cr]]
            cr += 1
            if cr > 90:
                break
    t = g[:, :91]
    u = np.zeros(91, np.uint8)
    u[rows] = (llr > 0).astype(np.uint8)[cols][:91]
    flips = list(rows[::-1][:singleflips])
    out = [bits_to_int((u @ t) & 1)]
    for i in range(singleflips):
        v = u.copy()
        v[flips[i]] ^= 1
        out.append(bits_to_int((v @ t) & 1))
    for i in range(singleflips):
        for j in range(doubleflips):
            if j < i:
                v = u.copy()
                v[flips[i]] ^= 1
                v[flips[j]] ^= 1
                out.append(bits_to_int((v @ t) & 1))
    return out


def osd(llr, singleflips=30, doubleflips=2):
    """First trial word with non-zero payload, CRC ok and valid payload; else None."""
    for b in osd_candidates(llr, singleflips, doubleflips):
        if crc_ok91(b) and valid77(b >> 14):
            return b
    return None


# --------------------------------------------------------------------------- C1 pass scheduler
class Cand:
    __slots__ = ("idx", "f0", "h0", "score", "payload", "tsec", "fHz", "ipass", "result", "bits91",
                 "notes", "tweaks", "llr_sd", "snr", "llr", "llr0", "source", "saved", "nsync",
                 "grid_sd", "fine_sd", "n_ldpc", "n_ldpc_its", "n_osd", "final_ipass")


def _try_good91(c, ap):
    if c.result is None:
        c.notes = f"{c.source}_{AP_PATTERNS[ap][0]}_GOOD91 "
        b = good91(c.llr)
        if b is not None:
            c.result, c.bits91 = "ok", b


def _try_ldpc(c, ap, nc0, its, save):
    if c.result is None:
        c.notes = f"{c.source}_{AP_PATTERNS[ap][0]}_LDPC{its}"
        st, n, b = ldpc_decode(c.llr, nc0, its)
        c.n_ldpc += 1
        if st == ST_OK:
            c.result, c.bits91 = "ok", b
        elif save and st == ST_FAIL:
            c.saved.append((f"{AP_PATTERNS[ap][0]}_LDPC{its}", c.llr))


def _try_osd(c, name, singleflips=30, doubleflips=2):
    if c.result is None:
        c.notes = f"{c.source}_{name}_OSD"
        c.n_osd += 1
        b = osd(c.llr, singleflips, doubleflips)     # osd_012(singleflips, doubleflips), decoders.py:223
        if b is not None:
            c.result, c.bits91 = "ok", b


def _set_llr(c, p, llr_sd_min=5):
    with np.errstate(all="ignore"):
        c.llr, c.llr_sd, c.snr = db_to_llr(p)
    if c.llr_sd <= llr_sd_min:             # Candidate(llr_sd_min), receiver.py:221-222
        c.result = "stop"


def decode_step(c, spec, llr_sd_min=5, osd_singleflips=30, osd_doubleflips=2):
    """Advance one candidate by one pass.  receiver.py:68-107."""
    if c.result == "stop":
        return
    ip = c.ipass
    if ip == 0:
        c.source = "grid"
        _set_llr(c, c.payload, llr_sd_min)
        c.grid_sd = float(c.llr_sd)
        c.llr0 = c.llr.copy()
        for ap in range(5):
            c.llr = set_ap(c.llr0, ap)
            _try_good91(c, ap)
            _try_ldpc(c, ap, 35, 5, False)
    elif ip == 1:
        c.source = "fine"
        r = llr_fine(spec, c.fHz, c.tsec)
        c.tweaks = f" t:{r['tt']:+03d} f:{r['ff']:+03d}"
        c.nsync = r["nsync"]
        if r["nsync"] > 6:
            c.tsec = float(c.tsec + r["tt"] / 200)
            c.fHz = float(c.fHz + r["ff"] / 16)
            with np.errstate(all="ignore"):
                _set_llr(c, 20 * np.log10(r["grid"][list(PAYLOAD_SYMS), :]), llr_sd_min)
            c.fine_sd = float(c.llr_sd)
        else:
            c.result = "stop"
    elif ip == 2:
        c.llr0 = c.llr.copy()
        for ap in range(2):
            c.llr = set_ap(c.llr0, ap)
            _try_good91(c, ap)
    elif ip == 3:
        for ap in range(2):
            c.llr = set_ap(c.llr0, ap)
            _try_ldpc(c, ap, 35, 5, False)
    elif ip == 4:
        for ap in range(5):
            c.llr = set_ap(c.llr0, ap)
            _try_ldpc(c, ap, 90, 20, True)
    elif ip == 5:
        for ap in range(5):
            c.llr = set_ap(c.llr0, ap)
            _try_osd(c, AP_PATTERNS[ap][0], osd_singleflips, osd_doubleflips)
    elif ip == 6:
        for name, llr in c.saved:
            c.llr = llr
            _try_osd(c, name, osd_singleflips, osd_doubleflips)
    elif ip == 7:
        c.result = "stop"
    c.ipass += 1


def decode_cycle(audio_i16, score_min=85, max_cands=200, odd_even=0, grid=None, cands=None, llr_sd_min=5,
                 osd_singleflips=30, osd_doubleflips=2):
    """Whole path for one isolated cycle.  Mirrors receiver.py:389-398 without time starvation.

    llr_sd_min: Candidate(llr_sd_min) (receiver.py:221-222); osd_singleflips / osd_doubleflips: osd_012(singleflips,
    doubleflips) (decoders.py:223).  The defaults are the reference's.

    Returns (records, cands): ``records`` are the emitted decodes in emission order, each a dict
    with bits77, bits91, tsec, fHz, snr, notes (pass name + tweaks), cand index.  Emission de-dup
    is on the 77-bit payload (the reference keys on the message text, receiver.py:53; identical
    except for hash-dependent '<...>' text, SURVEY H7).
    """
    if grid is None:
        grid = spectrogram(audio_i16)
    if cands is None:
        cands = search(grid, score_min, max_cands, odd_even)
    f0s, h0s, sc, pay = cands
    cl = []
    for i in range(len(f0s)):
        c = Cand()
        c.idx, c.f0, c.h0, c.score, c.payload = i, int(f0s[i]), int(h0s[i]), float(sc[i]), pay[i]
        c.tsec, c.fHz = c.h0 / 25.0, 3.125 * c.f0           # receiver.py:350-351
        c.ipass, c.result, c.bits91, c.notes, c.tweaks = 0, None, None, "", "t:+00 f:+00"
        c.llr_sd, c.snr, c.saved, c.nsync, c.source = 0, 0, [], 100, None
        c.grid_sd = c.fine_sd = float("nan")
        c.n_ldpc = c.n_ldpc_its = c.n_osd = 0
        c.final_ipass = -1
        cl.append(c)
    spec = None
    seen, records = set(), []
    for _ in range(9):
        todo = [c for c in cl if c.result is None]
        if not todo:
            break
        todo.sort(key=lambda c: c.llr_sd, reverse=True)
        for c in todo:
            if c.ipass == 1 and spec is None:
                spec = cycle_spectrum(audio_i16)
            ip = c.ipass
            decode_step(c, spec, llr_sd_min, osd_singleflips, osd_doubleflips)
            if c.result is not None:
                c.final_ipass = ip
            if c.result == "ok":
                b77 = c.bits91 >> 14
                if b77 not in seen:
                    seen.add(b77)
                    records.append(dict(bits77=b77, bits91=c.bits91, tsec=c.tsec, fHz=c.fHz, snr=int(c.snr),
                                        notes=c.notes + c.tweaks, cand=c.idx, ipass=ip))
                c.result = "stop"
    return records, cl


def work_counters(cl):
    """The library's per-call work counters (ft8_stats) of one decoded cycle's Cand list, counted as the kernels count:

    candidates  every candidate                                  stopped_sd  stopped by the ipass-0 sd gate
    fine_evals  candidates that reach ipass 1 (fine sync)        fine_pass   candidates that reach ipass 2
    ldpc_calls  every LDPC decode (iteration-0 rejects included)
    osd_calls   5 + len(saved) per candidate that reaches ipass 5: the library runs all of a candidate's OSD attempts and
                then takes the first success in reference order, where the oracle's own n_osd stops at the first success.
    """
    # every candidate ends in some pass (final_ipass); one that ends in ipass 0 undecoded was stopped by the sd gate
    return dict(candidates=len(cl), stopped_sd=sum(c.final_ipass == 0 and c.bits91 is None for c in cl),
                fine_evals=sum(c.final_ipass >= 1 for c in cl), fine_pass=sum(c.final_ipass >= 2 for c in cl),
                ldpc_calls=sum(c.n_ldpc for c in cl), osd_calls=sum(5 + len(c.saved) for c in cl if c.final_ipass >= 5))


# --------------------------------------------------------------------------- message text (host side)
def unpack77(b, hashes=None):
    """77-bit payload -> (call_a, call_b, extra) text tuple, or None.  decoders.py:16-105.

    ``hashes`` maps (hash, nbits) -> callsign for '<...>' resolution (databases.py:8-26); it is
    read only (the reference also inserts every decoded call; callers that want history do that).
    """
    if not valid77(b):
        return None
    hashes = hashes or {}
    i3, b74 = b & 7, b >> 3
    if i3 == 4:
        cq, rrr, swp = b74 & 1, (b74 >> 1) & 3, (b74 >> 3) & 1
        c58, h12 = (b74 >> 4) & ((1 << 58) - 1), (b74 >> 62) & 0xFFF
        ca = "CQ" if cq else "<%s>" % hashes.get((h12, 12), "...")
        cb = ""
        for _ in range(12):
            cb = " 0123456789ABCDEFGHIJKLMNOPQRSTUVWXYZ/"[c58 % 38] + cb
            c58 //= 38
        cb = cb.strip()
        if swp:
            ca, cb = cb, ca
        return (ca, cb, ("", "RRR", "RR73", "73")[rrr])
    g16 = b74 & 0xFFFF
    g15 = g16 & 0x7FFF
    if g15 < 32400:
        a, r = divmod(g15, 1800)
        bb, r = divmod(r, 100)
        extra = chr(65 + a) + chr(65 + bb) + "%d%d" % divmod(r, 10)
    elif g15 <= 32404:
        extra = ("", "", "RRR", "RR73", "73")[g15 - 32400]
    else:
        extra = ("R" if g16 >> 15 else "") + "%+03d" % (g15 - 32435)

    def call(c29):
        n28, p = c29 >> 1, c29 & 1
        if n28 < 3:
            return ("DE", "QRZ", "CQ")[n28]
        if n28 < 1004:
            return "CQ %03d" % (n28 - 3)
        if n28 < 21443:
            x, t = n28 - 1003, ""
            for _ in range(4):
                t = _A4[x % 27] + t
                x //= 27
            return "CQ " + t.strip()
        if n28 < NTOKENS + MAX22 - 1:
            return "<%s>" % hashes.get((n28 - NTOKENS, 22), "...")
        c = _call_text(n28)
        if p:
            c += "/P" if i3 == 2 else "/R"
        return c
    return (call((b74 >> 45) & 0x1FFFFFFF), call((b74 >> 16) & 0x1FFFFFFF), extra)
