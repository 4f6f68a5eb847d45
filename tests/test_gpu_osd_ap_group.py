"""Pass 5's OSD attempts as the decode runs them, against stand-alone OSD calls.

The decode runs the AP attempts RR73, 73 and RRR of a candidate on one reliability order and one basis: the three patterns
force the same positions 58..76 to +-5, so only the hard decisions differ between them.  ft8_debug_osd_ap runs that code on
host llrs; every attempt must equal ft8_osd (which finds order and basis per call) on the llr with that AP pattern applied,
found index and 91-bit word alike, and on a subset the oracle's osd_012.
"""
import numpy as np
import pytest

import ft8_oracle as o
from pyft8_b200 import synth
from pyft8_b200.engine import Engine, bits91_to_int

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    e = Engine(device=0, max_cycles=1)
    yield e
    e.close()


def ap_copies(x):
    return np.stack([np.stack([o.set_ap(row, ap) for ap in range(5)]) for row in x]).astype(np.float32)


def check_against_osd(eng, x, S=30, D=2):
    """Every attempt of ft8_debug_osd_ap equals ft8_osd on that AP copy; returns the found indices [N][5]."""
    found, bits = eng.debug_osd_ap(x, S, D)
    want_f, want_b = eng.osd(ap_copies(x).reshape(-1, 174), S, D)
    np.testing.assert_array_equal(found, want_f.reshape(-1, 5))
    np.testing.assert_array_equal(bits, want_b.reshape(-1, 5, 3))
    return found


def check_against_oracle(eng, x, rows, S=30, D=2):
    found, bits = eng.debug_osd_ap(x, S, D)
    for i in rows:
        for ap in range(5):
            cands = o.osd_candidates(o.set_ap(x[i], ap), S, D)
            want = next((k + 1 for k, b in enumerate(cands) if o.crc_ok91(b) and o.valid77(b >> 14)), 0)
            assert found[i, ap] == want, (i, ap)
            assert bits91_to_int(bits[i, ap]) == cands[want - 1 if want else 0], (i, ap)


def test_noisy_codewords(eng):
    found = np.concatenate([check_against_osd(eng, synth.make_llr_codewords(700 + e, 96, float(e))[0]) for e in (0, 1, 2)])
    # the shared attempts decode, and not all alike: the signs of 58..76 reach the result
    assert (found[:, 2:] > 0).sum() >= 20
    assert np.any((found[:, 2] > 0) != (found[:, 3] > 0)) or np.any((found[:, 3] > 0) != (found[:, 4] > 0))


def test_exact_ties_with_the_forced_values(eng):
    rng = np.random.default_rng(31)
    x, _ = synth.make_llr_codewords(31, 48, 1.0)
    for i in range(len(x)):
        q = rng.choice(np.r_[0:58, 77:174], size=int(rng.integers(5, 60)), replace=False)
        x[i, q] = np.where(rng.random(len(q)) < 0.5, 5.0, -5.0)
    check_against_osd(eng, x)
    check_against_oracle(eng, x, range(0, 48, 12))


def test_nan_zero_and_inf_outside_the_forced_range(eng):
    rng = np.random.default_rng(32)
    x, _ = synth.make_llr_codewords(32, 40, 1.5)
    for i in range(len(x)):
        q = rng.choice(np.r_[0:58, 77:174], size=6, replace=False)
        x[i, q[0]] = 0.0
        x[i, q[1]] = -0.0
        if i % 2:
            x[i, q[2]] = np.nan
        if i % 3 == 0:
            x[i, q[3]] = np.inf
        if i % 4 == 0:
            x[i, q[4]] = -np.inf
        if i % 5 == 0:
            x[i, q[5]] = np.nan
    check_against_osd(eng, x)
    check_against_oracle(eng, x, (0, 1, 3))


def test_sort_code_collisions(eng):
    """Magnitudes that share the 24-bit sort code with the forced 5.0 (or with each other) send the order to the exact
    counting path."""
    rng = np.random.default_rng(33)
    x, _ = synth.make_llr_codewords(33, 32, 1.5)
    ulp = lambda v, k: (np.float32(v).view(np.uint32) + np.uint32(k)).view(np.float32)
    for i in range(len(x)):
        q = rng.choice(np.r_[0:58, 77:174], size=10, replace=False)
        base = 5.0 if i % 2 == 0 else abs(x[i, q[0]])
        for j, p in enumerate(q):
            x[i, p] = ulp(base, (j * 3) % 16) * (1 if rng.random() < 0.5 else -1)
    check_against_osd(eng, x)
    check_against_oracle(eng, x, (0, 1))


@pytest.mark.parametrize("S,D", [(45, 25), (0, 0), (91, 3), (10, 0), (2, 2)])
def test_flip_parameters(eng, S, D):
    x, _ = synth.make_llr_codewords(34, 64, 1.0)
    check_against_osd(eng, x, S, D)
    check_against_oracle(eng, x, (0, 5), S, D)
