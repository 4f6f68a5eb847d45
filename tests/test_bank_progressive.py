"""ReceiverBank(progressive=True) host logic with a stub decoder: when progress calls are made, at which hop, with which
audio, how queued calls collapse, when a buffer half is reused, and how messages of one cycle are de-duplicated across
calls."""
import threading

import numpy as np
import pytest

from pyft8_b200 import _lib as L
from pyft8_b200 import synth
from pyft8_b200.bank import CYCLE_SAMPLES, ReceiverBank

S = 260


def _rec(r, call):
    from test_host_logic import _words_from_bits77
    rec = np.zeros(1, L.RECORD_DTYPE)
    rec[0]["bits91"] = _words_from_bits77([synth.pack77("CQ", call, "IO90")])[0]
    rec[0]["cycle"] = r
    return rec


class Stub:
    """decoder seam: records (hop, copy of the valid samples); receiver 0 gets the same message from every call.  With a
    gate, each call sets `entered` and then waits for the gate."""

    def __init__(self, gate=None):
        self.calls, self.gate, self.entered = [], gate, threading.Event()

    def __call__(self, audio, hop):
        if self.gate is not None:
            self.entered.set()
            self.gate.wait(10)
        self.calls.append((hop, audio[:, :480 * hop].copy()))
        return _rec(0, "K1ABC"), np.array([hop], np.uint16)


def _bank(stub, n=2, hops=1):
    return ReceiverBank(n, decoder=stub, clock=lambda: 45.0, progressive=True, progress_hops=hops)


def _expected(block, hops=1):
    """progress hops of one cycle fed in `block`-sample steps: the slowest position's hop after each block, rounded down to
    a multiple of progress_hops, when it passed the previous call and the first hop that can release a message"""
    out, last = [], 0
    for end in range(block, CYCLE_SAMPLES, block):
        h = end // 480
        h -= h % hops
        if S + 1 <= h < 375 and h > last:
            out.append(h)
            last = h
    return out + [375]


@pytest.mark.parametrize("block,hops", [(480, 1), (1000, 1), (480, 7), (CYCLE_SAMPLES, 1)])
def test_progress_schedule(block, hops):
    stub = Stub()
    bank = _bank(stub, hops=hops)
    rng = np.random.default_rng(block)
    x = rng.integers(-3000, 3000, (2, 2 * CYCLE_SAMPLES)).astype(np.int16)
    got = []
    for c in range(2):
        want = _expected(block, hops)
        for p in range(0, CYCLE_SAMPLES, block):
            n_before = len(got)
            bank.feed_all(x[:, c * CYCLE_SAMPLES + p:c * CYCLE_SAMPLES + min(p + block, CYCLE_SAMPLES)])
            end = min(p + block, CYCLE_SAMPLES)
            if (end < CYCLE_SAMPLES and end // 480 - (end // 480) % hops in want and
                    (not got or got[-1][1] != end // 480 - (end // 480) % hops)) or end == CYCLE_SAMPLES:
                got.append(bank.results(timeout=10))
            assert len(got) - n_before <= 1
        hops_c = [h for no, h, _ in got if no == c]
        assert hops_c == want
    # every call saw exactly the samples that had arrived, and nothing was decoded before the search hop had passed
    for (hop, a), (no, h, _) in zip(stub.calls, got):
        assert hop == h and np.array_equal(a, x[:, no * CYCLE_SAMPLES:no * CYCLE_SAMPLES + 480 * hop])
    # the message of receiver 0 comes once per cycle, from its first call, with its decode hop
    first = [m for no, h, ms in got for m in ms]
    assert len(first) == 2 and all(m["receiver"] == 0 and m["decode_hop"] == _expected(block, hops)[0] for m in first)
    bank.close()


def test_slowest_receiver_decides():
    stub = Stub()
    bank = _bank(stub, n=3)
    x = np.zeros((3, CYCLE_SAMPLES), np.int16)
    bank.feed(0, x[0, :480 * 300])
    bank.feed(1, x[1, :480 * 280])
    bank.feed(2, x[2, :480 * 262 + 10])
    assert bank.results(timeout=10)[:2] == (0, 262)
    bank.feed(1, x[1, 480 * 280:480 * 290])
    bank.feed(2, x[2, 480 * 262 + 10:480 * 270])
    assert bank.results(timeout=10)[:2] == (0, 270)          # receiver 2 is the slowest again
    bank.close()


def test_queued_calls_collapse_and_half_is_reused_after_the_final_call():
    gate = threading.Event()
    stub = Stub(gate)
    bank = _bank(stub)
    x = np.zeros((2, 3 * CYCLE_SAMPLES), np.int16)
    bank.feed_all(x[:, :480 * 262])                           # hop 262: a call that waits at the gate
    assert stub.entered.wait(10)                              # the worker has taken hop 262 before more is fed
    bank.feed_all(x[:, 480 * 262:480 * 300])                  # hops 263..300 queue up behind it
    bank.feed_all(x[:, 480 * 300:CYCLE_SAMPLES + 480 * 10])   # the final call of cycle 0, cycle 1 begins
    assert bank._busy[0] == 0                                 # cycle 0's half is held until its final call
    done = threading.Event()

    def feed_cycle_2():                                       # cycle 2 reuses half 0
        bank.feed_all(x[:, CYCLE_SAMPLES + 480 * 10:2 * CYCLE_SAMPLES + 100])
        done.set()
    t = threading.Thread(target=feed_cycle_2)
    t.start()
    assert not done.wait(0.5)
    gate.set()
    t.join(10)
    assert done.is_set()
    got = []
    while True:
        no, hop, ms = bank.results(timeout=10)
        got.append((no, hop))
        if (no, hop) == (1, 375):
            break
    assert got[0] == (0, 262) and got[1] == (0, 375)         # the queued calls collapsed into the latest one
    assert [h for no, h in got if no == 1][-1] == 375
    bank.close()


def test_progressive_needs_the_live_ring():
    with pytest.raises(ValueError):
        ReceiverBank(2, decoder=Stub(), progressive=True, live_ring=False)
