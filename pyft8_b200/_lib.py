"""ctypes binding of libft8_b200.so (the C ABI declared in include/ft8_b200.h).

The shared library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no CPU
fallback: if the library is missing or no CUDA device can be opened, loading / ``Engine()`` raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PYFT8_B200_LIB") or os.path.join(_HERE, "libft8_b200.so")   # env override: A/B builds

OK, E_BADARG, E_CUDA, E_CAPACITY, E_NODEVICE = 0, -1, -2, -3, -4
MEM_HOST, MEM_DEVICE = 0, 1
HOST_WRITE_COMBINED = 1
AUDIO_I16, AUDIO_F32 = 0, 1
GRID_ROWS, GRID_ROWS_LIVE, GRID_COLS, SPEC_BINS = 376, 750, 976, 96001
LDPC_REJECT, LDPC_OK, LDPC_FAIL, LDPC_STALL = 0, 1, 2, 3
METHOD_NAMES = ("GOOD91 ", "LDPC5", "LDPC20", "OSD", "LDPC20_OSD")   # decode_notes suffixes, receiver.py:121,126,133
AP_NAMES = ("NoAP", "CQ", "RR73", "73", "RRR")                          # receiver.py:21-27


class Cfg(C.Structure):
    _fields_ = [("max_cycles", C.c_int32), ("max_cands", C.c_int32), ("sync_score_min", C.c_float),
                ("llr_sd_min", C.c_float), ("osd_singleflips", C.c_int32), ("osd_doubleflips", C.c_int32),
                ("max_codewords", C.c_int32), ("fine_mode", C.c_int32),
                ("search_f0_lo", C.c_int16), ("search_f0_hi", C.c_int16), ("search_h0_lo", C.c_int16), ("search_h0_hi", C.c_int16),
                ("reserved", C.c_int32 * 2)]


class Record(C.Structure):
    _fields_ = [("bits91", C.c_uint32 * 3), ("cycle", C.c_int32), ("cand", C.c_int16), ("f0_idx", C.c_int16),
                ("h0_idx", C.c_int16), ("snr", C.c_int8), ("ipass", C.c_uint8), ("ap", C.c_uint8),
                ("method", C.c_uint8), ("ttweak", C.c_int8), ("ftweak", C.c_int8), ("nsync", C.c_uint8),
                ("emitted", C.c_uint8), ("n_its", C.c_uint16), ("score", C.c_float), ("tsec", C.c_float),
                ("fHz", C.c_float), ("grid_sd", C.c_float), ("fine_sd", C.c_float), ("reserved", C.c_uint32 * 3)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("cycles", "candidates", "stopped_sd", "fine_evals", "fine_pass",
                                         "ldpc_calls", "ldpc_iters", "osd_calls", "decoded", "emitted",
                                         "kernel_launches", "fine_rechecked")] + [("reserved", C.c_int64 * 4)]


# numpy structured dtype with the same layout as ft8_record
import numpy as _np  # noqa: E402

RECORD_DTYPE = _np.dtype([("bits91", "<u4", (3,)), ("cycle", "<i4"), ("cand", "<i2"), ("f0_idx", "<i2"),
                          ("h0_idx", "<i2"), ("snr", "i1"), ("ipass", "u1"), ("ap", "u1"), ("method", "u1"),
                          ("ttweak", "i1"), ("ftweak", "i1"), ("nsync", "u1"), ("emitted", "u1"), ("n_its", "<u2"),
                          ("score", "<f4"), ("tsec", "<f4"), ("fHz", "<f4"), ("grid_sd", "<f4"), ("fine_sd", "<f4"),
                          ("reserved", "<u4", (3,))], align=True)
assert RECORD_DTYPE.itemsize == C.sizeof(Record) == 64

# name -> (restype, argtypes); every symbol declared in include/ft8_b200.h
_P = C.c_void_p
SIGNATURES = {
    "ft8_default_cfg": (None, [C.POINTER(Cfg)]),
    "ft8_create": (C.c_int, [C.c_int, C.POINTER(Cfg), C.POINTER(_P)]),
    "ft8_destroy": (None, [_P]),
    "ft8_last_error": (C.c_char_p, [_P]),
    "ft8_get_stats": (C.c_int, [_P, C.POINTER(Stats)]),
    "ft8_synchronize": (C.c_int, [_P]),
    "ft8_stream": (_P, [_P]),
    "ft8_last_kernel_ms": (C.c_int, [_P, C.c_int, C.POINTER(C.c_float)]),
    "ft8_spectrogram": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, C.c_int]),
    "ft8_hop_spectrum": (C.c_int, [_P, _P, C.c_int, _P, C.c_int]),
    "ft8_sync": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P, _P, C.c_int]),
    "ft8_llr": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, C.c_int]),
    "ft8_cycle_spectrum": (C.c_int, [_P, _P, C.c_int, C.c_int, _P, C.c_int]),
    "ft8_fine": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P, _P, C.c_int]),
    "ft8_ldpc": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, _P, C.c_int]),
    "ft8_osd": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, _P, C.c_int]),
    "ft8_crc14": (C.c_int, [_P, _P, C.c_int, _P, C.c_int]),
    "ft8_prefetch_audio": (C.c_int, [_P, _P, C.c_int, C.c_int]),
    "ft8_host_alloc": (C.c_int, [C.c_size_t, C.c_int, C.POINTER(_P)]),
    "ft8_host_free": (C.c_int, [_P]),
    "ft8_decode_cycles": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int]),
    "ft8_decode_cycles_live": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int]),
    "ft8_decode_cycles_live_seq": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, C.c_int]),
    "ft8_live_reset": (C.c_int, [_P]),
    "ft8_decode_cycles_stream": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int, _P, C.c_int, _P, _P]),
    "ft8_synth_cycles": (C.c_int, [_P, _P, _P, _P, _P, C.c_int, C.c_int, C.c_float, C.c_uint64, _P, C.c_int]),
    "ft8_debug_fft": (C.c_int, [_P, C.c_int, C.c_int, _P, _P, C.c_int]),
}

_lib = None


def load():
    """Load the CUDA library; raises RuntimeError when it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(pyft8_b200 has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)       # AttributeError here means the .so is stale
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib
