"""k_fscan_mma phase timing (library built with -DFS_PROFILE): clock64 sums per role/phase, per event."""
import ctypes as C, json, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np, torch
from pyft8_b200 import workload, _lib as L
from pyft8_b200.engine import Engine
B = int(sys.argv[1]) if len(sys.argv) > 1 else 1024
eng = Engine(max_cycles=B)
params = workload.make_params("cfg2_50sig", B, seed=2000)
audio = torch.empty((B, 180000), dtype=torch.int16, device="cuda:0")
workload.device_cycles(eng, params, audio.data_ptr())
torch.cuda.synchronize()
lib = C.CDLL(L.LIB_PATH)
buf = (C.c_ulonglong * 16)()
eng.decode_cycles_dev(audio.data_ptr(), L.AUDIO_I16, B)
lib.ft8_debug_fs_prof(buf, 1)
eng.decode_cycles_dev(audio.data_ptr(), L.AUDIO_I16, B)
lib.ft8_debug_fs_prof(buf, 0)
v = [int(x) for x in buf]
n_i, n_g, n_p = max(v[5], 1), max(v[9], 1), max(v[12], 1)
print(json.dumps({"issuer_per_chunk_clk": {"issue_b(wait free it-2)": v[0] / n_i, "wait acc_free": v[1] / n_i, "wait a_ready": v[2] / n_i,
                                            "wait b_full": v[3] / n_i, "mma issue+commit": v[4] / n_i, "chunks": n_i},
                  "generator_warp0_per_own_chunk_clk": {"issue next loads": v[6] / n_g, "wait stage free": v[7] / n_g, "compute+split+st+wait+arrive": v[8] / n_g, "chunks": n_g},
                  "generator_warp0_per_pass_clk": {"chunk loop": v[10] / n_p, "wait acc_ready": v[11] / n_p, "passes": n_p}}))
