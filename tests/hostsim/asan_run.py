"""Runs the host build of the team kernels' phases (rollout teams of 4, act selection) under AddressSanitizer + UBSan:
every shared-memory index and every shift of the device source is exercised on the CPU (compute-sanitizer is not available on
the GPU pool).  Started by tests/test_hostsim.py::test_team_phases_under_sanitizers with libasan preloaded; argv[1] = the .so."""
import sys, ctypes as C, numpy as np
import os
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'tests'))
from oracle import loader as O
from conftest import harvest_positions
H = C.CDLL(sys.argv[1]); P = C.c_void_p
H.hs_team_rollout.argtypes = [C.c_int, P, C.c_long, C.c_uint64, C.c_uint64, C.c_int, P, P]
H.hs_act_team.argtypes = [P, C.c_long, C.c_uint64, C.c_uint64, P, C.c_uint32, P]
mid = harvest_positions(O, 200, 5, 41, seed=5)
for recs in (O.new_envs(300), mid):
    b = recs.copy(); tr = np.zeros((260, len(b)), O.TRACE_DTYPE); st = np.zeros(1, O.STATS_DTYPE)
    assert H.hs_team_rollout(4, b.ctypes.data, len(b), 5, 9, 260, tr.ctypes.data, st.ctypes.data) == 0
q = np.random.default_rng(1).uniform(-0.3, 0.3, (len(mid), 96)).astype(np.float32)
got = np.zeros(len(mid), np.uint16)
assert H.hs_act_team(mid.ctypes.data, len(mid), 0, 1, q.ctypes.data, 1 << 28, got.ctypes.data) == 0
print("asan/ubsan clean")
