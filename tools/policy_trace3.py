"""Phase timeline of the three-chain tcgen05 policy kernel (library built with -DQS_TC_TRACE):
    QS_LIB_TAG=trace QS_NVCC_DEFINES="-DQS_TC_TRACE" python -m rl_aerial_manipulator_b200._build
    QS_LIB_PATH=.../lib/libquadsim_trace.so python tools/policy_trace3.py
Threads 0 (MMA issuer warp) and 32 of the three groups of CTA 0, fourth tile: clock64 stamps relative to the earliest."""
import ctypes as C, os, sys
sys.path.insert(0, os.getcwd())
import numpy as np, torch
from rl_aerial_manipulator_b200.policy import MlpPolicyKernel
from rl_aerial_manipulator_b200._cabi import load_library
n = 1 << 20
g = torch.Generator(device="cuda").manual_seed(0)
obs = torch.randn((n, 20), device="cuda", generator=g) * 0.7
noise = torch.randn((n, 4), device="cuda", generator=g)
pol = MlpPolicyKernel.from_npz("tests/golden/policy_v2.npz", device="cuda", impl="tensor_fast")
for _ in range(3): pol.forward(obs, noise)
torch.cuda.synchronize()
lib = load_library()
buf = np.zeros((3, 2, 80), np.int64)
assert lib.qs_policy_debug_trace3(buf.ctypes.data_as(C.c_void_p)) == 0
names = ["start"]
for net in range(2):
    for ph in ("L1a", "L2a+L1b", "L2b", "L3"):
        names += [f"n{net} {ph} issued", f"n{net} {ph} mma-done", f"n{net} {ph} epi-done", f"n{net} {ph} synced"]
t0 = buf[buf > 0].min()
print(f"{'event':22s} " + " ".join(f"g{g}t{t*32:<3d}       " for g in range(3) for t in range(2)))
for i, nm in enumerate(names):
    print(f"{nm:22s} " + " ".join(f"{int(buf[g, t, i] - t0):6d} ({int(buf[g, t, i] - buf[g, t, i - 1]) if i else 0:5d})" for g in range(3) for t in range(2)))
