"""Debug aid: per-(layer, tile) timeline (clock64) of CTA 0 of the two-tiles-per-CTA step kernel (step_duo.cu), which
runs the fp16 precision mode."""
import sys, os, ctypes
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
from helpers import cuda_dynamics, cuda_agent
from mobody_b200 import _ffi
from mobody_b200.dynamics import StepWorkspace

prec = sys.argv[1] if len(sys.argv) > 1 else "fp16"
B = int(sys.argv[2]) if len(sys.argv) > 2 else 256 * 148
S, A = 17, 6
dyn, p = cuda_dynamics(S, A, 1, "halfcheetah", 5.0, precision=prec)
ag, _ = cuda_agent(S, A, 1)
obs = torch.randn(B, S, device="cuda") * 0.3
ws = StepWorkspace(B, S, A, "cuda", want_act=True)
NL = 73
trace = torch.zeros(NL * 2 * 8, dtype=torch.int64, device="cuda")
L = _ffi.lib()
for it in range(3):
    dyn.launch_step(obs, None, ws, policy=ag.policy.network, max_action=1.0, step=it)
torch.cuda.synchronize()
L.mobody_debug_set_trace(ctypes.c_void_p(trace.data_ptr()))
dyn.launch_step(obs, None, ws, policy=ag.policy.network, max_action=1.0, step=9)
torch.cuda.synchronize()
L.mobody_debug_set_trace(None)
t = trace.cpu().numpy().reshape(NL * 2, 8)
t0 = t[0, 0]
names = ["P1", "P2", "P3"] + sum([[f"{e}.zs1", f"{e}.zs2", f"{e}.zs3", f"{e}.za1", f"{e}.za2", f"{e}.t1", f"{e}.t2", f"{e}.t3"] for e in range(7)], []) + sum([[f"{e}.r1", f"{e}.r2"] for e in range(7)], [])
print("unit        mma_start first_issue mma_end | L:epi_wait  L:d_full  L:epi_end | P:epi_wait P:d_full P:epi_end")
for i in range(NL * 2):
    r = t[i] - t0
    print(f"{names[i // 2]:6s}{'XY'[i & 1]} {r[0]:9d} {r[1]:9d} {r[2]:9d} | {r[3]:9d} {r[4]:9d} {r[5]:9d} | {r[6]:9d} {r[7]:9d}")
print("total cycles", t[NL * 2 - 1, 5] - t0)
