"""Multi-GPU check of parallel.sharded_rollout on real hardware (launch with torchrun, >= 2 ranks): the transitions gathered
from the shards -- through the peer-memory push (csrc/peer.cu) and through the NCCL padded all-gather -- must equal what a
single GPU produces for the same global start states (parallel.self_check), with real terminations and a real filter.
`nccl_check.py pen` runs the same check at Adroit's pen shape in the bf16x2_t64 mode."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch, torch.distributed as dist

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
from mobody_b200 import parallel as P
from helpers import cuda_agent, cuda_dynamics, cuda_module

if sys.argv[1:] == ["pen"]:   # Adroit's pen (S45/A24) in bf16x2_t64, the 64-row tensor-core mode; its predicate fires on part of the rows
    import mobody_b200 as mb
    S, A = 45, 24
    m, _ = cuda_module(S, A, 21, "halfcheetah", t3_gain=2.0)
    with torch.no_grad():
        m.transition3.bias[..., 26] += 0.16
    dyn = mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, m, None, None,
                                    mb.get_termination_fn("pen-human-v0"), penalty_coef=5.0, precision="bf16x2_t64")
    env_filter = 1e9
else:
    S, A = 17, 6
    dyn, _ = cuda_dynamics(S, A, 21, "walker2d", 5.0, precision="bf16x2", h0=1.0, t3_gain=6.0)
    env_filter = 0.78
dyn.seed = 5
ag, _ = cuda_agent(S, A, 21, env_filter=env_filter)
ag.dynamics = dyn
res = P.self_check(ag, 10_007, rounds=6)                      # 10 007: not divisible by the world size
if rank == 0:
    print("NCCL_CHECK", "OK" if res["ok"] else "FAILED", res)
dist.destroy_process_group()
sys.exit(0 if res["ok"] else 1)
