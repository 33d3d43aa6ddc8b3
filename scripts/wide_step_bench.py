#!/usr/bin/env python
"""Benchmark of the wide tensor-core step mode (bf16x2_wide) against the fp32 CUDA-core kernel at Ant's shape; prints one
JSON line.

  rollout:    S111/A8, ant termination, 100 000 start states, T = 1 rollouts (MOBODY.rollout_device: one mobody_rollout
              call, policy fused), fp32 and bf16x2_wide alternated in the same run.  The start states rotate over a pool
              of buffers larger than the 126 MB L2, so every rollout reads them from HBM; every shape is warmed up first.
  kernel:     the step kernel alone (MOBODYEnsembleDynamics.launch_step, policy fused, CUDA events around many launches,
              same input rotation) and its algorithmic rate: 4 768 768 FLOP per transition at S111/A8 (SURVEY.md 8d).
  model_eval: MOBODY.evaluate_in_model, 100 000 start states, H = 1 000, a predicate that never fires (every step runs at
              full width), both modes.
  outputs:    the two modes' T = 1 rollouts of the same seeded start states and Philox key, compared element-wise.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

S, A = 111, 8
FLOP_PER_TRANSITION = 4_768_768
MODES = ("fp32", "bf16x2_wide")
CFG = dict(max_action=1.0, hidden_sizes=256, gamma=0.99, tau=0.005, actor_lr=3e-4, critic_lr=3e-4, weight=2.5,
           bc_coef=1.0, penalty_type="none", filter_bad_rollout=1, env_filter=1e9)


def make_agent(mb, prec, task, dev, seed=3):
    """Agent with the reference module's random initialiser (seeded: both modes get the same weights); transition3's
    bias puts x0 at 0.6, inside Ant's healthy range, so part of the rows terminate."""
    torch.manual_seed(seed)
    model = mb.MOBODYModule(S, A, 256, 7, 5, device=dev, config={"mopo": 0, "latent_reward": 0})
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if name.endswith(".bias"):
                prm.normal_(0.0, 0.1)
        model.transition3.bias[:, :, 0] += 0.6
    dyn = mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, model, None, None,
                                    mb.get_termination_fn(task), penalty_coef=1.0, precision=prec)
    torch.manual_seed(seed + 1)
    ag = mb.MOBODY(dict(CFG, state_dim=S, action_dim=A), dev)
    ag.dynamics = dyn
    return ag


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1])} if len(q) == 2 else {"name": torch.cuda.get_device_name(0), "power_limit_w": None}


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--horizon", type=int, default=1000)
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    import mobody_b200 as mb
    from mobody_b200.dynamics import StepWorkspace
    dev, B = torch.device("cuda:0"), a.rows
    if not torch.cuda.is_available():
        raise SystemExit("wide_step_bench: needs a CUDA device")
    out = {"card": card(), "rows": B, "shape": f"S{S}/A{A}", "flop_per_transition": FLOP_PER_TRANSITION}
    gen = torch.Generator(device=dev).manual_seed(0)
    n_pool = max(2, -(-160 * 1024 * 1024 // (B * S * 4)))
    pool = [0.2 * torch.randn(B, S, generator=gen, device=dev) for _ in range(n_pool)]
    for x in pool:
        x[:, 0] += 0.6
    ags = {p: make_agent(mb, p, "ant-medium-v2", dev) for p in MODES}
    wss = {p: StepWorkspace(B, S, A, dev, want_act=True) for p in MODES}
    it = [0]

    def nxt():
        it[0] += 1
        return pool[it[0] % n_pool]

    def rollout(p):
        return ags[p].rollout_device(nxt(), 1, sync=False, step0=0)

    def kernel(p):
        ag = ags[p]
        ag.dynamics.launch_step(nxt(), None, wss[p], policy=ag.policy.network, step=0, verify_images=False)

    for p in MODES:                                              # warm-up of every shape and both paths
        for _ in range(3):
            rollout(p)
        ags[p].dynamics.launch_step(pool[0], None, wss[p], policy=ags[p].policy.network, step=0)
        kernel(p)
    torch.cuda.synchronize()
    ro = {p: [] for p in MODES}
    kt = {p: [] for p in MODES}
    for _ in range(a.rounds):
        for p in MODES:
            ro[p].append(timed(lambda: rollout(p), a.reps))
            kt[p].append(timed(lambda: kernel(p), a.reps))
    res = {}
    for p in MODES:
        r, k = float(np.median(ro[p])), float(np.median(kt[p]))
        res[p] = {"rollout_T1_ms": [round(1e3 * t, 3) for t in ro[p]], "rollout_transitions_per_s": round(B / r, 0),
                  "kernel_ms": [round(1e3 * t, 3) for t in kt[p]], "kernel_transitions_per_s": round(B / k, 0),
                  "kernel_tflops": round(FLOP_PER_TRANSITION * B / k * 1e-12, 2)}
    res["speedup_rollout"] = round(res["bf16x2_wide"]["rollout_transitions_per_s"] / res["fp32"]["rollout_transitions_per_s"], 2)
    res["speedup_kernel"] = round(res["bf16x2_wide"]["kernel_transitions_per_s"] / res["fp32"]["kernel_transitions_per_s"], 2)
    out["rollout"] = res

    # ---- the same seeded start states and Philox key through both modes: outputs side by side ----
    from helpers import rel_err, rel_err_strict
    got = {}
    for p in MODES:
        _, info = ags[p].rollout_device(pool[0], 1, step0=0)
        ws = ags[p]._rollout_workspace(1, B, S, A, 0)
        got[p] = {"next_obs": ws["nexts"][0].cpu().numpy(), "reward": ws["rews"][0].cpu().numpy(),
                  "terminal": ws["terms"][0].cpu().numpy(), "kept": info["kept"]}
    w, f = got["bf16x2_wide"], got["fp32"]
    out["outputs"] = {k: {"rel_err": rel_err(w[k], f[k]), "rel_err_strict": rel_err_strict(w[k], f[k])} for k in ("next_obs", "reward")}
    out["outputs"]["terminal_mismatches"] = int((w["terminal"] != f["terminal"]).sum())
    out["outputs"]["terminal_rows"] = int(f["terminal"].sum())
    out["outputs"]["kept"] = [w["kept"], f["kept"]]

    # ---- evaluate_in_model, H = 1000, every row live throughout ----
    ev = {}
    for p in MODES:
        ag = make_agent(mb, p, "halfcheetahvel", dev)
        ag.evaluate_in_model(pool[0], 8, step0=0)
        ts = [timed(lambda: ag.evaluate_in_model(pool[0], a.horizon, step0=0), 1) for _ in range(2)]
        ev[p] = {"total_s": [round(t, 3) for t in ts], "transitions_per_s": round(B * a.horizon / min(ts), 0)}
    ev["speedup"] = round(ev["bf16x2_wide"]["transitions_per_s"] / ev["fp32"]["transitions_per_s"], 2)
    out["model_eval"] = dict(ev, workload=f"S{S}/A{A}, {B} start states, H={a.horizon}, predicate never fires")
    print(json.dumps(out))


if __name__ == "__main__":
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    main()
