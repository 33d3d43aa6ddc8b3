#!/usr/bin/env python
"""Benchmark of the 64-row tensor-core step modes at Adroit's shapes (bf16x2_t64, and fp16_t64: fp16's arithmetic on the
same tiles) against the fp32 CUDA-core kernel; prints one JSON line.  Speedups are against fp32, and fp16_t64's also
against bf16x2_t64.

  rollout:    pen S45/A24, door S39/A28, relocate S39/A30 and hammer S46/A26, 100 000 start states, T = 1 rollouts
              (MOBODY.rollout_device: one mobody_rollout call, policy fused), fp32, bf16x2_t64 and fp16_t64 alternated in
              the same run.  pen uses its predicate (part of the rows terminate); door's predicate never fires, and relocate and
              hammer have none in the reference, so they run with the never-firing one.  The start states rotate over a
              pool of buffers larger than the 126 MB L2, so every rollout reads them from HBM; every shape is warmed up first.
  kernel:     the step kernel alone (MOBODYEnsembleDynamics.launch_step, policy fused, CUDA events around many launches,
              same input rotation) and its algorithmic rate, 2 [7 (dyn + rew) + policy] FLOP per transition (SURVEY.md 8d):
              3 861 504 at pen.
  outputs:    each tensor-core mode's T = 1 rollout of the same seeded start states and Philox key against fp32's,
              compared element-wise.
  model_eval: at pen, MOBODY.evaluate_in_model, 100 000 start states, H = 1 000, a predicate that never fires (every step
              runs at full width), every mode.
  train:      at pen, MOBODY.train updates/s at batch 128 with penalty_type="par" (one 128-row dynamics step inside every
              update), every mode alternated.
The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

from helpers import AGENT_CFG, rel_err, rel_err_strict  # noqa: E402

SHAPES = {"pen": (45, 24, "pen-human-v0"), "door": (39, 28, "door-human-v0"), "relocate": (39, 30, "door-human-v0"),
          "hammer": (46, 26, "door-human-v0")}
MODES = ("fp32", "bf16x2_t64", "fp16_t64")
PAIRS = (("bf16x2_t64", "fp32"), ("fp16_t64", "fp32"), ("fp16_t64", "bf16x2_t64"))
CFG = dict(AGENT_CFG, env_filter=1e9)
PEN_X = 0.16   # transition3's bias puts the pen's object height (column 26) here: part of the rows fall below 0.075


def flop_per_transition(S, A, H=256, E=7):
    dyn = S * H + H * H + 32 * H + (16 + A) * 32 + 32 * 32 + 16 * H + H * H + H * S
    rew = (2 * S + A) * H + H * H + 2 * H
    return 2 * (E * (dyn + rew) + S * H + H * H + H * A)


def make_agent(mb, prec, S, A, task, dev, seed=3, **cfg):
    """Agent with the reference module's random initialiser (seeded: every mode gets the same weights)."""
    torch.manual_seed(seed)
    model = mb.MOBODYModule(S, A, 256, 7, 5, device=dev, config={"mopo": 0, "latent_reward": 0})
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if name.endswith(".bias"):
                prm.normal_(0.0, 0.1)
        if task.startswith("pen"):
            model.transition3.bias[:, :, 26] += PEN_X
    dyn = mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, model, None, None,
                                    mb.get_termination_fn(task), penalty_coef=1.0, precision=prec)
    torch.manual_seed(seed + 1)
    ag = mb.MOBODY(dict(CFG, state_dim=S, action_dim=A, **cfg), dev)
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


def bench_shape(mb, env, a, dev):
    from mobody_b200.dynamics import StepWorkspace
    S, A, task = SHAPES[env]
    B, fpt = a.rows, flop_per_transition(S, A)
    gen = torch.Generator(device=dev).manual_seed(0)
    n_pool = max(2, -(-160 * 1024 * 1024 // (B * S * 4)))
    pool = [0.2 * torch.randn(B, S, generator=gen, device=dev) for _ in range(n_pool)]
    if env == "pen":
        for x in pool:
            x[:, 26] += PEN_X
    ags = {p: make_agent(mb, p, S, A, task, dev) for p in MODES}
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

    for p in MODES:                                              # warm-up of every shape and every path
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
    res = {"shape": f"S{S}/A{A}", "termination": task.split("-")[0] if env in ("pen", "door") else "none (never fires)",
           "flop_per_transition": fpt}
    for p in MODES:
        r, k = float(np.median(ro[p])), float(np.median(kt[p]))
        res[p] = {"rollout_T1_ms": [round(1e3 * t, 3) for t in ro[p]], "rollout_transitions_per_s": round(B / r, 0),
                  "kernel_ms": [round(1e3 * t, 3) for t in kt[p]], "kernel_transitions_per_s": round(B / k, 0),
                  "kernel_tflops": round(fpt * B / k * 1e-12, 2)}
    for p, base in PAIRS:
        res[f"speedup_rollout_{p}_vs_{base}"] = round(res[p]["rollout_transitions_per_s"] / res[base]["rollout_transitions_per_s"], 2)
        res[f"speedup_kernel_{p}_vs_{base}"] = round(res[p]["kernel_transitions_per_s"] / res[base]["kernel_transitions_per_s"], 2)
    # the same seeded start states and Philox key through every mode: outputs side by side
    got = {}
    for p in MODES:
        _, info = ags[p].rollout_device(pool[0], 1, step0=0)
        ws = ags[p]._rollout_workspace(1, B, S, A, 0)
        got[p] = {"next_obs": ws["nexts"][0].cpu().numpy(), "reward": ws["rews"][0].cpu().numpy(),
                  "terminal": ws["terms"][0].cpu().numpy(), "kept": info["kept"]}
    f = got["fp32"]
    res["outputs"] = {"terminal_rows_fp32": int(f["terminal"].sum()), "kept_fp32": f["kept"]}
    for p in MODES[1:]:
        w = got[p]
        o = {k: {"rel_err": rel_err(w[k], f[k]), "rel_err_strict": rel_err_strict(w[k], f[k])} for k in ("next_obs", "reward")}
        o["terminal_mismatches"] = int((w["terminal"] != f["terminal"]).sum())
        o["kept"] = w["kept"]
        res["outputs"][f"{p}_vs_fp32"] = o
    del pool, ags, wss
    torch.cuda.empty_cache()
    return res


def bench_model_eval(mb, a, dev):
    S, A, _ = SHAPES["pen"]
    B = a.rows
    x0 = 0.2 * torch.randn(B, S, generator=torch.Generator(device=dev).manual_seed(1), device=dev)
    ev = {}
    for p in MODES:
        ag = make_agent(mb, p, S, A, "door-human-v0", dev)
        ag.evaluate_in_model(x0, 8, step0=0)
        ts = [timed(lambda: ag.evaluate_in_model(x0, a.horizon, step0=0), 1) for _ in range(2)]
        ev[p] = {"total_s": [round(t, 3) for t in ts], "transitions_per_s": round(B * a.horizon / min(ts), 0)}
    for p, base in PAIRS:
        ev[f"speedup_{p}_vs_{base}"] = round(ev[p]["transitions_per_s"] / ev[base]["transitions_per_s"], 2)
    ev["workload"] = f"S{S}/A{A}, {B} start states, H={a.horizon}, predicate never fires"
    return ev


def bench_train(mb, a, dev):
    S, A, _ = SHAPES["pen"]
    rng = np.random.default_rng(4)

    def ds(n):
        hs = np.zeros(S, np.float32)
        hs[26] = PEN_X
        return dict(observations=(hs + 0.2 * rng.standard_normal((n, S))).astype(np.float32),
                    actions=rng.uniform(-1, 1, (n, A)).astype(np.float32),
                    next_observations=(hs + 0.2 * rng.standard_normal((n, S))).astype(np.float32),
                    rewards=rng.standard_normal(n).astype(np.float32), terminals=np.zeros(n, bool))
    src, tar = mb.ReplayBuffer(S, A, "cuda"), mb.ReplayBuffer(S, A, "cuda")
    src.convert_D4RL(ds(200_000)); tar.convert_D4RL(ds(20_000))
    ags = {p: make_agent(mb, p, S, A, "pen-human-v0", dev, penalty_type="par", penalty_coef=0.1, env_filter=10.0) for p in MODES}
    for p in MODES:                       # the first call refreshes the synthetic buffer; then warm up the update
        for _ in range(20):
            ags[p].train(src, tar, 128, None, None)
    tt = {p: [] for p in MODES}
    for _ in range(a.rounds):
        for p in MODES:
            tt[p].append(timed(lambda: ags[p].train(src, tar, 128, None, None), a.train_steps))
    tr = {p: {"updates_per_s": [round(1.0 / t, 0) for t in tt[p]]} for p in MODES}
    for p, base in PAIRS:
        tr[f"speedup_{p}_vs_{base}"] = round(float(np.median(tt[base]) / np.median(tt[p])), 2)
    tr["workload"] = f"S{S}/A{A}, batch 128, penalty_type='par' (a 128-row dynamics step in every update)"
    return tr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--horizon", type=int, default=1000)
    ap.add_argument("--train-steps", type=int, default=500)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("adroit_step_bench: needs a CUDA device")
    import __graft_entry__ as g
    g.build()
    import mobody_b200 as mb
    dev = torch.device("cuda:0")
    out = {"card": card(), "rows": a.rows}
    out["rollout"] = {}
    for env in a.shapes.split(","):
        out["rollout"][env] = bench_shape(mb, env, a, dev)
        print(json.dumps({env: out["rollout"][env]}), file=sys.stderr, flush=True)
    out["model_eval_pen"] = bench_model_eval(mb, a, dev)
    out["train_pen"] = bench_train(mb, a, dev)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
