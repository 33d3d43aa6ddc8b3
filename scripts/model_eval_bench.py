#!/usr/bin/env python
"""Benchmark of policy evaluation in the learned model (MOBODY.evaluate_in_model / mobody_model_eval); prints one JSON line.

  no_termination: 100 000 start states, S17/A6, a termination predicate that never fires (MOBODY_TERM_NEVER), H = 1 000,
                  bf16x2: ms per step and transitions/s of the whole call (CUDA events around the public API call, host
                  read included), next to a single-stream mobody_rollout with T = 1 over the same 100 000 states, the two
                  alternated in the same run.  Also times the same evaluation split into two halves on the two
                  rollout_streams() (separate workspaces), the candidate for filling the step kernel's tail round.
  termination:    hopper S11/A3, H = 1 000, 100 000 start states whose rows end at different steps: the live-row curve and
                  the total time, the tail after most rows ended included.
  dead_steps:     per-step cost once every row has ended (all 100 000 rows end at step 0, 999 steps follow).
The card's name and power limit are read in the same run.  Weights are the reference module's own random initialiser.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402
import torch  # noqa: E402

CFG = dict(max_action=1.0, hidden_sizes=256, gamma=0.99, tau=0.005, actor_lr=3e-4, critic_lr=3e-4, weight=2.5,
           bc_coef=1.0, penalty_type="none", filter_bad_rollout=1, env_filter=1e9)


def make_agent(mb, S, A, task, dev, h0=None, gain=1.0, seed=3):
    torch.manual_seed(seed)
    model = mb.MOBODYModule(S, A, 256, 7, 5, device=dev, config={"mopo": 0, "latent_reward": 0})
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if name.endswith(".bias"):
                prm.normal_(0.0, 0.1)
        if h0 is not None:                                       # decoder bias in the healthy set, rows end at different steps
            model.transition3.weight.mul_(gain)
            model.transition3.bias.mul_(0.1)
            model.transition3.bias[:, :, 0] += h0
    dyn = mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, model, None, None,
                                    mb.get_termination_fn(task), penalty_coef=1.0, precision="bf16x2")
    ag = mb.MOBODY(dict(CFG, state_dim=S, action_dim=A), dev)
    ag.dynamics = dyn
    return ag


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True).stdout.strip().split(", ")
    return {"name": q[0], "power_limit_w": float(q[1])} if len(q) == 2 else {"name": torch.cuda.get_device_name(0), "power_limit_w": None}


def timed(fn, reps=1):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def split2(ag, obs, H):
    """The evaluation as two halves on the two rollout streams, each with its own workspace (per-start results are the same)."""
    cur = torch.cuda.current_stream()
    ag.verify_images(True)
    B, outs = obs.shape[0], []
    for k, (st, lo, hi) in enumerate(zip(ag.rollout_streams(), (0, B // 2), (B // 2, B))):
        st.wait_stream(cur)
        with torch.cuda.stream(st):
            outs.append(ag._launch_model_eval(obs[lo:hi], H, 0.99, False, True, lo, 0, ws_slot=k, verify_images=False))
    for st in ag.rollout_streams():
        cur.wait_stream(st)
    return outs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=100_000)
    ap.add_argument("--horizon", type=int, default=1000)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--rollout-reps", type=int, default=200)
    a = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    import mobody_b200 as mb
    dev, B, H = torch.device("cuda:0"), a.rows, a.horizon
    out = {"card": card(), "rows": B, "horizon": H}
    gen = torch.Generator(device=dev).manual_seed(0)

    # ---- no termination: S17/A6, MOBODY_TERM_NEVER ----
    ag = make_agent(mb, 17, 6, "halfcheetahvel", dev)
    obs = 0.3 * torch.randn(B, 17, generator=gen, device=dev)
    ag.evaluate_in_model(obs, 8, step0=0); split2(ag, obs, 8); ag.rollout_device(obs, 1, sync=False, step0=0)   # warm-up
    ev, sp, ro = [], [], []
    for _ in range(a.rounds):
        ev.append(timed(lambda: ag.evaluate_in_model(obs, H, step0=0)))
        sp.append(timed(lambda: split2(ag, obs, H)))
        ro.append(timed(lambda: ag.rollout_device(obs, 1, sync=False, step0=0), a.rollout_reps))
    res, info = ag.evaluate_in_model(obs, H, step0=0)
    halves = split2(ag, obs, H)
    torch.cuda.synchronize()
    same = all(torch.equal(res[k], torch.cat([h[0][k] for h in halves])) for k in res)
    ms_eval = [1e3 * t / H for t in ev]
    out["no_termination"] = {
        "workload": f"S17/A6 bf16x2, {B} start states, H={H}, MOBODY_TERM_NEVER",
        "eval_ms_per_step": [round(x, 4) for x in ms_eval],
        "eval_transitions_per_s": round(B * H / float(np.median(ev)), 0),
        "rollout_T1_ms": [round(1e3 * t, 4) for t in ro],
        "rollout_T1_transitions_per_s": round(B / float(np.median(ro)), 0),
        "eval_step_over_rollout_T1": round(float(np.median(ms_eval)) / (1e3 * float(np.median(ro))), 4),
        "two_streams_ms_per_step": [round(1e3 * t / H, 4) for t in sp],
        "two_streams_over_one": round(float(np.median(sp)) / float(np.median(ev)), 4),
        "two_streams_results_identical": bool(same),
        "all_live": info["live_per_step"] == [B] * (H + 1),
        "workspace_bytes": int(ag._eval_workspace(B, 17, 6).numel()),
    }

    # ---- every row ends at step 0 (humanoid's predicate x0 in (1, 2) fails at these states): cost of a dead step ----
    ag.dynamics.terminal_fn = mb.get_termination_fn("humanoid")
    ag.evaluate_in_model(obs, 8, step0=0)
    dead = [timed(lambda: ag.evaluate_in_model(obs, H, step0=0)) for _ in range(a.rounds)]
    _, dinfo = ag.evaluate_in_model(obs, H, step0=0)
    out["dead_steps"] = {"live_after_step0": dinfo["live_per_step"][1],
                         "us_per_step": [round(1e6 * t / H, 2) for t in dead]}

    # ---- termination: hopper S11/A3 ----
    hop = make_agent(mb, 11, 3, "hopper-medium-v2", dev, h0=0.8, gain=4.0)
    hobs = 0.2 * torch.randn(B, 11, generator=gen, device=dev)
    hobs[:, 0] += 1.25
    hop.evaluate_in_model(hobs, 8, step0=0)
    ht = [timed(lambda: hop.evaluate_in_model(hobs, H, step0=0, penalized=True)) for _ in range(a.rounds)]
    _, hinfo = hop.evaluate_in_model(hobs, H, step0=0, penalized=True)
    c = hinfo["live_per_step"]
    marks = [t for t in (0, 1, 2, 3, 5, 10, 20, 50, 100, 200, 500, H) if t <= H]
    out["termination"] = {
        "workload": f"hopper S11/A3 bf16x2, {B} start states, H={H}, penalized reward",
        "total_s": [round(t, 4) for t in ht],
        "live_per_step": {str(t): c[t] for t in marks},
        "first_step_below_1pct": next((t for t, n in enumerate(c) if n < B / 100), None),
        "first_step_zero": next((t for t, n in enumerate(c) if n == 0), None),
        "transitions": int(sum(c[:H])),
        "return_mean": hinfo["return_mean"], "length_mean": hinfo["length_mean"],
    }
    print(json.dumps(out))


if __name__ == "__main__":
    main()
