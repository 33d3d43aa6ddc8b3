"""CPU reference of policy evaluation in the learned model (mobody_model_eval), built on the oracle's step and policy forward
(test infrastructure).  The quantity is the one the reference's evaluators print (train_mobody.py:53-205): the sum of the
step rewards up to and including the first done step, one episode per start state."""
import numpy as np
import torch

from oracle import mobody_oracle as M
from oracle.philox import rollout_elite_slot, rollout_noise


@torch.no_grad()
def model_return(dyn_p, pol_p, max_action, init_obs, H, gamma, seed, step0, row0, term_kind, penalty_coef,
                 use_penalty=False, use_trg=True, record=False):
    """Episode returns of the deterministic policy in the learned dynamics with the production Philox draws: step t of the
    row with global id row0 + i uses the noise and elite pick keyed on (seed, step0 + t, row0 + i).  A row keeps the reward
    of the step whose next state is terminal and then stops; survivors keep their order.  Runs in the dtype of the
    parameters (float64 parameters -> float64 rollout).  Accumulates in float64, in step order, like the device:
    ret += r, ret_disc += disc * r, disc *= gamma after every step.
    Returns dict(returns, discounted_returns, lengths, counts[H+1]); with ``record``, also ``trace``: per step the global
    ids of the live rows and their next states (the termination inputs)."""
    dt = dyn_p["zs1.weight"].dtype
    obs = torch.as_tensor(np.asarray(init_obs)).to(dt)
    B, S = obs.shape
    A = pol_p["network.network.4.bias"].shape[0]
    elites = np.asarray(dyn_p["elites"])
    ids = np.arange(B, dtype=np.int64)                                        # local ids: global id = row0 + id
    ret, ret_disc = np.zeros(B), np.zeros(B)
    length, counts = np.zeros(B, np.int32), np.zeros(H + 1, np.int32)
    trace, disc = [], 1.0
    for t in range(H):
        counts[t] = len(ids)
        if len(ids) == 0:
            continue
        g = (row0 + ids).astype(np.uint64)
        members = elites[rollout_elite_slot(seed, step0 + t, g, len(elites))]
        eps = torch.zeros(M.E_MEMBERS, len(ids), S, dtype=dt)
        eps[members, np.arange(len(ids))] = torch.from_numpy(rollout_noise(seed, step0 + t, g, S)).to(dt)
        act = M.policy_forward(pol_p, obs, max_action).reshape(-1, A)
        r = M.step(dyn_p, obs, act, eps, members, term_kind, penalty_coef, use_penalty, use_trg)
        rew = r["reward"].reshape(-1).numpy().astype(np.float64)
        ret[ids] += rew
        ret_disc[ids] += disc * rew
        length[ids] = t + 1
        if record:
            trace.append((row0 + ids, r["next_obs"].numpy().copy()))
        alive = ~r["terminal"].reshape(-1)
        ids, obs = ids[alive], r["next_obs"][torch.from_numpy(alive)]
        disc *= gamma
    counts[H] = len(ids)
    out = dict(returns=ret, discounted_returns=ret_disc, lengths=length, counts=counts)
    if record:
        out["trace"] = trace
    return out
