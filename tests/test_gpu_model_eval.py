"""GPU checks of policy evaluation in the learned model (mobody_model_eval / MOBODY.evaluate_in_model): parity with the
float64 oracle, bit equality with the per-start sums of mobody_rollout's transitions, independence from batching,
long horizons, isolation from the training draws and the evaluator wrapper."""
import numpy as np
import pytest
import torch

from helpers import cuda_agent, cuda_dynamics, healthy, rel_err_strict
from model_eval_oracle import model_return

pytestmark = pytest.mark.gpu

COEF = 5.0
# (env, S, A, h0, t3_gain, termination kind, penalized): hopper rows end at different steps (about 20 % of the live rows per
# step at first); halfcheetah's predicate (|x| >= 100) never fires at these states, so its returns run the whole horizon
CASES = [("hopper", 11, 3, 0.8, 2.0, 2, True), ("halfcheetah", 17, 6, None, 1.0, 1, False)]
MARGIN = 1e-4      # rows whose termination input came this close to a threshold may end one step apart in fp32 arithmetic


def _agent(env, S, A, prec, h0=None, t3=1.0, seed=3):
    dyn, p = cuda_dynamics(S, A, seed, env, COEF, precision=prec, h0=h0, t3_gain=t3)
    ag, st = cuda_agent(S, A, seed, env_filter=1e9)
    ag.dynamics = dyn
    return ag, p, st


def _starts(env, S, B, h0=None, seed=1):
    return (healthy(env, S, h0)[None] + 0.1 * np.random.default_rng(seed).standard_normal((B, S))).astype(np.float32)


def _term_distance(env, x):
    """Distance of each next state to its termination predicate's thresholds (terminal_funs.py)."""
    if env == "hopper":
        return np.minimum(np.minimum(np.abs(x[:, 0] - 0.7), np.abs(np.abs(x[:, 1]) - 0.2)), 100.0 - x[:, 1:].max(1))
    return 100.0 - np.abs(x).max(1)


@pytest.mark.parametrize("prec", ["fp32", "bf16x2"])
@pytest.mark.parametrize("env,S,A,h0,t3,kind,penalized", CASES, ids=[c[0] for c in CASES])
def test_returns_match_float64_oracle(env, S, A, h0, t3, kind, penalized, prec):
    check_against_float64_oracle(env, S, A, h0, t3, kind, penalized, prec, row0=1000, step0=7)


def check_against_float64_oracle(env, S, A, h0, t3, kind, penalized, prec, row0, step0, H=24):
    """Per-start returns, discounted returns and lengths of evaluate_in_model against the float64 reference."""
    ag, p, st = _agent(env, S, A, prec, h0, t3)
    B, gamma = 300, 0.99                                                     # 300 rows: the last 128-row tile is ragged
    obs = _starts(env, S, B, h0)
    res, info = ag.evaluate_in_model(torch.from_numpy(obs).cuda(), H, gamma=gamma, penalized=penalized, row0=row0, step0=step0)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in st.policy.items()}
    ref = model_return(p64, pol64, 1.0, obs.astype(np.float64), H, gamma, ag.eval_seed, step0, row0, kind, COEF,
                         use_penalty=penalized, record=True)
    dist = np.full(B, np.inf)
    for ids, x in ref["trace"]:
        dist[ids - row0] = np.minimum(dist[ids - row0], _term_distance(env, x))
    near = dist < MARGIN
    assert near.mean() < 0.05, near.mean()
    got = {k: v.cpu().numpy() for k, v in res.items()}
    assert np.array_equal(got["lengths"][~near], ref["lengths"][~near])
    assert info["live_per_step"] == ref["counts"].tolist() or near.any()
    worst = 0.0
    for k in ("returns", "discounted_returns"):
        err = rel_err_strict(got[k][~near], ref[k][~near])
        assert err < 1e-4, (k, err)
        worst = max(worst, err / 1e-4)
    if kind == 2:
        assert 0 < ref["counts"][H] < B and len(set(ref["lengths"].tolist())) > 5
    print(f"\n[model eval parity] {env} {prec} row0={row0} step0={step0}: worst err/bound {worst:.3f}, {int(near.sum())}/{B} rows within {MARGIN} of a "
          f"termination threshold excluded, lengths {ref['lengths'].min()}..{ref['lengths'].max()}")


@pytest.mark.parametrize("prec", ["bf16x2", "fp32"])
def test_bit_exact_against_rollout_transitions(prec):
    """mobody_rollout with T = H, the same Philox key / step0 / row0, no filter, penalized reward: per-start float64 sums of its
    workspace rewards in step order equal the evaluator's outputs bit for bit, and the live counts agree."""
    ag, p, st = _agent("hopper", 11, 3, prec, 0.8, 2.0)
    ag.config["filter_bad_rollout"] = 0
    B, H, row0, step0, gamma, S, A = 333, 5, 77, 40, 0.9, 11, 3
    obs = torch.from_numpy(_starts("hopper", S, B, 0.8, seed=4)).cuda()
    res, info = ag.evaluate_in_model(obs, H, gamma=gamma, penalized=True, row0=row0, step0=step0)
    seed = ag.dynamics.seed
    ag.dynamics.seed = ag.eval_seed
    try:
        _, ri = ag.rollout_device(obs, H, row0=row0, step0=step0)
    finally:
        ag.dynamics.seed = seed
    ws = ag._rollout_workspace(H, B, S, A, 0)
    counts, rews = ws["counts"].cpu().numpy(), ws["rews"][:, :, 0].cpu().numpy()
    terms, ids = ws["terms"].cpu().numpy(), ws["row_ids"].cpu().numpy()
    ret, ret_disc, length = np.zeros(B), np.zeros(B), np.zeros(B, np.int32)
    disc = 1.0
    for t in range(H):
        n = counts[t]
        i = ids[t, :n] - row0
        r = rews[t, :n].astype(np.float64)
        ret[i] += r
        ret_disc[i] += disc * r
        length[i] = t + 1
        disc *= gamma
    assert info["live_per_step"][:H] == ri["rows_per_step"] == counts[:H].tolist()
    assert info["live_per_step"][H] == int(counts[H - 1] - terms[H - 1, :counts[H - 1]].sum())
    assert 0 < info["live_per_step"][H] < counts[1] < B                    # rows really ended inside the horizon
    assert np.array_equal(res["lengths"].cpu().numpy(), length)
    assert np.array_equal(res["returns"].cpu().numpy(), ret)
    assert np.array_equal(res["discounted_returns"].cpu().numpy(), ret_disc)


def test_chunk_invariance_and_determinism():
    ag, _, _ = _agent("hopper", 11, 3, "bf16x2", 0.8, 2.0)
    B, H = 300, 30
    obs = torch.from_numpy(_starts("hopper", 11, B, 0.8, seed=6)).cuda()
    full, fi = ag.evaluate_in_model(obs, H, step0=3, penalized=True)
    cuts = [0, 101, 250, B]
    parts = [ag.evaluate_in_model(obs[lo:hi].contiguous(), H, row0=lo, step0=3, penalized=True)[0] for lo, hi in zip(cuts[:-1], cuts[1:])]
    again, ai = ag.evaluate_in_model(obs, H, step0=3, penalized=True)
    assert fi == ai and 0 < fi["live_per_step"][H] < B
    for k in full:
        assert torch.equal(full[k], again[k]), k
        assert torch.equal(full[k], torch.cat([q[k] for q in parts])), k


def test_long_horizon_without_termination():
    """1 000 steps of 20 000 start states with a termination predicate that never fires (MOBODY_TERM_NEVER)."""
    import mobody_b200 as mb
    ag, _, _ = _agent("halfcheetah", 17, 6, "bf16x2")
    ag.dynamics.terminal_fn = mb.get_termination_fn("halfcheetahvel")
    assert ag.dynamics.terminal_fn.kind == 0
    B, H = 20_000, 1000
    res, info = ag.evaluate_in_model(torch.from_numpy(_starts("halfcheetah", 17, B)).cuda(), H)
    assert info["live_per_step"] == [B] * (H + 1)
    assert bool((res["lengths"] == H).all()) and info["length_mean"] == H
    assert bool(torch.isfinite(res["returns"]).all()) and bool(torch.isfinite(res["discounted_returns"]).all())
    assert abs(info["return_mean"] - float(res["returns"].mean())) <= 1e-12 * abs(info["return_mean"])


def test_long_horizon_with_termination():
    ag, _, _ = _agent("hopper", 11, 3, "bf16x2", 0.8, 2.0)
    B, H = 2000, 1000
    res, info = ag.evaluate_in_model(torch.from_numpy(_starts("hopper", 11, B, 0.8)).cuda(), H, penalized=True)
    c = np.array(info["live_per_step"])
    assert c[0] == B and np.all(np.diff(c) <= 0) and c[-1] < B // 2
    lengths = res["lengths"].cpu().numpy()
    assert lengths.min() >= 1 and lengths.max() <= H
    assert int(lengths.sum()) == int(c[:H].sum())
    assert int((lengths == H).sum()) == int(c[H])


def test_evaluation_leaves_training_draws_alone():
    """Two identical agents: one evaluates before its rollout, the other does not.  The rollouts are bit-identical, the
    training draw counter does not move, and each evaluation call draws fresh noise from its own counter."""
    obs = torch.from_numpy(_starts("hopper", 11, 500, 0.8, seed=8)).cuda()
    a, _, _ = _agent("hopper", 11, 3, "bf16x2", 0.8, 2.0)
    b, _, _ = _agent("hopper", 11, 3, "bf16x2", 0.8, 2.0)
    a.rollout_device(obs, 2)
    b.rollout_device(obs, 2)
    draw = a.dynamics._draw
    e1, _ = a.evaluate_in_model(obs, 40)
    e2, _ = a.evaluate_in_model(obs, 40)
    assert a.dynamics._draw == draw and a._eval_draw == 80
    assert not torch.equal(e1["returns"], e2["returns"])
    ra, ia = a.rollout_device(obs, 3)
    rb, ib = b.rollout_device(obs, 3)
    assert ia["kept"] == ib["kept"] and torch.equal(ia["packed"][:ia["kept"]], ib["packed"][:ib["kept"]])


def test_eval_policy_in_model_reports_the_mean_return(capsys):
    import mobody_b200 as mb
    ag, _, _ = _agent("hopper", 11, 3, "bf16x2", 0.8, 2.0)
    obs = torch.from_numpy(_starts("hopper", 11, 300, 0.8, seed=9)).cuda()
    base = ag._eval_draw
    avg = mb.eval_policy_in_model(ag, obs, horizon=40, eval_cnt=3)
    assert "[3] Evaluation in the learned target model over 300 episodes:" in capsys.readouterr().out
    res, _ = ag.evaluate_in_model(obs, 40, step0=base)
    assert avg == float(res["returns"].mean())
