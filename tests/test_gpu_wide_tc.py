"""The wide tensor-core step mode ("bf16x2_wide": 64-row tiles, 65 <= S <= 128, A <= 32; csrc/step_wide.cu) against the
float64 oracle, the numpy Philox oracle and the fp32 CUDA-core kernel.

Bounds: next_obs, reward, raw_reward, penalty and the ensemble means within 1e-4 under both rel_err and rel_err_strict.
Termination masks match exactly except for rows whose oracle next state lies within NEAR of a threshold of the
predicate; those rows are counted and reported.  Production-mode noise and member picks are held to
oracle.philox.rollout_noise under test_gpu_philox_draws.py's bound for the SFU sine / cosine (the kernel draws with the
same philox_normal1 as the bf16x2 kernel)."""
import numpy as np
import pytest
import torch

from helpers import cuda_agent, cuda_dynamics, healthy, rel_err, rel_err_strict
from model_eval_oracle import model_return
from oracle import mobody_oracle as M
from test_gpu_philox_draws import check_step_noise

pytestmark = pytest.mark.gpu

PREC = "bf16x2_wide"
NEAR = 1e-4
# env -> (termination kind, healthy x0, transition3 gain): each termination predicate fires on a part of the rows
ENVS = {"ant": (4, 0.95, 2.0), "hopper": (2, 0.8, 2.0), "walker2d": (3, 0.95, 4.0), "halfcheetah": (1, None, 1.0)}


def _term_distance(env, x):
    """Distance of each next state to its termination predicate's thresholds (terminal_funs.py)."""
    x = np.asarray(x, np.float64)
    if env == "ant":
        return np.minimum(np.abs(x[:, 0] - 0.2), np.abs(x[:, 0] - 1.0))
    if env == "hopper":
        return np.minimum(np.minimum(np.abs(x[:, 0] - 0.7), np.abs(np.abs(x[:, 1]) - 0.2)), np.abs(100.0 - x[:, 1:]).min(1))
    if env == "walker2d":
        return np.minimum(np.minimum(np.abs(x[:, 0] - 0.8), np.abs(x[:, 0] - 2.0)), np.abs(np.abs(x[:, 1]) - 1.0))
    return np.abs(100.0 - np.abs(x)).min(1)


def _check_outputs(got, ref, env):
    """got / ref: dicts of numpy arrays.  Returns (worst err / 1e-4, rows excused from the mask check)."""
    worst = 0.0
    for k in ("next_obs", "reward", "raw_reward", "penalty", "mean"):
        e = max(rel_err(got[k], ref[k]), rel_err_strict(got[k], ref[k]))
        assert e < 1e-4, (k, e)
        worst = max(worst, e / 1e-4)
    bad = np.flatnonzero(got["terminal"].reshape(-1) != ref["terminal"].reshape(-1))
    near = _term_distance(env, ref["next_obs"]) < NEAR
    assert near[bad].all(), bad[~near[bad]]
    return worst, len(bad)


CASES = [(S, A) for S in (65, 80, 111, 128) for A in (1, 8, 32)]


@pytest.mark.parametrize("S,A", CASES)
def test_step_matches_float64_oracle(S, A):
    """Batches of 1, 63, 64, 65 and 1 000 rows (ragged 64-row tiles); use_trg, use_penalty and the termination kind vary
    over the batches; injected eps / idx."""
    worst, flips, fired = 0.0, 0, 0
    for bi, B in enumerate((1, 63, 64, 65, 1000)):
        env = list(ENVS)[(bi + S + A) % 4]
        kind, h0, t3 = ENVS[env]
        use_trg, use_pen = bool((bi + A) & 1), bool(((bi + S) >> 1) & 1)
        dyn, p = cuda_dynamics(S, A, S + A + bi, env, 2.0, precision=PREC, h0=h0, t3_gain=t3)
        assert dyn.precision == PREC
        p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
        rng = np.random.default_rng(1000 * S + 10 * A + bi)
        obs = (healthy(env, S, h0)[None] + 0.2 * rng.standard_normal((B, S))).astype(np.float32)
        act = rng.uniform(-1, 1, (B, A)).astype(np.float32)
        eps = rng.standard_normal((7, B, S)).astype(np.float32)
        idx = rng.integers(0, 7, B)
        r = M.step(p64, torch.from_numpy(obs).double(), torch.from_numpy(act).double(), torch.from_numpy(eps).double(), idx,
                   kind, 2.0, use_penalty=use_pen, use_trg=use_trg)
        nobs, rew, term, info = dyn.step(torch.from_numpy(obs).cuda(), torch.from_numpy(act).cuda(), use_pen, use_trg, eps=eps, idx=idx)
        got = dict(next_obs=nobs.cpu().numpy(), reward=rew.cpu().numpy(), raw_reward=info["raw_reward"].cpu().numpy(),
                   penalty=info["penalty"].cpu().numpy(), mean=info["samples"].cpu().numpy(), terminal=term)
        ref = {k: (v.numpy() if torch.is_tensor(v) else v) for k, v in r.items()}
        w, f = _check_outputs(got, ref, env)
        worst, flips, fired = max(worst, w), flips + f, fired + int(ref["terminal"].sum())
    assert fired > 0                                   # the mask comparison is not vacuous
    print(f"\n[wide step parity] S={S} A={A}: worst err/bound {worst:.3f}, {flips} mask flips within {NEAR} of a threshold")


@pytest.mark.parametrize("S,A", [(65, 1), (111, 8), (128, 32)])
def test_production_draws_match_philox_oracle(S, A):
    """Philox noise and member picks: row ids across 2^32, step words 0 and 2^32 - 1, 1, 5 and 7 elites."""
    from mobody_b200.dynamics import StepWorkspace
    dyn, _ = cuda_dynamics(S, A, 3, "halfcheetah", 1.0, precision=PREC)
    dyn.seed = 1234
    rng = np.random.default_rng(S + A)
    worst = 0.0
    for B, row0, step, elites in ((1000, 0, 0, [6, 0, 3, 5, 1]), (129, (1 << 32) - 64, (1 << 32) - 1, [3, 6, 0, 2, 5, 1, 4]),
                                  (65, (1 << 40) + 3, 7, [4])):
        dyn.model.set_elites(elites)
        obs = torch.from_numpy((0.5 * rng.standard_normal((B, S))).astype(np.float32)).cuda()
        act = torch.from_numpy(rng.uniform(-1, 1, (B, A)).astype(np.float32)).cuda()
        ws = StepWorkspace(B, S, A, obs.device)
        dyn.launch_step(obs, act, ws, step=step, row0=row0)
        torch.cuda.synchronize()
        # "bf16x2": the bound of the SFU sine / cosine, which this kernel's draws share
        worst = max(worst, check_step_noise("bf16x2", ws.next_obs.cpu(), ws.mean.cpu(), 1234, step, row0 + np.arange(B), elites))
    print(f"\n[wide step Philox] S={S} A={A}: worst err/bound {worst:.3f}")


def _ant_agent(prec, seed=5):
    S, A = 111, 8
    kind, h0, t3 = ENVS["ant"]
    dyn, p = cuda_dynamics(S, A, seed, "ant", 2.0, precision=prec, h0=h0, t3_gain=t3)
    ag, st = cuda_agent(S, A, seed, env_filter=1e9)
    ag.dynamics = dyn
    return ag, p, st


def test_fused_policy_rollout_matches_oracle():
    """mobody_rollout with the policy fused, T = 3, ant termination (rows end at every step): transition counts and the
    compaction order bit-exact, values within the bound."""
    S, A, B, T = 111, 8, 300, 3
    kind, h0, _ = ENVS["ant"]
    ag, p, st = _ant_agent(PREC)
    rng = np.random.default_rng(11)
    obs = (healthy("ant", S, h0)[None] + 0.2 * rng.standard_normal((B, S))).astype(np.float32)
    eps_t = rng.standard_normal((T, 7, B, S)).astype(np.float32)
    idx_t = rng.integers(0, 7, (T, B))
    tr, inf = ag.rollout(torch.from_numpy(obs).cuda(), T, True, eps=eps_t, idx=idx_t)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in st.policy.items()}
    want, winf = M.rollout(p64, pol64, 1.0, torch.from_numpy(obs).double(), T,
                           [lambda n, t=t: torch.from_numpy(eps_t[t][:, :n]).double() for t in range(T)],
                           [lambda n, t=t: idx_t[t][:n] for t in range(T)], kind, 2.0, 1e9, True)
    assert inf["num_transitions"] == winf["num_transitions"]
    assert 0 < want["terminals"].sum() < len(want["terminals"]) and winf["num_transitions"] > B
    assert np.array_equal(tr["terminals"].numpy().reshape(-1), want["terminals"].numpy().reshape(-1))
    assert _term_distance("ant", want["next_obss"].numpy()).min() > NEAR
    for k in ("obss", "actions", "next_obss", "rewards"):
        assert tuple(tr[k].shape) == tuple(want[k].shape), k
        e = max(rel_err(tr[k].numpy(), want[k].numpy()), rel_err_strict(tr[k].numpy(), want[k].numpy()))
        assert e < 1e-4, (k, e)
    print(f"\n[wide rollout] T={T}: {winf['num_transitions']} transitions, {int(want['terminals'].sum())} terminal")


def test_evaluate_in_model_matches_float64_oracle():
    S, A, B, H, gamma, row0, step0 = 111, 8, 300, 8, 0.99, (1 << 32) - 10, 7
    kind, h0, _ = ENVS["ant"]
    ag, p, st = _ant_agent(PREC)
    obs = (healthy("ant", S, h0)[None] + 0.1 * np.random.default_rng(1).standard_normal((B, S))).astype(np.float32)
    res, info = ag.evaluate_in_model(torch.from_numpy(obs).cuda(), H, gamma=gamma, penalized=True, row0=row0, step0=step0)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in st.policy.items()}
    ref = model_return(p64, pol64, 1.0, obs.astype(np.float64), H, gamma, ag.eval_seed, step0, row0, kind, 2.0,
                       use_penalty=True, record=True)
    dist = np.full(B, np.inf)
    for ids, x in ref["trace"]:
        dist[ids - row0] = np.minimum(dist[ids - row0], _term_distance("ant", x))
    near = dist < NEAR
    assert near.mean() < 0.05, near.mean()
    got = {k: v.cpu().numpy() for k, v in res.items()}
    assert np.array_equal(got["lengths"][~near], ref["lengths"][~near])
    assert info["live_per_step"] == ref["counts"].tolist() or near.any()
    assert 0 < ref["counts"][H] < B and len(set(ref["lengths"].tolist())) > 3
    worst = 0.0
    for k in ("returns", "discounted_returns"):
        e = rel_err_strict(got[k][~near], ref[k][~near])
        assert e < 1e-4, (k, e)
        worst = max(worst, e / 1e-4)
    print(f"\n[wide model eval] worst err/bound {worst:.3f}, {int(near.sum())}/{B} rows within {NEAR} of a threshold excluded, "
          f"lengths {ref['lengths'].min()}..{ref['lengths'].max()}")


def test_matches_the_fp32_kernel_on_100k_rows():
    """Production mode, same seed / step / row ids: identical member picks and noise (both held to the Philox oracle),
    next_obs and reward within the bound of each other."""
    from mobody_b200.dynamics import StepWorkspace
    S, A, B = 111, 8, 100_000
    out = {}
    rng = np.random.default_rng(2)
    obs = torch.from_numpy((healthy("ant", S, 0.6)[None] + 0.2 * rng.standard_normal((B, S))).astype(np.float32)).cuda()
    act = torch.from_numpy(rng.uniform(-1, 1, (B, A)).astype(np.float32)).cuda()
    elites = [6, 0, 3, 5, 1]
    for prec in ("fp32", PREC):
        dyn, _ = cuda_dynamics(S, A, 9, "ant", 2.0, precision=prec, h0=0.6)
        dyn.seed = 77
        dyn.model.set_elites(elites)
        ws = StepWorkspace(B, S, A, obs.device)
        dyn.launch_step(obs, act, ws, step=3, row0=(1 << 32) - 50_000)
        torch.cuda.synchronize()
        out[prec] = {k: getattr(ws, k).cpu().numpy() for k in ("next_obs", "reward", "raw_reward", "penalty", "terminal", "mean")}
        sub = np.arange(0, B, 97)            # the Philox oracle on a sample of the rows (both kernels, same rows)
        check_step_noise("bf16x2" if prec == PREC else "fp32", out[prec]["next_obs"][sub], out[prec]["mean"][:, sub], 77, 3,
                         (1 << 32) - 50_000 + sub, elites)
    a, b = out[PREC], out["fp32"]
    worst = 0.0
    for k in ("next_obs", "reward", "raw_reward", "penalty", "mean"):
        e = rel_err(a[k], b[k])
        assert e < 1e-4, (k, e)
        worst = max(worst, e / 1e-4)
    flips = np.flatnonzero(a["terminal"] != b["terminal"])
    assert (_term_distance("ant", b["next_obs"][flips]) < NEAR).all()
    print(f"\n[wide vs fp32, 100k rows] worst err/bound {worst:.3f}, {len(flips)} mask flips near a threshold")


@pytest.mark.parametrize("S,A", [(64, 8), (129, 8), (111, 33)])
def test_rejects_shapes_outside_its_range(S, A):
    dyn, _ = cuda_dynamics(S, A, 3, "halfcheetah", 1.0, precision=PREC)
    rng = np.random.default_rng(0)
    obs, act = rng.standard_normal((4, S)).astype(np.float32), rng.uniform(-1, 1, (4, A)).astype(np.float32)
    with pytest.raises(RuntimeError, match=r"mobody_b200 \[-1\].*bf16x2_wide takes 65 <= S <= 128"):
        dyn.step(torch.from_numpy(obs).cuda(), torch.from_numpy(act).cuda())
