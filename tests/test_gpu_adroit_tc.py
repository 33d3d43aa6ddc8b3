"""The 64-row tensor-core step mode for the S <= 64 shapes bf16x2 refuses ("bf16x2_t64": A > 16 or 2S+A > 96, A <= 32;
csrc/step_wide.cu), at Adroit's shapes (pen 45/24, door 39/28, relocate 39/30, hammer 46/26), the truncated Humanoid
observation (45/17) and the edges of the range, against the float64 oracle, the numpy Philox oracle and the fp32 CUDA-core
kernel.

Bounds: next_obs, reward, raw_reward, penalty and the ensemble means within 1e-4 under both rel_err and rel_err_strict.
Termination masks match exactly except for rows whose oracle next state lies within NEAR of a threshold of the
predicate; those rows are counted and reported.  Production-mode noise and member picks are held to
oracle.philox.rollout_noise under test_gpu_philox_draws.py's bound for the SFU sine / cosine (the kernel draws with the
same philox_normal1 as the bf16x2 kernel)."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import cuda_agent, cuda_module, healthy, rel_err, rel_err_strict
from model_eval_oracle import model_return
from oracle import mobody_oracle as M
from test_gpu_philox_draws import check_step_noise

pytestmark = pytest.mark.gpu

PREC = "bf16x2_t64"
NEAR = 1e-4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# termination kind -> (task name the predicate is dispatched from, kind id, healthy x0)
KINDS = {"pen": ("pen-human-v0", 6, None), "humanoid": ("humanoid-v2", 5, 1.05), "never": ("door-human-v0", 0, None),
         "halfcheetah": ("halfcheetah-medium-v2", 1, None)}
PEN_X = 0.16    # transition3's bias puts the pen's object height (column 26) here: part of the rows fall below 0.075


def make_dynamics(S, A, seed, kind, coef=2.0, precision=PREC, t3_gain=2.0):
    """MOBODYEnsembleDynamics with the oracle's recipe weights; transition3's bias holds the next states around a point
    where ``kind``'s predicate fires on part of the rows."""
    import mobody_b200 as mb
    task, _, h0 = KINDS[kind]
    m, p = cuda_module(S, A, seed, "halfcheetah", h0=h0, t3_gain=t3_gain)
    if kind == "pen":
        with torch.no_grad():
            m.transition3.bias[..., 26] += PEN_X
        p["transition3.bias"] = p["transition3.bias"].clone()
        p["transition3.bias"][..., 26] += PEN_X
    dyn = mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, m, None, None,
                                    mb.get_termination_fn(task), penalty_coef=coef, precision=precision)
    assert dyn.terminal_fn.kind == KINDS[kind][1]
    return dyn, p


def start_states(kind, S, B, rng, spread=0.2):
    hs = healthy("halfcheetah", S, KINDS[kind][2])
    if kind == "pen":
        hs[26] = PEN_X
    return (hs[None] + spread * rng.standard_normal((B, S))).astype(np.float32)


def _term_distance(kind, x):
    """Distance of each next state to its termination predicate's thresholds (terminal_funs.py)."""
    x = np.asarray(x, np.float64)
    if kind == "pen":
        return np.abs(x[:, 26] - 0.075)
    if kind == "humanoid":
        return np.minimum(np.abs(x[:, 0] - 1.0), np.abs(x[:, 0] - 2.0))
    if kind == "halfcheetah":
        return np.abs(100.0 - np.abs(x)).min(1)
    return np.full(len(x), np.inf)


def _check_outputs(got, ref, kind):
    """got / ref: dicts of numpy arrays.  Returns (worst err / 1e-4, rows excused from the mask check)."""
    worst = 0.0
    for k in ("next_obs", "reward", "raw_reward", "penalty", "mean"):
        e = max(rel_err(got[k], ref[k]), rel_err_strict(got[k], ref[k]))
        assert e < 1e-4, (k, e)
        worst = max(worst, e / 1e-4)
    bad = np.flatnonzero(got["terminal"].reshape(-1) != ref["terminal"].reshape(-1))
    near = _term_distance(kind, ref["next_obs"]) < NEAR
    assert near[bad].all(), bad[~near[bad]]
    return worst, len(bad)


ADROIT = [(45, 24), (39, 28), (39, 30), (46, 26)]
EDGES = [(45, 17), (2, 17), (48, 1), (64, 16), (64, 32), (40, 17)]


@pytest.mark.parametrize("S,A", ADROIT + EDGES)
def test_step_matches_float64_oracle(S, A):
    """Batches of 1, 63, 64, 65 and 1 000 rows (ragged 64-row tiles); use_trg, use_penalty and the termination kind vary
    over the batches (pen where S >= 27); injected eps / idx."""
    worst, flips, fired = 0.0, 0, 0
    for bi, B in enumerate((1, 63, 64, 65, 1000)):
        kind = list(KINDS)[(bi + S + A) % 4]
        if kind == "pen" and S < 27:
            kind = "humanoid"
        use_trg, use_pen = bool((bi + A) & 1), bool(((bi + S) >> 1) & 1)
        dyn, p = make_dynamics(S, A, S + A + bi, kind)
        assert dyn.precision == PREC
        p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
        rng = np.random.default_rng(1000 * S + 10 * A + bi)
        obs = start_states(kind, S, B, rng)
        act = rng.uniform(-1, 1, (B, A)).astype(np.float32)
        eps = rng.standard_normal((7, B, S)).astype(np.float32)
        idx = rng.integers(0, 7, B)
        r = M.step(p64, torch.from_numpy(obs).double(), torch.from_numpy(act).double(), torch.from_numpy(eps).double(), idx,
                   KINDS[kind][1], 2.0, use_penalty=use_pen, use_trg=use_trg)
        nobs, rew, term, info = dyn.step(torch.from_numpy(obs).cuda(), torch.from_numpy(act).cuda(), use_pen, use_trg, eps=eps, idx=idx)
        got = dict(next_obs=nobs.cpu().numpy(), reward=rew.cpu().numpy(), raw_reward=info["raw_reward"].cpu().numpy(),
                   penalty=info["penalty"].cpu().numpy(), mean=info["samples"].cpu().numpy(), terminal=term)
        ref = {k: (v.numpy() if torch.is_tensor(v) else v) for k, v in r.items()}
        w, f = _check_outputs(got, ref, kind)
        worst, flips, fired = max(worst, w), flips + f, fired + int(ref["terminal"].sum())
    assert fired > 0                                   # the mask comparison is not vacuous
    print(f"\n[t64 step parity] S={S} A={A}: worst err/bound {worst:.3f}, {flips} mask flips within {NEAR} of a threshold")


@pytest.mark.parametrize("S,A", [(45, 24), (64, 32), (2, 17)])
def test_production_draws_match_philox_oracle(S, A):
    """Philox noise and member picks: row ids across 2^32, step words 0 and 2^32 - 1, 1, 5 and 7 elites."""
    from mobody_b200.dynamics import StepWorkspace
    dyn, _ = make_dynamics(S, A, 3, "never", 1.0, t3_gain=1.0)
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
    print(f"\n[t64 step Philox] S={S} A={A}: worst err/bound {worst:.3f}")


def _pen_agent(prec, seed=5, **overrides):
    S, A = 45, 24
    dyn, p = make_dynamics(S, A, seed, "pen", precision=prec)
    ag, st = cuda_agent(S, A, seed, **dict(dict(env_filter=1e9), **overrides))
    ag.dynamics = dyn
    return ag, p, st


def test_fused_policy_rollout_matches_oracle():
    """mobody_rollout with the policy fused, T = 3, pen termination (rows end at every step): transition counts and the
    compaction order bit-exact, values within the bound."""
    S, A, B, T = 45, 24, 300, 3
    ag, p, st = _pen_agent(PREC)
    rng = np.random.default_rng(11)
    obs = start_states("pen", S, B, rng)
    eps_t = rng.standard_normal((T, 7, B, S)).astype(np.float32)
    idx_t = rng.integers(0, 7, (T, B))
    tr, inf = ag.rollout(torch.from_numpy(obs).cuda(), T, True, eps=eps_t, idx=idx_t)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in st.policy.items()}
    want, winf = M.rollout(p64, pol64, 1.0, torch.from_numpy(obs).double(), T,
                           [lambda n, t=t: torch.from_numpy(eps_t[t][:, :n]).double() for t in range(T)],
                           [lambda n, t=t: idx_t[t][:n] for t in range(T)], 6, 2.0, 1e9, True)
    assert inf["num_transitions"] == winf["num_transitions"]
    assert 0 < want["terminals"].sum() < len(want["terminals"]) and winf["num_transitions"] > B
    assert np.array_equal(tr["terminals"].numpy().reshape(-1), want["terminals"].numpy().reshape(-1))
    assert _term_distance("pen", want["next_obss"].numpy()).min() > NEAR
    for k in ("obss", "actions", "next_obss", "rewards"):
        assert tuple(tr[k].shape) == tuple(want[k].shape), k
        e = max(rel_err(tr[k].numpy(), want[k].numpy()), rel_err_strict(tr[k].numpy(), want[k].numpy()))
        assert e < 1e-4, (k, e)
    print(f"\n[t64 rollout] T={T}: {winf['num_transitions']} transitions, {int(want['terminals'].sum())} terminal")


def test_evaluate_in_model_matches_float64_oracle():
    S, A, B, H, gamma, row0, step0 = 45, 24, 300, 8, 0.99, (1 << 32) - 10, 7
    ag, p, st = _pen_agent(PREC)
    obs = start_states("pen", S, B, np.random.default_rng(1), spread=0.1)
    res, info = ag.evaluate_in_model(torch.from_numpy(obs).cuda(), H, gamma=gamma, penalized=True, row0=row0, step0=step0)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in st.policy.items()}
    ref = model_return(p64, pol64, 1.0, obs.astype(np.float64), H, gamma, ag.eval_seed, step0, row0, 6, 2.0,
                       use_penalty=True, record=True)
    dist = np.full(B, np.inf)
    for ids, x in ref["trace"]:
        dist[ids - row0] = np.minimum(dist[ids - row0], _term_distance("pen", x))
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
    print(f"\n[t64 model eval] worst err/bound {worst:.3f}, {int(near.sum())}/{B} rows within {NEAR} of a threshold excluded, "
          f"lengths {ref['lengths'].min()}..{ref['lengths'].max()}")


def test_matches_the_fp32_kernel_on_100k_rows():
    """Production mode, same seed / step / row ids: identical member picks and noise (both held to the Philox oracle),
    next_obs and reward within the bound of each other."""
    from mobody_b200.dynamics import StepWorkspace
    S, A, B = 45, 24, 100_000
    out = {}
    rng = np.random.default_rng(2)
    obs = torch.from_numpy(start_states("pen", S, B, rng)).cuda()
    act = torch.from_numpy(rng.uniform(-1, 1, (B, A)).astype(np.float32)).cuda()
    elites = [6, 0, 3, 5, 1]
    for prec in ("fp32", PREC):
        dyn, _ = make_dynamics(S, A, 9, "pen", precision=prec)
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
    assert 0 < b["terminal"].sum() < B
    flips = np.flatnonzero(a["terminal"] != b["terminal"])
    assert (_term_distance("pen", b["next_obs"][flips]) < NEAR).all()
    print(f"\n[t64 vs fp32, 100k rows] worst err/bound {worst:.3f}, {len(flips)} mask flips near a threshold")


def _d4rl(rng, n, S, A):
    hs = np.zeros(S, np.float32)
    hs[26] = PEN_X
    return dict(observations=(hs + 0.2 * rng.standard_normal((n, S))).astype(np.float32),
                actions=rng.uniform(-1, 1, (n, A)).astype(np.float32),
                next_observations=(hs + 0.2 * rng.standard_normal((n, S))).astype(np.float32),
                rewards=rng.standard_normal(n).astype(np.float32), terminals=np.zeros(n, bool))


def test_par_penalty_and_train_steps_at_pen():
    """penalty_type='par': the dynamics step inside every MOBODY.train update runs in this mode.  With injected
    par_eps / par_idx the penalised rewards of the two precisions agree within the bound; then whole train() calls
    (the first one refreshes the synthetic buffer through rollouts and the dataset step) finish with finite losses."""
    import mobody_b200 as mb
    S, A, B = 45, 24, 128
    rng = np.random.default_rng(4)
    src, tar = mb.ReplayBuffer(S, A, "cuda"), mb.ReplayBuffer(S, A, "cuda")
    src.convert_D4RL(_d4rl(rng, 60000, S, A)); tar.convert_D4RL(_d4rl(rng, 5000, S, A))
    sel = rng.integers(0, src.size, B)
    eps, idx = rng.standard_normal((7, B, S)).astype(np.float32), rng.integers(0, 7, B)
    shift = {}
    for prec in ("fp32", PREC):
        ag, _, _ = _pen_agent(prec, penalty_type="par", penalty_coef=0.1)
        rows = src.sample_rows(B, sel)
        before = rows[:, 2 * S + A].clone()
        ag.total_it = 1
        ag._par_penalty(rows, B, None, eps, idx)
        torch.cuda.synchronize()
        shift[prec] = (before - rows[:, 2 * S + A]).cpu().numpy()
    assert (shift["fp32"] > 0).all()
    e = max(rel_err(shift[PREC], shift["fp32"]), rel_err_strict(shift[PREC], shift["fp32"]))
    assert e < 1e-4, e
    ag, _, _ = _pen_agent(PREC, penalty_type="par", penalty_coef=0.1, env_filter=10.0)
    before = ag.policy.network.network[0].weight.detach().clone()
    for _ in range(4):
        ag.train(src, tar, B, None, None)
    torch.cuda.synchronize()
    assert ag.dynamics.precision == PREC and ag.fake_replay_buffer.size > 0
    v = ag.loss_scalars()
    assert np.isfinite(list(v.values())).all() and not torch.equal(before, ag.policy.network.network[0].weight.detach())
    print(f"\n[t64 par] penalised rewards vs fp32: err/bound {e / 1e-4:.3f}; fake buffer {ag.fake_replay_buffer.size} rows")


@pytest.mark.parametrize("S,A", [(17, 6), (40, 16), (2, 16), (65, 8), (64, 33)])
def test_rejects_shapes_outside_its_range(S, A):
    """Shapes bf16x2 takes, one of bf16x2_wide's, and A > 32."""
    dyn, _ = make_dynamics(S, A, 3, "never", 1.0)
    rng = np.random.default_rng(0)
    obs, act = rng.standard_normal((4, S)).astype(np.float32), rng.uniform(-1, 1, (4, A)).astype(np.float32)
    with pytest.raises(RuntimeError, match=r"mobody_b200 \[-1\].*bf16x2_t64 takes S <= 64, A <= 32 with A > 16 or 2S\+A > 96"):
        dyn.step(torch.from_numpy(obs).cuda(), torch.from_numpy(act).cuda())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_sharded_pen_rollout_over_two_gpus_equals_single_gpu():
    """parallel.p2p_rollout at pen in this mode: the transitions gathered from two GPUs equal one GPU's, bit for bit."""
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29535", os.path.join(ROOT, "scripts", "nccl_check.py"), "pen"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0 and "NCCL_CHECK OK" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
