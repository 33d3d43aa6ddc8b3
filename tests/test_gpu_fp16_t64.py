"""The fp16 step mode on 64-row tiles ("fp16_t64": the shapes of the fp32 mode outside fp16's S <= 64, A <= 16,
2S+A <= 112; csrc/step_wide.cu's F16 instantiation), at Ant's S111/A8, Adroit's pen 45/24, door 39/28, relocate 39/30 and
hammer 46/26 and the edges of the range, against the float64 oracle, the numpy Philox oracle, the bf16x2 64-row modes
and the fp32 kernel.

Bound: the fp16 mode's own, rel_err < 5e-3 on next_obs, reward, raw_reward, penalty and the ensemble means.  Termination
masks match exactly except for rows whose oracle next state lies within NEAR of a threshold of the predicate (fp16
rounding moves a next state by up to a few 1e-3 of the tensor's scale); those rows are counted and reported.
Production-mode noise and member picks are held to oracle.philox.rollout_noise under test_gpu_philox_draws.py's "fp16"
bound."""
import numpy as np
import pytest
import torch

from helpers import cuda_agent, cuda_module, healthy, rel_err, rel_err_strict
from model_eval_oracle import model_return
from oracle import mobody_oracle as M
from test_gpu_philox_draws import check_step_noise

pytestmark = pytest.mark.gpu

PREC = "fp16_t64"
TOL = 5e-3
NEAR = 1e-2
# termination kind -> (task the predicate is dispatched from, kind id, module env, healthy x0, transition3 gain)
KINDS = {"ant": ("ant-medium-v2", 4, "ant", 0.95, 2.0), "hopper": ("hopper-medium-v2", 2, "hopper", 0.8, 2.0),
         "walker2d": ("walker2d-medium-v2", 3, "walker2d", 0.95, 4.0),
         "halfcheetah": ("halfcheetah-medium-v2", 1, "halfcheetah", None, 1.0),
         "pen": ("pen-human-v0", 6, "halfcheetah", None, 2.0), "never": ("door-human-v0", 0, "halfcheetah", None, 2.0)}
PEN_X = 0.16    # transition3's bias puts the pen's object height (column 26) here: part of the rows fall below 0.075


def make_dynamics(S, A, seed, kind, coef=2.0, precision=PREC):
    """MOBODYEnsembleDynamics with the oracle's recipe weights; transition3's bias holds the next states around a point
    where ``kind``'s predicate fires on part of the rows."""
    import mobody_b200 as mb
    task, kid, env, h0, t3 = KINDS[kind]
    m, p = cuda_module(S, A, seed, env, h0=h0, t3_gain=t3)
    if kind == "pen":
        with torch.no_grad():
            m.transition3.bias[..., 26] += PEN_X
        p["transition3.bias"] = p["transition3.bias"].clone()
        p["transition3.bias"][..., 26] += PEN_X
    dyn = mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, m, None, None,
                                    mb.get_termination_fn(task), penalty_coef=coef, precision=precision)
    assert dyn.terminal_fn.kind == kid
    return dyn, p


def start_states(kind, S, B, rng, spread=0.2):
    _, _, env, h0, _ = KINDS[kind]
    hs = healthy(env, S, h0)
    if kind == "pen":
        hs[26] = PEN_X
    return (hs[None] + spread * rng.standard_normal((B, S))).astype(np.float32)


def term_distance(kind, x):
    """Distance of each next state to its termination predicate's thresholds (terminal_funs.py)."""
    x = np.asarray(x, np.float64)
    if kind == "ant":
        return np.minimum(np.abs(x[:, 0] - 0.2), np.abs(x[:, 0] - 1.0))
    if kind == "hopper":
        return np.minimum(np.minimum(np.abs(x[:, 0] - 0.7), np.abs(np.abs(x[:, 1]) - 0.2)), np.abs(100.0 - x[:, 1:]).min(1))
    if kind == "walker2d":
        return np.minimum(np.minimum(np.abs(x[:, 0] - 0.8), np.abs(x[:, 0] - 2.0)), np.abs(np.abs(x[:, 1]) - 1.0))
    if kind == "halfcheetah":
        return np.abs(100.0 - np.abs(x)).min(1)
    if kind == "pen":
        return np.abs(x[:, 26] - 0.075)
    return np.full(len(x), np.inf)


def check_outputs(got, ref, kind):
    """got / ref: dicts of numpy arrays.  Returns (worst rel_err / TOL, rows excused from the mask check)."""
    worst = 0.0
    for k in ("next_obs", "reward", "raw_reward", "penalty", "mean"):
        e = rel_err(got[k], ref[k])
        assert e < TOL, (k, e)
        worst = max(worst, e / TOL)
    bad = np.flatnonzero(got["terminal"].reshape(-1) != ref["terminal"].reshape(-1))
    near = term_distance(kind, ref["next_obs"]) < NEAR
    assert near[bad].all(), bad[~near[bad]]
    return worst, len(bad)


WIDE = [(S, A) for S in (65, 80, 111, 128) for A in (1, 8, 32)]
ADROIT = [(45, 24), (39, 28), (39, 30), (46, 26), (45, 17)]
EDGES = [(2, 17), (56, 1), (64, 16), (48, 17)]


@pytest.mark.parametrize("S,A", WIDE + ADROIT + EDGES)
def test_step_matches_float64_oracle(S, A):
    """Batches of 1, 63, 64, 65 and 1 000 rows (ragged 64-row tiles); use_trg, use_penalty and the termination kind vary
    over the batches (pen where S >= 27); injected eps / idx."""
    worst, flips, fired = 0.0, 0, 0
    for bi, B in enumerate((1, 63, 64, 65, 1000)):
        kind = list(KINDS)[(bi + S + A) % len(KINDS)]
        if kind == "pen" and S < 27:
            kind = "ant"
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
        w, f = check_outputs(got, ref, kind)
        worst, flips, fired = max(worst, w), flips + f, fired + int(ref["terminal"].sum())
    assert fired > 0                                   # the mask comparison is not vacuous
    print(f"\n[fp16_t64 step parity] S={S} A={A}: worst rel_err/bound {worst:.3f}, {flips} mask flips within {NEAR} of a threshold")


@pytest.mark.parametrize("S,A", [(65, 1), (111, 8), (128, 32), (45, 24), (2, 17)])
def test_production_draws_match_philox_oracle(S, A):
    """Philox noise and member picks: row ids across 2^32, step words 0 and 2^32 - 1, 1, 5 and 7 elites."""
    from mobody_b200.dynamics import StepWorkspace
    dyn, _ = make_dynamics(S, A, 3, "never", 1.0)
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
        worst = max(worst, check_step_noise("fp16", ws.next_obs.cpu(), ws.mean.cpu(), 1234, step, row0 + np.arange(B), elites))
    print(f"\n[fp16_t64 step Philox] S={S} A={A}: worst err/bound {worst:.3f}")


AGENTS = {"ant": (111, 8), "pen": (45, 24)}


def _agent(kind, prec, seed=5, **overrides):
    S, A = AGENTS[kind]
    dyn, p = make_dynamics(S, A, seed, kind, precision=prec)
    ag, st = cuda_agent(S, A, seed, **dict(dict(env_filter=1e9), **overrides))
    ag.dynamics = dyn
    return ag, p, st


@pytest.mark.parametrize("kind", list(AGENTS))
def test_fused_policy_rollout_matches_oracle(kind):
    """mobody_rollout with the policy fused, T = 3, rows ending at every step.  The first step's B transitions (the start
    states, in order in both) within the bound.  Without an oracle next state within NEAR of a threshold the whole
    result must match: transition count and terminals exactly, every value within the bound.  Otherwise a row may end
    on the other side of a threshold, which changes the rows of later steps: the counts then differ by at most the number
    of such rows."""
    S, A = AGENTS[kind]
    B, T = 300, 3
    ag, p, st = _agent(kind, PREC)
    rng = np.random.default_rng(11)
    obs = start_states(kind, S, B, rng)
    eps_t = rng.standard_normal((T, 7, B, S)).astype(np.float32)
    idx_t = rng.integers(0, 7, (T, B))
    tr, inf = ag.rollout(torch.from_numpy(obs).cuda(), T, True, eps=eps_t, idx=idx_t)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in st.policy.items()}
    want, winf = M.rollout(p64, pol64, 1.0, torch.from_numpy(obs).double(), T,
                           [lambda n, t=t: torch.from_numpy(eps_t[t][:, :n]).double() for t in range(T)],
                           [lambda n, t=t: idx_t[t][:n] for t in range(T)], KINDS[kind][1], 2.0, 1e9, True)
    assert 0 < want["terminals"].sum() < len(want["terminals"]) and winf["num_transitions"] > B
    n_near = int((term_distance(kind, want["next_obss"].numpy()) < NEAR).sum())
    worst = 0.0
    for k in ("obss", "actions", "next_obss", "rewards"):
        e = rel_err(tr[k].numpy()[:B], want[k].numpy()[:B])
        assert e < TOL, (k, e)
        worst = max(worst, e / TOL)
    assert abs(inf["num_transitions"] - winf["num_transitions"]) <= n_near
    if n_near == 0:
        assert np.array_equal(tr["terminals"].numpy().reshape(-1), want["terminals"].numpy().reshape(-1))
        for k in ("obss", "actions", "next_obss", "rewards"):
            assert tuple(tr[k].shape) == tuple(want[k].shape), k
            e = rel_err(tr[k].numpy(), want[k].numpy())
            assert e < TOL, (k, e)
            worst = max(worst, e / TOL)
    print(f"\n[fp16_t64 rollout {kind}] T={T}: {inf['num_transitions']} / {winf['num_transitions']} transitions, "
          f"{int(want['terminals'].sum())} terminal, {n_near} oracle next states within {NEAR} of a threshold, "
          f"worst rel_err/bound {worst:.3f}")


@pytest.mark.parametrize("kind", list(AGENTS))
def test_evaluate_in_model_matches_float64_oracle(kind):
    """Per-start returns over H = 8 steps with Philox draws; rows whose oracle trajectory passes within NEAR of a
    threshold are excluded (counted), the others must end at the same step with returns within the bound."""
    S, A = AGENTS[kind]
    B, H, gamma, row0, step0 = 300, 8, 0.99, (1 << 32) - 10, 7
    ag, p, st = _agent(kind, PREC)
    obs = start_states(kind, S, B, np.random.default_rng(1), spread=0.1)
    res, info = ag.evaluate_in_model(torch.from_numpy(obs).cuda(), H, gamma=gamma, penalized=True, row0=row0, step0=step0)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in st.policy.items()}
    ref = model_return(p64, pol64, 1.0, obs.astype(np.float64), H, gamma, ag.eval_seed, step0, row0, KINDS[kind][1], 2.0,
                       use_penalty=True, record=True)
    dist = np.full(B, np.inf)
    for ids, x in ref["trace"]:
        dist[ids - row0] = np.minimum(dist[ids - row0], term_distance(kind, x))
    near = dist < NEAR
    assert (~near).sum() >= B // 2, near.sum()
    got = {k: v.cpu().numpy() for k, v in res.items()}
    assert np.array_equal(got["lengths"][~near], ref["lengths"][~near])
    assert info["live_per_step"] == ref["counts"].tolist() or near.any()
    assert 0 < ref["counts"][H] < B and len(set(ref["lengths"].tolist())) > 3
    worst = 0.0
    for k in ("returns", "discounted_returns"):
        e = rel_err(got[k][~near], ref[k][~near])
        assert e < TOL, (k, e)
        worst = max(worst, e / TOL)
    print(f"\n[fp16_t64 model eval {kind}] worst rel_err/bound {worst:.3f}, {int(near.sum())}/{B} rows within {NEAR} of a "
          f"threshold excluded, lengths {ref['lengths'].min()}..{ref['lengths'].max()}")


@pytest.mark.parametrize("kind,other", [("ant", "bf16x2_wide"), ("pen", "bf16x2_t64")])
def test_matches_the_bf16x2_64_row_mode_on_100k_rows(kind, other):
    """Production mode, the same seeded start states, seed, step and row ids: both kernels' member picks and noise held
    to the Philox oracle, next_obs, rewards, penalty and means within the bound of the fp32-parity mode's, mask
    differences counted (each one within NEAR of a threshold)."""
    from mobody_b200.dynamics import StepWorkspace
    S, A = AGENTS[kind]
    B = 100_000
    out = {}
    rng = np.random.default_rng(2)
    obs = torch.from_numpy(start_states(kind, S, B, rng)).cuda()
    act = torch.from_numpy(rng.uniform(-1, 1, (B, A)).astype(np.float32)).cuda()
    elites = [6, 0, 3, 5, 1]
    for prec in (other, PREC):
        dyn, _ = make_dynamics(S, A, 9, kind, precision=prec)
        dyn.seed = 77
        dyn.model.set_elites(elites)
        ws = StepWorkspace(B, S, A, obs.device)
        dyn.launch_step(obs, act, ws, step=3, row0=(1 << 32) - 50_000)
        torch.cuda.synchronize()
        out[prec] = {k: getattr(ws, k).cpu().numpy() for k in ("next_obs", "reward", "raw_reward", "penalty", "terminal", "mean")}
        sub = np.arange(0, B, 97)            # the Philox oracle on a sample of the rows (both kernels, same rows)
        check_step_noise("fp16" if prec == PREC else "bf16x2", out[prec]["next_obs"][sub], out[prec]["mean"][:, sub], 77, 3,
                         (1 << 32) - 50_000 + sub, elites)
    a, b = out[PREC], out[other]
    worst = 0.0
    for k in ("next_obs", "reward", "raw_reward", "penalty", "mean"):
        e = rel_err(a[k], b[k])
        assert e < TOL, (k, e)
        worst = max(worst, e / TOL)
    assert 0 < b["terminal"].sum() < B
    flips = np.flatnonzero(a["terminal"] != b["terminal"])
    assert (term_distance(kind, b["next_obs"][flips]) < NEAR).all()
    print(f"\n[fp16_t64 vs {other}, 100k rows] worst rel_err/bound {worst:.3f} (rel_err_strict of next_obs "
          f"{rel_err_strict(a['next_obs'], b['next_obs']):.2e}), {len(flips)} mask differences near a threshold")


def _d4rl(rng, n, S, A):
    hs = np.zeros(S, np.float32)
    hs[26] = PEN_X
    return dict(observations=(hs + 0.2 * rng.standard_normal((n, S))).astype(np.float32),
                actions=rng.uniform(-1, 1, (n, A)).astype(np.float32),
                next_observations=(hs + 0.2 * rng.standard_normal((n, S))).astype(np.float32),
                rewards=rng.standard_normal(n).astype(np.float32), terminals=np.zeros(n, bool))


def test_par_penalty_and_train_steps_at_pen():
    """penalty_type='par': the dynamics step inside every MOBODY.train update runs in this mode.  With injected
    par_eps / par_idx the penalised rewards agree with the fp32 kernel's within the bound; then whole train() calls
    (the first one refreshes the synthetic buffer through rollouts and the dataset step) finish with finite losses and
    the synthetic buffer's size accounting intact."""
    import mobody_b200 as mb
    S, A = AGENTS["pen"]
    B = 128
    rng = np.random.default_rng(4)
    src, tar = mb.ReplayBuffer(S, A, "cuda"), mb.ReplayBuffer(S, A, "cuda")
    src.convert_D4RL(_d4rl(rng, 60000, S, A)); tar.convert_D4RL(_d4rl(rng, 5000, S, A))
    sel = rng.integers(0, src.size, B)
    eps, idx = rng.standard_normal((7, B, S)).astype(np.float32), rng.integers(0, 7, B)
    shift = {}
    for prec in ("fp32", PREC):
        ag, _, _ = _agent("pen", prec, penalty_type="par", penalty_coef=0.1)
        rows = src.sample_rows(B, sel)
        before = rows[:, 2 * S + A].clone()
        ag.total_it = 1
        ag._par_penalty(rows, B, None, eps, idx)
        torch.cuda.synchronize()
        shift[prec] = (before - rows[:, 2 * S + A]).cpu().numpy()
    assert (shift["fp32"] > 0).all()
    e = rel_err(shift[PREC], shift["fp32"])
    assert e < TOL, e
    ag, _, _ = _agent("pen", PREC, penalty_type="par", penalty_coef=0.1, env_filter=10.0)
    before = ag.policy.network.network[0].weight.detach().clone()
    sizes = []
    for _ in range(4):
        ag.train(src, tar, B, None, None)
        sizes.append(ag.fake_replay_buffer.size)
    torch.cuda.synchronize()
    assert ag.dynamics.precision == PREC and 0 < sizes[0] <= ag.fake_replay_buffer.max_size
    assert sizes == sorted(sizes) and sizes[-1] <= ag.fake_replay_buffer.max_size
    v = ag.loss_scalars()
    assert np.isfinite(list(v.values())).all() and not torch.equal(before, ag.policy.network.network[0].weight.detach())
    print(f"\n[fp16_t64 par] penalised rewards vs fp32: rel_err/bound {e / TOL:.3f}; fake buffer {sizes} rows")


@pytest.mark.parametrize("S,A", [(17, 6), (55, 2), (27, 8), (40, 16), (129, 8), (111, 33)])
def test_rejects_shapes_outside_its_range(S, A):
    """fp16's shapes (2S+A = 112 at S55/A2 included), S > 128 and A > 32."""
    dyn, _ = make_dynamics(S, A, 3, "never", 1.0)
    rng = np.random.default_rng(0)
    obs, act = rng.standard_normal((4, S)).astype(np.float32), rng.uniform(-1, 1, (4, A)).astype(np.float32)
    with pytest.raises(RuntimeError, match=r"mobody_b200 \[-1\].*fp16_t64 takes S <= 128, A <= 32 outside fp16's "
                                           r"S <= 64, A <= 16, 2S\+A <= 112"):
        dyn.step(torch.from_numpy(obs).cuda(), torch.from_numpy(act).cuda())
