"""GPU parity of the fused train step (critic TD update + Polyak + Q-weighted BC actor update + Adam).

(a) against post-step parameters produced by the reference's MOBODY.train (golden, indices injected);
(b) against the CPU oracle on larger / ragged batches.  Tolerance: 1e-4 relative (helpers.rel_err)
on every parameter tensor after several steps, losses within 1e-4.
"""
import os

import numpy as np
import pytest
import torch

from helpers import cuda_agent, rel_err
from oracle import mobody_oracle as M

pytestmark = pytest.mark.gpu
CFG = dict(gamma=0.99, tau=0.005, actor_lr=3e-4, critic_lr=3e-4, weight=2.5, bc_coef=1.0, max_action=1.0)


def adam_close(got, want, lr, steps, tag):
    """Post-Adam parameters: 1e-4 relative (helpers.rel_err metric) for all but <= 0.5% of the elements.
    Two discrete effects make a handful of elements ill-conditioned: (i) a hidden unit whose pre-activation is within
    rounding of 0 for some row takes the other ReLU branch, which changes that unit's whole weight row of the
    gradient; (ii) Adam's normalised update m/sqrt(v) ~ sign(g) amplifies 1e-7 differences where |g| ~ 0.  Those rare
    outliers are bounded by the largest possible Adam displacement, 2 * lr * steps, instead."""
    got, want = np.asarray(got, np.float64).reshape(-1), np.asarray(want, np.float64).reshape(-1)
    scale = np.mean(np.abs(want)) + 1e-12
    rel = np.abs(got - want) / (np.abs(want) + scale)
    assert np.mean(rel > 1e-4) <= 5e-3, (tag, float(np.mean(rel > 1e-4)), float(rel.max()))
    assert np.max(np.abs(got - want)) <= 2 * lr * steps, tag


def _buffers(g, S, A):
    import mobody_b200 as mb
    bufs = {}
    for nm in ("src", "tar", "fake"):
        n = int(g["n_" + nm])
        b = mb.ReplayBuffer(S, A, "cuda", max_size=n)
        b.add_batch({"obss": torch.from_numpy(g[f"{nm}_state"]), "actions": torch.from_numpy(g[f"{nm}_action"]),
                     "next_obss": torch.from_numpy(g[f"{nm}_next_state"]), "rewards": torch.from_numpy(g[f"{nm}_reward"]),
                     "terminals": torch.from_numpy(1.0 - g[f"{nm}_not_done"])})
        assert b.size == n
        bufs[nm] = b
    return bufs


@pytest.mark.parametrize("name", ["train_S17A6_B32.npz", "train_S11A3_B16.npz"])
def test_train_matches_reference_golden(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name))
    S, A, B, seed, n_steps = (int(g[k]) for k in ("S", "A", "B", "seed", "n_steps"))
    ag, _ = cuda_agent(S, A, seed)
    bufs = _buffers(g, S, A)
    ag.fake_replay_buffer = bufs["fake"]
    ag.total_it = 1                                     # steady state: no refresh, like the golden run
    for it in range(n_steps):
        ag.train(bufs["src"], bufs["tar"], B, None, None,
                 _inject={"src": g[f"ind{3 * it}"], "tar": g[f"ind{3 * it + 1}"], "fake": g[f"ind{3 * it + 2}"]})
    torch.cuda.synchronize()
    assert ag.total_it == 1 + n_steps
    for grp, mod in (("pi", ag.policy), ("q", ag.q_funcs), ("qt", ag.target_q_funcs)):
        for k, v in mod.state_dict().items():
            flat = v.cpu().numpy().reshape(-1)
            want = g[f"post_{grp}_{k}_sub"]
            assert rel_err(flat[::37], want) < 1e-4, (grp, k, rel_err(flat[::37], want))
            np.testing.assert_allclose(flat.astype(np.float64).sum(), float(g[f"post_{grp}_{k}_sum"]), rtol=2e-4, atol=1e-4)


@pytest.mark.parametrize("S,A,N,n_true", [(17, 6, 320, 256), (11, 3, 77, 64), (27, 8, 1500, 1200), (27, 8, 10240, 8192)])
def test_train_on_rows_matches_oracle(S, A, N, n_true):
    from mobody_b200 import _ffi
    rng = np.random.default_rng(N)
    ag, st = cuda_agent(S, A, 55)
    RW = _ffi.lib().mobody_row_width(S, A)
    s, a = rng.standard_normal((N, S)).astype(np.float32), rng.uniform(-1, 1, (N, A)).astype(np.float32)
    s2, r = rng.standard_normal((N, S)).astype(np.float32), rng.standard_normal((N, 1)).astype(np.float32)
    nd = (rng.random((N, 1)) > 0.1).astype(np.float32)
    rows = np.zeros((N, RW), np.float32)
    rows[:, :S], rows[:, S:S + A], rows[:, S + A:2 * S + A], rows[:, 2 * S + A:2 * S + A + 1], rows[:, 2 * S + A + 1:2 * S + A + 2] = s, a, s2, r, nd
    rows_d = torch.from_numpy(rows).cuda()
    batch = tuple(torch.from_numpy(x) for x in (s, a, s2, r, nd))
    for it in range(3):
        want = M.train_step(st, batch, n_true, CFG)
        ag.train_on_rows(rows_d, n_true)
        got = ag.loss_scalars()
        for k in ("q_loss", "pi_loss", "bc_loss", "q1_mean", "q_policy", "w_mean", "w_min", "w_max"):
            # w_min / w_max are EXTREME values over the batch of exp(3 q/mean|q|): with mean|q| ~ 0.04 at initialisation an
            # absolute fp32-round-off difference of 2e-6 in one row's q is amplified 75x in the exponent, and the extreme
            # over 8192 rows picks the worst row; they are print-only diagnostics (mobody.py:269-270), held to 1e-3
            tol = 1e-3 if k in ("w_min", "w_max") else 1e-4
            assert abs(got[k] - want[k]) <= tol * (abs(want[k]) + 1e-2), (it, k, got[k], want[k])
    for grp, mod, ref in (("pi", ag.policy, st.policy), ("q", ag.q_funcs, st.q), ("qt", ag.target_q_funcs, st.q_target)):
        for k, v in mod.state_dict().items():
            adam_close(v.cpu().numpy(), ref[k].numpy(), 3e-4, 3, (grp, k))


def test_train_end_to_end_with_refresh_runs():
    """First train() call triggers the synthetic-data refresh (two rollouts + dataset step -> fake buffer), then steps."""
    import mobody_b200 as mb
    from helpers import cuda_dynamics
    S, A = 17, 6
    rng = np.random.default_rng(1)
    ag, _ = cuda_agent(S, A, 3, penalty_type="par", penalty_coef=0.1)
    ag.dynamics, _ = cuda_dynamics(S, A, 3, "halfcheetah", 0.1)

    def ds(n):
        return dict(observations=0.3 * rng.standard_normal((n, S)).astype(np.float32), actions=rng.uniform(-1, 1, (n, A)).astype(np.float32),
                    next_observations=0.3 * rng.standard_normal((n, S)).astype(np.float32), rewards=rng.standard_normal(n).astype(np.float32),
                    terminals=np.zeros(n, bool))
    src, tar = mb.ReplayBuffer(S, A, "cuda"), mb.ReplayBuffer(S, A, "cuda")
    src.convert_D4RL(ds(60000)); tar.convert_D4RL(ds(5000))
    before = ag.policy.network.network[0].weight.detach().clone()
    ag.train(src, tar, 128, None, None)
    assert ag.fake_replay_buffer.size == 50000 + 2000 + 50000            # halfcheetah: nothing terminates, penalty << env_filter
    ag.train(src, tar, 128, None, None)
    torch.cuda.synchronize()
    v = ag.loss_scalars()
    assert np.isfinite(list(v.values())).all() and not torch.equal(before, ag.policy.network.network[0].weight.detach())
    # README headline setting: penalty_type='dara' -> 5000-step classifier prologue + one-off reward relabel, then the same step
    ag2, _ = cuda_agent(S, A, 3, penalty_type="dara", penalty_coef=0.1)
    ag2.dynamics = ag.dynamics
    r0 = src.reward.clone()
    ag2.train(src, tar, 128, None, None)
    assert ag2._t_cls == 5000 and not torch.equal(r0, src.reward)          # classifier trained, source rewards relabelled (:364-378)
    assert float((src.reward - r0).abs().max()) <= 0.1 * 10.0 + 1e-5       # |penalty| is clamped to 10
    r1 = src.reward.clone()
    ag2.train(src, tar, 128, None, None)
    torch.cuda.synchronize()
    assert ag2._t_cls == 5000 and torch.equal(r1, src.reward)              # the prologue runs once
    assert np.isfinite(list(ag2.loss_scalars().values())).all()
    # rollout_from_src (mobody.py:477-510): source-head rollout from 50 000 + 100 starts, classifier-penalised rewards
    ag3, _ = cuda_agent(S, A, 3, penalty_type="par", penalty_coef=0.1, rollout_from_src=1, rollout_from_src_length=1)
    ag3.dynamics = ag.dynamics
    ag3.train(src, tar, 128, None, None)
    assert ag3._t_cls == 1 and ag3.fake_replay_buffer.size == 50000 + 2000 + 50000 + 50100


@pytest.mark.parametrize("S,A,N,n_true", [(17, 6, 77, 64), (27, 8, 1500, 1200)])
def test_weight_gradient_row_splits_agree(S, A, N, n_true):
    """The weight-gradient GEMMs (3xTF32 tensor-core tiles + narrow heads) split the rows `nsplit` ways and Adam adds the
    partial sums in split order: any split count -- one, a ragged one, more splits than 32-row chunks (empty splits) --
    must give the same update up to fp32 summation order, and the same count must give it bit for bit."""
    from mobody_b200 import _ffi
    rng = np.random.default_rng(7 * N)
    RW = _ffi.lib().mobody_row_width(S, A)
    rows = np.zeros((N, RW), np.float32)
    rows[:, :2 * S + A] = rng.standard_normal((N, 2 * S + A)).astype(np.float32)
    rows[:, S:S + A] = rng.uniform(-1, 1, (N, A)).astype(np.float32)
    rows[:, 2 * S + A] = rng.standard_normal(N).astype(np.float32)
    rows[:, 2 * S + A + 1] = (rng.random(N) > 0.1).astype(np.float32)
    rows_d = torch.from_numpy(rows).cuda()

    def run(nsplit):
        ag, _ = cuda_agent(S, A, 55)
        for _ in range(2):
            ag.train_on_rows(rows_d, n_true, nsplit=nsplit)
        torch.cuda.synchronize()
        return {f"{g}.{k}": v.detach().cpu().numpy().copy() for g, m in (("pi", ag.policy), ("q", ag.q_funcs), ("qt", ag.target_q_funcs))
                for k, v in m.state_dict().items()}

    base = run(1)
    again = run(1)
    for k in base:
        assert np.array_equal(base[k], again[k]), k                        # fixed summation order: bit-reproducible
    for nsplit in (3, 7, 64):
        other = run(nsplit)
        for k in base:
            adam_close(other[k], base[k], 3e-4, 2, (nsplit, k))


_PARAM_DIGEST = r"""
import hashlib, sys, os
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import numpy as np, torch
from helpers import cuda_agent
from mobody_b200 import _ffi
h = hashlib.sha256()
for S, A, N, n_true, steps in ((17, 6, 320, 256, 30), (27, 8, 5120, 4096, 6)):
    rng = np.random.default_rng(N)
    RW = _ffi.lib().mobody_row_width(S, A)
    rows = np.zeros((N, RW), np.float32)
    rows[:, :2 * S + A + 1] = rng.standard_normal((N, 2 * S + A + 1)).astype(np.float32)
    rows[:, S:S + A] = rng.uniform(-1, 1, (N, A)).astype(np.float32)
    rows[:, 2 * S + A + 1] = (rng.random(N) > 0.1).astype(np.float32)
    rows_d = torch.from_numpy(rows).cuda()
    ag, _ = cuda_agent(S, A, 9)
    for _ in range(steps):
        ag.train_on_rows(rows_d, n_true)
    torch.cuda.synchronize()
    for m in (ag.policy, ag.q_funcs, ag.target_q_funcs):
        for v in m.state_dict().values():
            h.update(v.detach().cpu().numpy().tobytes())
    h.update(np.asarray(list(ag.loss_scalars().values()), np.float32).tobytes())
print("DIGEST", h.hexdigest())
"""


def test_launch_mode_and_tiling_switches_in_subprocess():
    """The update is a chain of kernels with fixed-order reductions, so how the chain is LAUNCHED must not change a bit of
    it: programmatic dependent launch on / off (MOBODY_PDL) give identical parameters and losses after 30 small-batch and
    6 large-batch updates (a missing grid dependency would show up as a difference)."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def digest(**env):
        r = subprocess.run([sys.executable, "-c", _PARAM_DIGEST], env=dict(os.environ, **env), capture_output=True, text=True,
                           timeout=300, cwd=root)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return [ln.split()[1] for ln in r.stdout.splitlines() if ln.startswith("DIGEST")][0]

    base = digest(MOBODY_PDL="1")
    assert base == digest(MOBODY_PDL="0")
    assert base == digest(MOBODY_TRAIN_SIDE="0")          # large-batch update: side-stream overlap on / off


@pytest.mark.parametrize("name", ["train_S17A6_B32.npz"])
def test_optimizer_checkpoints_match_reference_and_round_trip(golden_dir, name, tmp_path):
    """MOBODY.save / load write and read the reference's FOUR files (mobody.py:584-594).  The optimizer files are
    torch.optim.Adam.state_dict()s: after the golden's train steps the fused kernels' moments must equal the reference's
    exp_avg / exp_avg_sq / step per parameter index and the param_groups must be the reference's; a saved agent must
    resume bit-identically; and an optimizer file written by a stock torch.optim.Adam (what the reference writes) must load."""
    import json
    g = np.load(os.path.join(golden_dir, name))
    S, A, B, seed, n_steps = (int(g[k]) for k in ("S", "A", "B", "seed", "n_steps"))
    ag, _ = cuda_agent(S, A, seed)
    bufs = _buffers(g, S, A)
    ag.fake_replay_buffer = bufs["fake"]
    ag.total_it = 1
    inj = lambda it: {"src": g[f"ind{3 * it}"], "tar": g[f"ind{3 * it + 1}"], "fake": g[f"ind{3 * it + 2}"]}   # noqa: E731
    for it in range(n_steps):
        ag.train(bufs["src"], bufs["tar"], B, None, None, _inject=inj(it))
    torch.cuda.synchronize()
    for grp, opt in (("q", ag.q_optimizer), ("pi", ag.policy_optimizer)):
        sd = opt.state_dict()
        want_groups = json.loads(str(g[f"opt_{grp}_groups"]))
        got_groups = json.loads(json.dumps(sd["param_groups"]))
        assert got_groups == want_groups, grp                                   # same keys, lr, betas, eps, param indices
        assert sorted(sd["state"]) == list(range(len(want_groups[0]["params"])))
        for i, stt in sd["state"].items():
            assert float(stt["step"]) == float(g[f"opt_{grp}_{i}_step"]) == n_steps
            for mk, tol in (("exp_avg", 1e-4), ("exp_avg_sq", 2e-4)):
                flat = stt[mk].cpu().numpy().reshape(-1)
                want = g[f"opt_{grp}_{i}_{mk}_sub"]
                scale = np.abs(want).mean() + 1e-30
                bad = np.abs(flat[::37] - want) > tol * (np.abs(want) + scale)
                assert bad.mean() <= 5e-3, (grp, i, mk, float(bad.mean()))        # (ReLU-edge outliers: see adam_close)
    # round trip: save, load into a fresh agent, continue both with the same batch -> bit-identical parameters
    fn = str(tmp_path / "ckpt")
    ag.save(fn)
    assert sorted(os.listdir(tmp_path)) == ["ckpt_actor", "ckpt_actor_optimizer", "ckpt_critic", "ckpt_critic_optimizer"]
    ag2, _ = cuda_agent(S, A, seed + 1)                                          # different initial weights
    ag2.load(fn)
    ag2.target_q_funcs.load_state_dict(ag.target_q_funcs.state_dict())           # (targets are not checkpointed by the reference either)
    assert ag2._t_q == ag._t_q == n_steps and ag2._t_pi == n_steps
    rows = bufs["src"].sample_rows(80, np.arange(80))
    ag.train_on_rows(rows, 64); ag2.train_on_rows(rows, 64)
    torch.cuda.synchronize()
    for m1, m2 in ((ag.policy, ag2.policy), (ag.q_funcs, ag2.q_funcs)):
        for (k, v1), v2 in zip(m1.state_dict().items(), m2.state_dict().values()):
            assert torch.equal(v1, v2), k
    # a file written by stock torch.optim.Adam on the reference's module layout (mobody.py:585) loads and is used
    import copy
    ref_q = copy.deepcopy(ag.q_funcs).cpu()
    ref_opt = torch.optim.Adam(ref_q.parameters(), lr=3e-4)
    x = torch.randn(16, S + A)
    (ref_q.network1(x).sum() + ref_q.network2(x).sum()).backward()
    ref_opt.step(); ref_opt.step()
    torch.save(ref_q.state_dict(), fn + "_critic"); torch.save(ref_opt.state_dict(), fn + "_critic_optimizer")
    ag2.load(fn)
    assert ag2._t_q == 2
    m_ref = ref_opt.state_dict()["state"][2]["exp_avg"]
    (q1_m, _), _ = ag2._moments("q", (ag2.q_funcs.network1, ag2.q_funcs.network2))
    assert q1_m[2].is_cuda and torch.equal(q1_m[2].cpu(), m_ref)
    ag2.train_on_rows(rows, 64)                                                  # continues from the loaded moments
    torch.cuda.synchronize()
    assert ag2._t_q == 3 and float(ag2.q_optimizer.state_dict()["state"][0]["step"]) == 3.0


@pytest.mark.parametrize("override", [dict(advantage=1), dict(scale_Q=0), dict(q_weighted=0)])
def test_non_default_update_branches_run_through_the_torch_path(override):
    """advantage=1 / scale_Q=0 / q_weighted=0 (mobody.py:210-310, 533-559) are off in every shipped config; they must keep
    working (SURVEY section 2 #4) -- through torch autograd on the same device-resident rows and the same optimizers --
    and must match the CPU oracle's restatement of the default math where the branch reduces to it."""
    import mobody_b200 as mb
    S, A, B = 11, 3, 64
    rng = np.random.default_rng(3)
    ag, st = cuda_agent(S, A, 21, **override)

    def ds(n):
        return dict(observations=rng.standard_normal((n, S)).astype(np.float32), actions=rng.uniform(-1, 1, (n, A)).astype(np.float32),
                    next_observations=rng.standard_normal((n, S)).astype(np.float32), rewards=rng.standard_normal(n).astype(np.float32),
                    terminals=(rng.random(n) < 0.1))
    src, tar = mb.ReplayBuffer(S, A, "cuda"), mb.ReplayBuffer(S, A, "cuda")
    src.convert_D4RL(ds(3000)); tar.convert_D4RL(ds(500)); ag.fake_replay_buffer.convert_D4RL(ds(800))
    ag.total_it = 1
    before = {k: v.clone() for k, v in ag.policy.state_dict().items()}
    qb = {k: v.clone() for k, v in ag.q_funcs.state_dict().items()}
    vb = {k: v.clone() for k, v in ag.v_func.state_dict().items()}
    for _ in range(3):
        ag.train(src, tar, B, None, None)
    torch.cuda.synchronize()
    assert ag._t_q == 3 and ag._t_pi == 3 and float(ag.q_optimizer.state_dict()["state"][0]["step"]) == 3.0
    assert any(not torch.equal(v, before[k]) for k, v in ag.policy.state_dict().items())
    assert any(not torch.equal(v, qb[k]) for k, v in ag.q_funcs.state_dict().items())
    moved_v = any(not torch.equal(v, vb[k]) for k, v in ag.v_func.state_dict().items())
    assert moved_v == bool(override.get("advantage", 0))                          # the value function trains only with advantage=1
    assert all(bool(torch.isfinite(v).all()) for v in ag.policy.state_dict().values())
    # switching back to the default config continues on the fused kernels from the same Adam state
    ag.config.update(advantage=0, scale_Q=1, q_weighted=1)
    ag.train(src, tar, B, None, None)
    torch.cuda.synchronize()
    assert ag._t_q == 4 and np.isfinite(list(ag.loss_scalars().values())).all()


def test_torch_path_equals_fused_path_on_the_default_math():
    """Cross-check of the two update paths: with the default flags forced through the torch path (autograd) one update must
    give the parameters the fused kernels give (1e-4), which pins the torch path's formulas to the golden-checked ones."""
    from mobody_b200 import _ffi
    S, A, N, n_true = 17, 6, 320, 256
    rng = np.random.default_rng(11)
    RW = _ffi.lib().mobody_row_width(S, A)
    rows = np.zeros((N, RW), np.float32)
    rows[:, :2 * S + A + 1] = rng.standard_normal((N, 2 * S + A + 1)).astype(np.float32)
    rows[:, S:S + A] = rng.uniform(-1, 1, (N, A)).astype(np.float32)
    rows[:, 2 * S + A + 1] = (rng.random(N) > 0.1).astype(np.float32)
    rows_d = torch.from_numpy(rows).cuda()
    a1, _ = cuda_agent(S, A, 9)
    a2, _ = cuda_agent(S, A, 9)
    for _ in range(2):
        a1.train_on_rows(rows_d, n_true)
        a2._train_torch_path(rows_d, n_true, None, None)
    torch.cuda.synchronize()
    for m1, m2, tag in ((a1.policy, a2.policy, "pi"), (a1.q_funcs, a2.q_funcs, "q"), (a1.target_q_funcs, a2.target_q_funcs, "qt")):
        for (k, v1), v2 in zip(m1.state_dict().items(), m2.state_dict().values()):
            adam_close(v1.cpu().numpy(), v2.cpu().numpy(), 3e-4, 2, (tag, k))
