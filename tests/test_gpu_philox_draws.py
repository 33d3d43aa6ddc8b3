"""The device's own Philox draws (production mode: no injected eps / idx / noise) against the numpy oracle.

Step noise and member picks are recovered from the step kernel's outputs alone.  The kernel writes every member's
ensemble mean (info["samples"], [7,B,S]); from them the float64 ensemble std sd follows, and the noise it drew is
eps_k = (next_obs - mean[member]) / sd.  eps_k is held, element by element, to oracle.philox.rollout_noise:
  fp32 (precise logf / sincosf):   |eps_k - eps| <= 2e-6 (1 + |eps|)     + 2 ulp(next_obs) / sd
  bf16x2, fp16 (SFU sine/cosine):  |eps_k - eps| <= 2e-6 (1 + |eps| + r) + 2 ulp(next_obs) / sd
with r the Box-Muller radius of the entry (the derivation is next to philox_normal1 in csrc/philox.cuh).  The member is
bit-exact: the oracle's member is the only elite whose mean[e] + eps sd reproduces next_obs within that bound.

The classifier and dynamics-fit kernels are run twice from identical state: once drawing their own noise and once
with the oracle's restatement of that stream injected (oracle.philox.classifier_noise / fit_noise).  Losses, the
gradients recovered from Adam's first moments, and the parameters must agree; injecting a neighbouring draw or the
other classifier's noise must not.
"""
import numpy as np
import pytest
import torch

import test_grad_reference as R
from helpers import cuda_agent, cuda_dynamics
from oracle import mobody_oracle as M
from oracle.philox import (classifier_noise, fit_noise, philox4x32_10, rollout_elite_slot, rollout_noise, rollout_radius,
                           STREAM_CLSN)
from test_gpu_grad_parity import _moments, _snap
from test_gpu_model_eval import CASES as EVAL_CASES, check_against_float64_oracle
from test_gpu_train import adam_close
from test_philox_streams import EXTREME_NOISE_WORDS, EXTREME_S, EXTREME_SEED, EXTREME_STEP, SEED_HI

pytestmark = pytest.mark.gpu

SFU = {"fp32": False, "bf16x2": True, "fp16": True}       # philox_normal1's __sinf / __cosf
WORST = {}                                                 # precision -> worst |eps_k - eps| / bound over the file


def _report(prec, ratio):
    WORST[prec] = max(WORST.get(prec, 0.0), ratio)
    print(f"\n[philox step noise] {prec}: worst err/bound {ratio:.3f} (file so far {WORST[prec]:.3f})")


def _step(dyn, obs, act, *, step, seed, row0=0, row_ids=None):
    from mobody_b200.dynamics import StepWorkspace
    dyn.seed = seed
    ws = StepWorkspace(obs.shape[0], obs.shape[1], act.shape[1], obs.device)
    dyn.launch_step(obs, act, ws, step=step, row0=row0, row_ids=row_ids)
    torch.cuda.synchronize()
    return ws


def check_step_noise(prec, next_obs, mean, seed, step, gids, elites):
    """Recover the noise and the member of every row from next_obs [n,S] and the kernel's means [7,n,S]; hold them to the
    oracle's draws for the global row ids ``gids``.  Returns the worst err / bound."""
    nobs = np.asarray(next_obs, np.float64)
    mean = np.asarray(mean, np.float64)
    n, S = nobs.shape
    assert np.isfinite(nobs).all()
    elites = np.asarray(elites)
    gids = np.asarray(gids, np.uint64)
    member = elites[rollout_elite_slot(seed, step, gids, len(elites))]
    eps = rollout_noise(seed, step, gids, S).astype(np.float64)
    sd = mean.std(axis=0, ddof=1)
    assert (sd > 0).all()
    bound = 2e-6 * (1.0 + np.abs(eps) + (rollout_radius(seed, step, gids, S) if SFU[prec] else 0.0))
    bound = bound + 2.0 * np.spacing(np.abs(np.asarray(next_obs, np.float32))).astype(np.float64) / sd
    rows = np.arange(n)
    eps_k = (nobs - mean[member, rows]) / sd
    ratio = np.abs(eps_k - eps) / bound
    assert ratio.max() <= 1.0, (prec, float(ratio.max()), np.unravel_index(ratio.argmax(), ratio.shape))
    uniq = np.unique(elites)
    if len(uniq) > 1:
        # member pick: every other elite misses next_obs by more than the bound in some dimension of every row ...
        for e in uniq:
            miss = (np.abs(nobs - (mean[e] + eps * sd)) / (bound * sd)).max(axis=1)
            assert (miss[member != e] > 1.0).all(), (prec, int(e))
        # ... and that is no accident of a bound wider than the members' spread
        gap = np.min([(np.abs(mean[e] - mean[member, rows]) / (bound * sd)).max(axis=1)[member != e].min(initial=np.inf)
                      for e in uniq])
        assert gap > 10.0, gap
    return float(ratio.max())


# ----------------------------------------------------------------------------------------------------------- step
def _grid():
    out = []
    for prec, widths in (("fp32", (2, 3, 5, 17, 40, 64, 128)), ("bf16x2", (2, 3, 5, 17, 40, 47)), ("fp16", (2, 3, 5, 17, 40, 55))):
        for S in widths:
            out.append((prec, S, 6 if S == 17 else 2))
    return out


@pytest.mark.parametrize("prec,S,A", _grid())
def test_step_noise_and_member_picks(prec, S, A):
    """Production-mode step at every precision and width: batches of 1, 129 and 1 000 rows; row0 0, 2^32 - 64 (the batch
    straddles the high row word) and 2^40 + 3; step words 0, 7 and 2^32 - 1; 1, 5 or 7 elites in an order where slot !=
    member; explicit descending, gapped row ids across 2^32 with duplicates; seeds 1234 and 2^32 + 1234 give the same
    result bit for bit (only the low seed word keys the generator)."""
    from mobody_b200.dynamics import tc_step_supports
    assert prec == "fp32" or tc_step_supports(S, A, prec)
    dyn, _ = cuda_dynamics(S, A, 3, "halfcheetah", 1.0, precision=prec)
    rng = np.random.default_rng(S * 10 + len(prec))

    def inputs(B):
        obs = torch.from_numpy((0.5 * rng.standard_normal((B, S))).astype(np.float32)).cuda()
        return obs, torch.from_numpy(rng.uniform(-1, 1, (B, A)).astype(np.float32)).cuda()

    worst = 0.0
    for B, row0, step, elites in ((1000, 0, 0, [6, 0, 3, 5, 1]), (129, (1 << 32) - 64, 7, [3, 6, 0, 2, 5, 1, 4]),
                                  (1, (1 << 40) + 3, (1 << 32) - 1, [4])):
        dyn.model.set_elites(elites)
        obs, act = inputs(B)
        ws = _step(dyn, obs, act, step=step, seed=1234, row0=row0)
        worst = max(worst, check_step_noise(prec, ws.next_obs.cpu(), ws.mean.cpu(), 1234, step, row0 + np.arange(B), elites))
        hi = _step(dyn, obs, act, step=step, seed=SEED_HI, row0=row0)
        for k in ("next_obs", "reward", "penalty", "terminal", "mean"):
            assert torch.equal(getattr(hi, k), getattr(ws, k)), (k, B)
    # explicit row ids: descending with gaps of 1..3 across 2^32, the first five repeated at the end
    dyn.model.set_elites([6, 0, 3, 5, 1])
    ids = (1 << 32) + 60 - np.cumsum(rng.integers(1, 4, 124))
    ids = np.concatenate([ids, ids[:5]])
    assert ids.min() < (1 << 32) <= ids.max() and len(ids) == 129
    obs, act = inputs(len(ids))
    obs[-5:], act[-5:] = obs[:5], act[:5]
    ws = _step(dyn, obs, act, step=7, seed=1234, row_ids=torch.from_numpy(ids).cuda())
    worst = max(worst, check_step_noise(prec, ws.next_obs.cpu(), ws.mean.cpu(), 1234, 7, ids, [6, 0, 3, 5, 1]))
    assert torch.equal(ws.next_obs[-5:], ws.next_obs[:5]) and torch.equal(ws.reward[-5:], ws.reward[:5])
    _report(prec, worst)


@pytest.mark.parametrize("prec", ["fp32", "bf16x2", "fp16"])
def test_step_noise_at_the_extreme_words(prec):
    """Rows whose noise word is at an end of the uniform range (x >> 9 = 2^23 - 1: r = 3.45e-4; x >> 9 = 0: r = 5.77), fed
    through explicit row ids, the first one twice: the sample is finite and inside the bound at every word."""
    S, A = EXTREME_S, 6
    dyn, _ = cuda_dynamics(S, A, 3, "halfcheetah", 1.0, precision=prec)
    ids = np.array([c[0] for c in EXTREME_NOISE_WORDS] + [EXTREME_NOISE_WORDS[0][0]])
    rng = np.random.default_rng(4)
    obs = torch.from_numpy((0.5 * rng.standard_normal((len(ids), S))).astype(np.float32)).cuda()
    act = torch.from_numpy(rng.uniform(-1, 1, (len(ids), A)).astype(np.float32)).cuda()
    obs[-1], act[-1] = obs[0], act[0]
    elites = dyn.model.elites.cpu().numpy()
    ws = _step(dyn, obs, act, step=EXTREME_STEP, seed=EXTREME_SEED, row_ids=torch.from_numpy(ids).cuda())
    nobs, mean = ws.next_obs.cpu().numpy(), ws.mean.cpu().numpy()
    _report(prec, check_step_noise(prec, nobs, mean, EXTREME_SEED, EXTREME_STEP, ids, elites))
    member = elites[rollout_elite_slot(EXTREME_SEED, EXTREME_STEP, ids.astype(np.uint64), len(elites))]
    eps = rollout_noise(EXTREME_SEED, EXTREME_STEP, ids, S)
    sd = mean.astype(np.float64).std(axis=0, ddof=1)
    for i, (row, blk, w, _) in enumerate(EXTREME_NOISE_WORDS):
        j = 4 * blk + w
        got = (float(nobs[i, j]) - float(mean[member[i], i, j])) / sd[i, j]
        print(f"  row {row} dim {j}: eps {eps[i, j]:+.6e} recovered {got:+.6e}")
    assert np.array_equal(nobs[-1], nobs[0])


# ----------------------------------------------------------------------------------------------------------- rollout
@pytest.mark.parametrize("prec", ["fp32", "bf16x2"])
def test_rollout_noise_is_keyed_on_the_global_row_id(prec):
    """mobody_rollout, production mode, T = 3, rows that terminate: after each compaction the surviving rows keep their
    global ids (row0 + start index, across 2^32), and the noise of step t recovered from the packed transitions and that
    step's ensemble means is the noise keyed on those ids and step word step0 + t."""
    S, A, B, row0, step0, seed = 11, 3, 300, (1 << 32) - 100, 5, 1234
    dyn, _ = cuda_dynamics(S, A, 3, "hopper", 5.0, precision=prec, h0=0.8, t3_gain=2.0)
    dyn.seed = seed
    elites = [6, 0, 3, 5, 1]
    dyn.model.set_elites(elites)
    ag, _ = cuda_agent(S, A, 3, env_filter=1e9)
    ag.dynamics = dyn
    obs = torch.from_numpy((np.r_[0.8, np.zeros(S - 1)][None] + 0.1 * np.random.default_rng(6).standard_normal((B, S)))
                           .astype(np.float32)).cuda()
    worst, prev = 0.0, None
    for T in (1, 2, 3):                  # the rollout of length T leaves step T - 1's ensemble means in its workspace
        _, info = ag.rollout_device(obs, T, row0=row0, step0=step0)
        ws = ag._rollout_workspace(T, B, S, A, 0)
        counts, t = info["rows_per_step"], T - 1
        n, off = counts[t], sum(counts[:t])
        assert info["kept"] == sum(counts)
        ids = ws["row_ids"][t, :n].cpu().numpy()
        if t == 0:
            assert np.array_equal(ids, row0 + np.arange(B))
        else:
            assert np.array_equal(ids, prev[0][prev[1] == 0]) and 0 < n < len(prev[0])
        rows = info["packed"][off:off + n].cpu().numpy()
        worst = max(worst, check_step_noise(prec, rows[:, S + A:2 * S + A], ws["mean"][:, :n].cpu().numpy(), seed, step0 + t, ids,
                                            elites))
        prev = (ids, rows[:, 2 * S + A + 1])
    _report(prec, worst)


@pytest.mark.parametrize("prec", ["fp32", "bf16x2"])
def test_model_eval_at_the_last_row_and_step_words(prec):
    """mobody_model_eval with start ids across 2^32 (row0 = 2^32 - 10) and the largest step base it accepts
    (step0 = 2^32 - H, so the last step uses step word 2^32 - 1), against the float64 reference."""
    env, S, A, h0, t3, kind, penalized = EVAL_CASES[0]
    H = 24
    check_against_float64_oracle(env, S, A, h0, t3, kind, penalized, prec, row0=(1 << 32) - 10, step0=(1 << 32) - H, H=H)


# ----------------------------------------------------------------------------------------------------------- classifier
CLS_S, CLS_A, CLS_N, CLS_SEED, CLS_STD = 17, 6, 256, 1234, 0.5
CLS_EXTREME = (1202, 1, 201, 1, 2)     # (draw, classifier, row, block, word): x >> 9 = 2^23 - 1 in the sa noise of seed 1234


def _cls_batch(draw):
    """Rows [N, RW] and labels whose classifier ReLU gates sit clear of their kinks under the draw's noise."""
    from mobody_b200 import _ffi
    S, A, N = CLS_S, CLS_A, CLS_N
    params = R.f64(M.ClassifierState(S, A, 11).params)
    n_sas, n_sa = (torch.from_numpy(classifier_noise(CLS_SEED, draw, N, K, k)).double() for k, K in ((0, 2 * S + A), (1, S + A)))
    rng = np.random.default_rng(draw)
    s, a, s2 = torch.zeros(N, S, dtype=torch.float64), torch.zeros(N, A, dtype=torch.float64), torch.zeros(N, S, dtype=torch.float64)
    label = torch.from_numpy((rng.random(N) < 0.5).astype(np.int64))
    todo = torch.ones(N, dtype=torch.bool)
    for _ in range(20):
        m = int(todo.sum())
        s[todo] = torch.from_numpy(rng.standard_normal((m, S)).astype(np.float32)).double()
        a[todo] = torch.from_numpy(rng.uniform(-1, 1, (m, A)).astype(np.float32)).double()
        s2[todo] = (s[todo] + torch.from_numpy(0.3 * rng.standard_normal((m, S))) + 0.25 * label[todo, None]).float().double()
        todo = ~torch.as_tensor(np.asarray(R.classifier_rows_ok(params, s, a, s2, n_sas, n_sa, CLS_STD)))
        if not todo.any():
            break
    assert not todo.any()
    rows = torch.zeros(N, _ffi.lib().mobody_row_width(S, A), dtype=torch.float32)
    rows[:, :S], rows[:, S:S + A], rows[:, S + A:2 * S + A] = s.float(), a.float(), s2.float()
    return rows.cuda(), label.to(torch.int32).cuda()


def _cls_step(rows, label, draw, noise=None):
    """One classifier step from the same initial state at Philox draw ``draw`` -> (losses, gradients, parameters)."""
    ag, _ = cuda_agent(CLS_S, CLS_A, 11, penalty_type="dara", penalty_coef=1.0, gaussian_noise_std=CLS_STD, actor_lr=3e-4,
                       penalize_fake=0)
    ag.config["seed"] = CLS_SEED                           # the classifier's Philox key
    ag.classifier.load_state_dict(M.ClassifierState(CLS_S, CLS_A, 11).params)
    ag._t_cls = draw - 1                                   # the step takes draw (and Adam step) _t_cls + 1
    kw = {} if noise is None else dict(noise_sas=noise[0], noise_sa=noise[1])
    losses = ag.classifier_step_on_rows(rows, label, **kw).cpu().numpy().astype(np.float64)
    m, _ = _moments(ag._opts["cls"], ag.classifier)
    grads = {k: R.grad_from_moments(np.zeros(v.shape), v) for k, v in m.items()}
    return losses, grads, _snap(ag.classifier)


def _cls_ratio(a, b):
    """max(loss err / 1e-5 |loss|, gradient err / 1e-4 (|g| + mean |g|)) of run a against run b: <= 1 is a match."""
    loss = float(np.max(np.abs(a[0] - b[0]) / (1e-5 * np.abs(b[0]))))
    return max(loss, max(R.strict_ratio(a[1][k], b[1][k]) for k in b[1]))


def _cls_noise(draw, swap=False):
    S, A, N = CLS_S, CLS_A, CLS_N
    ks = (1, 0) if swap else (0, 1)
    return classifier_noise(CLS_SEED, draw, N, 2 * S + A, ks[0]), classifier_noise(CLS_SEED, draw, N, S + A, ks[1])


def test_classifier_noise_is_the_keyed_stream():
    draw = 9
    rows, label = _cls_batch(draw)
    own = _cls_step(rows, label, draw)
    assert all(bool(torch.isfinite(v).all()) for v in own[2].values())
    r = _cls_ratio(own, _cls_step(rows, label, draw, _cls_noise(draw)))
    wrong_draw = _cls_ratio(own, _cls_step(rows, label, draw, _cls_noise(draw + 1)))
    swapped = _cls_ratio(own, _cls_step(rows, label, draw, _cls_noise(draw, swap=True)))
    print(f"\n[philox classifier] err/bound {r:.3f}; injected draw + 1: {wrong_draw:.1f}; sas / sa swapped: {swapped:.1f}")
    assert r <= 1.0
    assert wrong_draw > 10.0 and swapped > 10.0                 # the comparison tells the streams apart


def test_classifier_noise_at_the_top_word():
    """A draw whose sa noise has x >> 9 = 2^23 - 1 (u = 1 - 2^-24) in a row of the batch: parameters finite, and the step
    matches the one with the oracle's noise injected."""
    draw, k, row, blk, w = CLS_EXTREME
    out = philox4x32_10(np.array([row, (k << 16) | blk, draw, 0], np.uint32), np.array([CLS_SEED, STREAM_CLSN], np.uint32))
    assert int(out[w]) >> 9 == (1 << 23) - 1 and row < CLS_N and 4 * blk + w < CLS_S + CLS_A
    rows, label = _cls_batch(draw)
    own, inj = _cls_step(rows, label, draw), _cls_step(rows, label, draw, _cls_noise(draw))
    assert all(bool(torch.isfinite(v).all()) for v in own[2].values())
    r = _cls_ratio(own, inj)
    print(f"\n[philox classifier, top word] err/bound {r:.3f}")
    assert r <= 1.0
    for key in own[2]:
        adam_close(own[2][key].numpy(), inj[2][key].numpy(), 3e-4, 1, key)


# ----------------------------------------------------------------------------------------------------------- dynamics fit
def _fit_run(S, A, N, B, lo, use_trg, draw, seed, inject):
    dyn, _ = cuda_dynamics(S, A, 9, "walker2d", 1.0)
    dyn.seed = seed
    dyn._fit_state()["draw"] = draw
    rng = np.random.default_rng(S + N)
    data = [torch.from_numpy(rng.standard_normal((7, N, w)).astype(np.float32)).cuda() for w in (S, A, S, 1)]
    data[0][..., 0] += 1.25
    kw = {}
    if inject:
        kw = dict(eps_latent=fit_noise(1234, draw, 1, 6 * 7 * B * 16).reshape(6, 7, B, 16),
                  eps_next=fit_noise(1234, draw, 2, 7 * B * S).reshape(7, B, S))
    sc = dyn.fit_batch(use_trg, *data, rows=B, lo=lo, **kw).cpu().numpy().astype(np.float64)
    st = dyn._fit_state()
    out = {}
    for lay in M.fit_trained_layers(use_trg):
        for i, sfx in enumerate(("weight", "bias")):
            out[f"{lay}.{sfx}"] = tuple(x.cpu().numpy().astype(np.float64) for x in
                                        (getattr(getattr(dyn.model, lay), sfx).detach(), st["m"][lay][i], st["v"][lay][i]))
    return sc[:6], out


@pytest.mark.parametrize("S,A,N,B,lo,use_trg", [(17, 6, 300, 64, 100, True), (11, 3, 37, 37, 0, False)])
def test_fit_noise_is_the_keyed_stream(S, A, N, B, lo, use_trg):
    """fit_batch drawing its own noise (seed 2^32 + 1234) == fit_batch with fit_noise(1234, draw, 1 / 2) injected: loss
    scalars, gradients (from the first moments), second moments and parameters.  The (17, 6) case is a 64-row window
    at row 100 of 300-row epoch tensors: the noise is keyed on the row's index in the batch, not in the epoch tensor."""
    draw, lr = 5, 1e-3
    own, inj = _fit_run(S, A, N, B, lo, use_trg, draw, SEED_HI, False), _fit_run(S, A, N, B, lo, use_trg, draw, SEED_HI, True)
    assert np.all(np.abs(own[0] - inj[0]) <= 1e-5 * np.abs(inj[0])), (own[0], inj[0])
    worst = 0.0
    for k, (p, m, v) in inj[1].items():
        po, mo, vo = own[1][k]
        assert np.isfinite(po).all(), k
        worst = max(worst, R.strict_ratio(mo * 10.0, m * 10.0))
        assert R.strict_ratio(vo, v, R.V_TOL) <= 1.0, k
        adam_close(po, p, lr, 1, k)
    print(f"\n[philox dynfit] gradient err/bound {worst:.3f}")
    assert worst <= 1.0
