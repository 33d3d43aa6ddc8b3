"""Gradients of the update kernels against float64 autograd, element by element, across the shapes the C ABI accepts.

Before every step the parameters, target critics, Adam moments and step counts are read back from the device; the
oracle (M.train_step / M.classifier_update / M.fit_step) runs on them in float64, so multi-step cases never drift.  The
kernel's gradient is recovered from its moments and held to 1e-4 * (|g_ref| + mean |g_ref|) on EVERY element; batches
are conditioned away from ReLU / min kinks (test_grad_reference).  Adam's and Polyak's arithmetic are checked from the
kernel's own moments; tensors a step must not touch must stay bit-identical.

Train-step cases come in two kinds.  Gradient cases set critic_lr = 0: the critics' moments still take the gradient but
their weights stay put (p - 0 * x = p), so the actor's gradient -- taken on the critics after their Adam step -- is fully
determined by the state read before the step.  Adam cases use the real learning rates for three steps and check the
critic gradient, the Adam / Polyak arithmetic of every tensor and the loss scalars.

Each case prints one GRADPARITY line: rows dropped by the kink margin and the worst err / bound per kernel family.
"""
from collections import OrderedDict

import numpy as np
import pytest
import torch

import test_grad_reference as R
from helpers import cuda_agent, cuda_dynamics, rel_err, rel_err_strict
from oracle import mobody_oracle as M

pytestmark = pytest.mark.gpu
CFG = dict(gamma=0.99, tau=0.005, actor_lr=3e-4, critic_lr=3e-4, weight=2.5, bc_coef=1.0, max_action=1.0)
LOSS_KEYS = ("q_loss", "pi_loss", "bc_loss", "q1_mean", "q_policy", "w_mean", "w_min", "w_max")


def _snap(mod):
    return OrderedDict((k, v.detach().cpu().clone()) for k, v in mod.named_parameters())


def _moments(opt, mod):
    m = OrderedDict((k, opt.state[p]["exp_avg"].cpu().clone()) for k, p in mod.named_parameters())
    v = OrderedDict((k, opt.state[p]["exp_avg_sq"].cpu().clone()) for k, p in mod.named_parameters())
    return m, v


def _report(kind, case, worst, dropped=None):
    fam = {k: round(max(v.values()), 4) for k, v in worst.items() if v}
    print(f"GRADPARITY {kind} {case} dropped={dropped} worst={fam}")


class _Worst(dict):
    def add(self, family, ratios):
        d = self.setdefault(family, {})
        for k, r in ratios.items():
            d[k] = max(d.get(k, 0.0), r)


def _check_adam(worst, family, p0, p1, m1, v1, t, lr, tag):
    rat = {k: R.adam_ratio(p0[k], p1[k], m1[k], v1[k], t, lr) for k in p0}
    bad = {k: r for k, r in rat.items() if r > 1.0}
    assert not bad, (tag, family, bad)
    worst.add(family, rat)


def _check_moments(worst, family, m0, m1, v0, v1, g_ref, tag):
    """Gradient (from m) and its square (from v) against the float64 reference, every element."""
    got = {k: R.grad_from_moments(m0[k], m1[k]) for k in g_ref}
    worst.add(family, R.check_grads(got, g_ref, (tag, family)))
    got2 = {k: R.sq_grad_from_moments(v0[k], v1[k]) for k in g_ref}
    worst.add(family + "_v", R.check_grads(got2, {k: g ** 2 for k, g in g_ref.items()}, (tag, family, "v"), R.V_TOL))


# ----------------------------------------------------------------------------------------------------- train step
def _train_pool(S, A, n, rng):
    s, s2, r = (torch.from_numpy(rng.standard_normal(sh)) for sh in ((n, S), (n, S), (n, 1)))
    a = torch.from_numpy(rng.uniform(-1, 1, (n, A)))
    nd = torch.from_numpy((rng.random((n, 1)) > 0.1).astype(np.float64))
    return tuple(x.float().double() for x in (s, a, s2, r, nd))            # fp32-representable inputs


def _run_train(S, A, N, n_true, nsplit, steps, critic_lr, seed):
    from mobody_b200 import _ffi
    cfg = dict(CFG, critic_lr=critic_lr)
    ag, _ = cuda_agent(S, A, seed, critic_lr=critic_lr)
    ag.target_q_funcs.load_state_dict(M.AgentState(S, A, seed + 50).q)    # targets != critics: Polyak is not a no-op
    rng = np.random.default_rng(seed * 7919 + N)
    RW = _ffi.lib().mobody_row_width(S, A)
    oq, opi = ag._opts["q"], ag._opts["pi"]
    v_func0 = _snap(ag.v_func)
    worst, dropped = _Worst(), []
    grad_case = critic_lr == 0.0
    for it in range(steps):
        pol, q, qt = _snap(ag.policy), _snap(ag.q_funcs), _snap(ag.target_q_funcs)
        (mq, vq), (mpi, vpi) = _moments(oq, ag.q_funcs), _moments(opi, ag.policy)
        t_q, t_pi = ag._t_q, ag._t_pi
        for _ in range(16):
            pool = _train_pool(S, A, N + N // 4 + 64, rng)
            ok = R.train_rows_ok(R.f64(pol), R.f64(q), pool[0], pool[1], cfg["max_action"])
            idx = R.first_rows(ok, N)
            batch = tuple(x[idx] for x in pool)
            if R.td_cancellation(R.f64(pol), R.f64(q), R.f64(qt), batch, cfg["gamma"], cfg["max_action"]) >= R.TD_MIN_CANCELLATION:
                break
        dropped.append(1.0 - float(ok[:idx[-1] + 1].double().mean()))
        st = R.agent_state64(pol, q, qt, mq, vq, mpi, vpi, t_q, t_pi)
        gq_ref, gpi_ref, losses = R.train_reference(st, batch, n_true, cfg)
        rows = torch.zeros(N, RW, dtype=torch.float32)
        c0 = 0
        for x in batch:
            rows[:, c0:c0 + x.shape[1]] = x.float()
            c0 += x.shape[1]
        ag.train_on_rows(rows.cuda(), n_true, nsplit=nsplit)
        got = ag.loss_scalars()
        tag = (S, A, N, n_true, nsplit, it)
        for k in LOSS_KEYS:
            tol = 1e-3 if k in ("w_min", "w_max") else 1e-4                # extremes of exp(3 q / mean|q|): see test_gpu_train
            assert abs(got[k] - losses[k]) <= tol * (abs(losses[k]) + 1e-2), (tag, k, got[k], losses[k])
        pol1, q1, qt1 = _snap(ag.policy), _snap(ag.q_funcs), _snap(ag.target_q_funcs)
        (mq1, vq1), (mpi1, vpi1) = _moments(oq, ag.q_funcs), _moments(opi, ag.policy)
        assert ag._t_q == t_q + 1 and ag._t_pi == t_pi + 1
        _check_moments(worst, "critic", mq, mq1, vq, vq1, gq_ref, tag)
        if grad_case:
            _check_moments(worst, "actor", mpi, mpi1, vpi, vpi1, gpi_ref, tag)
            for k in q:
                assert torch.equal(q[k], q1[k]), (tag, k)                   # p - 0 * x = p
        _check_adam(worst, "adam", q, q1, mq1, vq1, t_q + 1, critic_lr, tag)
        _check_adam(worst, "adam", pol, pol1, mpi1, vpi1, t_pi + 1, cfg["actor_lr"], tag)
        rat = {k: R.polyak_ratio(qt[k], qt1[k], q1[k], cfg["tau"]) for k in qt}
        assert max(rat.values()) <= 1.0, (tag, rat)
        assert any(not torch.equal(qt[k], qt1[k]) for k in qt)
        worst.add("polyak", rat)
    for k, v in _snap(ag.v_func).items():
        assert torch.equal(v, v_func0[k]), k                                 # the value function is not part of the step
    return worst, max(dropped)


# (S, A, N, n_true, nsplit): S, S+A and 2S+A below, on and past the 64 / 128-column K-block edges; N on both sides of the
# 16-row tile and of MOBODY_TC_TRAIN_MIN_ROWS (1 280: mma.sync below, tcgen05 from there); nsplit default, 1, ragged, and
# more splits than 32-row chunks
GRAD_CASES = [
    (2, 1, 1, 1, None), (17, 6, 15, 15, None), (61, 3, 17, 9, None), (64, 1, 255, 100, None), (111, 8, 77, 64, None),
    (128, 32, 255, 200, None), (32, 32, 1279, 1000, None), (27, 8, 255, 200, 1), (27, 8, 255, 200, 64),
    (2, 1, 1280, 1, None), (61, 3, 1281, 1281, None), (64, 1, 1280, 1280, None), (111, 8, 1281, 777, None),
    (128, 32, 1280, 1000, None), (32, 32, 1281, 640, None), (27, 8, 5120, 4096, None), (17, 6, 10240, 8192, None),
    (27, 8, 1281, 1000, 1), (27, 8, 1281, 1000, 7), (17, 6, 1300, 1000, 64),
]


@pytest.mark.parametrize("S,A,N,n_true,nsplit", GRAD_CASES)
def test_train_step_gradients(S, A, N, n_true, nsplit):
    worst, dropped = _run_train(S, A, N, n_true, nsplit, 2, 0.0, 5)
    _report("train-grad", (S, A, N, n_true, nsplit), worst, round(dropped, 4))


@pytest.mark.parametrize("S,A,N,n_true", [(2, 1, 15, 15), (17, 6, 255, 200), (27, 8, 5120, 4096), (128, 32, 1281, 1000)])
def test_train_step_adam_and_polyak(S, A, N, n_true):
    worst, dropped = _run_train(S, A, N, n_true, None, 3, 3e-4, 8)
    _report("train-adam", (S, A, N, n_true), worst, round(dropped, 4))


# ----------------------------------------------------------------------------------------------------- classifier step
@pytest.mark.parametrize("S,A,N", [(2, 1, 5), (61, 3, 100), (128, 32, 37), (17, 6, 2367), (17, 6, 2368), (128, 32, 2367),
                                   (128, 32, 2368), (2, 1, 2368)])
def test_classifier_step_gradients(S, A, N):
    """N = 2 367 / 2 368 sit on either side of the switch from 16-row to 32-row tiles; (128, 32) has 2S+A = 288 inputs."""
    from mobody_b200 import _ffi
    seed, std, lr = 11, 0.5, 3e-4
    ag, _ = cuda_agent(S, A, seed, penalty_type="dara", penalty_coef=1.0, gaussian_noise_std=std, actor_lr=lr, penalize_fake=0)
    ag.classifier.load_state_dict(M.ClassifierState(S, A, seed).params)
    rng = np.random.default_rng(N * 31 + S)
    RW = _ffi.lib().mobody_row_width(S, A)
    opt, worst, dropped = ag._opts["cls"], _Worst(), []
    for it in range(2):
        p0 = _snap(ag.classifier)
        m0, v0 = _moments(opt, ag.classifier)
        t0 = ag._t_cls
        n = N + N // 4 + 64
        f = lambda *sh: rng.standard_normal(sh).astype(np.float32)          # noqa: E731
        s, s2, n_sas, n_sa, a = f(n, S), f(n, S), f(n, 2 * S + A), f(n, S + A), rng.uniform(-1, 1, (n, A)).astype(np.float32)
        label = (rng.random(n) < 0.5).astype(np.int64)
        s2[label == 1] += np.float32(0.25)                                   # the two domains differ in s'
        s, s2, n_sas, n_sa, a = (torch.from_numpy(x).double() for x in (s, s2, n_sas, n_sa, a))
        label = torch.from_numpy(label)
        ok = R.classifier_rows_ok(R.f64(p0), s, a, s2, n_sas, n_sa, std)
        idx = R.first_rows(ok, N)
        dropped.append(1.0 - float(ok[:idx[-1] + 1].double().mean()))
        s, a, s2, n_sas, n_sa, label = (x[idx] for x in (s, a, s2, n_sas, n_sa, label))
        g_ref, losses = R.classifier_reference(R.classifier_state64(p0, m0, v0, t0), s, a, s2, label, n_sas, n_sa, std, lr)
        rows = torch.zeros(N, RW, dtype=torch.float32)
        rows[:, :S], rows[:, S:S + A], rows[:, S + A:2 * S + A] = s.float(), a.float(), s2.float()
        got = ag.classifier_step_on_rows(rows.cuda(), label.to(torch.int32).cuda(), noise_sas=n_sas.float(), noise_sa=n_sa.float())
        got = got.cpu().numpy()
        assert np.all(np.abs(got - np.array(losses)) <= 1e-4 * np.abs(np.array(losses))), (it, got, losses)
        p1 = _snap(ag.classifier)
        m1, v1 = _moments(opt, ag.classifier)
        tag = (S, A, N, it)
        _check_moments(worst, "classifier", m0, m1, v0, v1, g_ref, tag)
        _check_adam(worst, "adam", p0, p1, m1, v1, t0 + 1, lr, tag)
    _report("classifier", (S, A, N), worst, round(max(dropped), 4))


# ----------------------------------------------------------------------------------------------------- dynamics fit
@pytest.mark.parametrize("S,A,B,nsplit,use_trg", [
    (2, 1, 1, 1, True), (2, 1, 256, 8, False), (17, 6, 37, 2, True), (17, 6, 300, 16, False), (64, 16, 256, 3, True),
    (64, 16, 37, 8, False), (96, 64, 300, 8, True), (96, 64, 1, 1, False), (112, 32, 256, 16, True), (112, 32, 300, 2, False),
])
def test_fit_step_gradients(S, A, B, nsplit, use_trg):
    """(96, 64): the 2S+A = 256 and A = 64 limits.  Two consecutive steps of one domain from a fresh optimiser state (the
    source domain's reward terms are scaled by 0.01: after target-domain steps its gradients would sit ~100x below the
    moments they are recovered from)."""
    dyn, _ = cuda_dynamics(S, A, 7, "halfcheetah", 1.0)
    dyn.FIT_NSPLIT = nsplit
    rng = np.random.default_rng(S * 100 + B)
    worst = _Worst()
    for it in range(2):
        f = lambda *sh: rng.standard_normal(sh).astype(np.float32)          # noqa: E731
        s = f(7, B, S); a = rng.uniform(-1, 1, (7, B, A)).astype(np.float32)
        ns = (s + 0.1 * f(7, B, S)).astype(np.float32); r = f(7, B, 1); el = f(6, 7, B, 16); en = f(7, B, S)
        st = dyn._fit_state()
        names = [n + sfx for n in M.dynamics_layer_shapes(S, A) for sfx in (".weight", ".bias")]
        lay = lambda k: k.rsplit(".", 1)                                    # noqa: E731
        get = lambda k, src: (src[lay(k)[0]][0 if lay(k)[1] == "weight" else 1]).detach().cpu().clone()   # noqa: E731
        p0 = {k: getattr(getattr(dyn.model, lay(k)[0]), lay(k)[1]).detach().cpu().clone() for k in names}
        m0, v0 = {k: get(k, st["m"]) for k in names}, {k: get(k, st["v"]) for k in names}
        t0 = dict(st["t"])
        other0 = {k: v.detach().cpu().clone() for k, v in dyn.model.state_dict().items()}
        trained = [n + sfx for n in M.fit_trained_layers(use_trg) for sfx in (".weight", ".bias")]
        t_after = {n: t0[n] + 1 for n in M.fit_trained_layers(use_trg)}
        p64, m64, v64 = R.f64(p0), R.f64({k: m0[k] for k in trained}), R.f64({k: v0[k] for k in trained})
        lr = dyn._fit_lr()
        want, g_ref = R.fit_reference(p64, m64, v64, t_after, *(torch.from_numpy(x) for x in (s, a, ns, r, el, en)), use_trg, lr)
        got = dyn.fit_batch(use_trg, *(torch.from_numpy(x).cuda() for x in (s, a, ns, r)), eps_latent=el, eps_next=en).cpu().numpy()
        tag = (S, A, B, nsplit, it, use_trg)
        for k in range(6):
            assert abs(got[k] - want[k]) <= 1e-4 * abs(want[k]), (tag, k, got[k], want[k])
        st = dyn._fit_state()
        p1 = {k: getattr(getattr(dyn.model, lay(k)[0]), lay(k)[1]).detach().cpu().clone() for k in names}
        m1, v1 = {k: get(k, st["m"]) for k in names}, {k: get(k, st["v"]) for k in names}
        for n in M.dynamics_layer_shapes(S, A):
            assert st["t"][n] == t_after.get(n, t0[n]), (tag, n)
        _check_moments(worst, "fit", m0, m1, v0, v1, g_ref, tag)
        for k in trained:
            rr = R.adam_ratio(p0[k], p1[k], m1[k], v1[k], t_after[lay(k)[0]], lr)
            assert rr <= 1.0, (tag, k, rr)
            worst.add("adam", {k: rr})
        for k in names:
            if k not in trained:                                            # the other domain's action encoder: untouched
                assert torch.equal(p0[k], p1[k]) and torch.equal(m0[k], m1[k]) and torch.equal(v0[k], v1[k]), (tag, k)
        for k, v in dyn.model.state_dict().items():
            if k not in trained:                                            # and every tensor without Adam state
                assert torch.equal(v.detach().cpu(), other0[k]), (tag, k)
    _report("fit", (S, A, B, nsplit), worst)


# ----------------------------------------------------------------------------------------------------- step forward edges
_NEAR = lambda x: min(abs(x[0] - 0.8), abs(x[0] - 2.0), abs(abs(x[1]) - 1.0)) < 1e-3   # noqa: E731  walker2d thresholds
STEP_TOL = {"fp32": 1e-4, "bf16x2": 1e-4, "fp16": 5e-3}


@pytest.mark.parametrize("prec,S,A", [("bf16x2", 2, 1), ("bf16x2", 2, 16), ("bf16x2", 47, 2), ("bf16x2", 40, 16),
                                      ("fp16", 2, 1), ("fp16", 2, 16), ("fp16", 55, 2), ("fp16", 48, 16),
                                      ("fp32", 2, 1), ("fp32", 128, 32), ("fp32", 64, 16)])
def test_step_forward_edges(prec, S, A):
    """The step kernels at the ends of the shapes they accept (tensor-core modes: S <= 64, A <= 16, 2S+A <= 96 for bf16x2,
    112 for fp16) against M.step in float64, injected noise and member picks; walker2d termination (its thresholds read
    columns 0 and 1)."""
    dyn, p = cuda_dynamics(S, A, 13, "walker2d", 5.0, precision=prec, h0=0.95, t3_gain=4.0)
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    for B in (1, 127, 128, 129, 1000):
        rng = np.random.default_rng(B * 7 + S)
        obs = (np.r_[1.25, np.zeros(S - 1)][None] + 0.2 * rng.standard_normal((B, S))).astype(np.float32)
        act = rng.uniform(-1, 1, (B, A)).astype(np.float32)
        eps = rng.standard_normal((7, B, S)).astype(np.float32)
        idx = rng.integers(0, 7, B)
        ref = M.step(p64, torch.from_numpy(obs).double(), torch.from_numpy(act).double(), torch.from_numpy(eps).double(), idx, 3, 5.0)
        nobs, rew, term, info = dyn.step(torch.from_numpy(obs).cuda(), torch.from_numpy(act).cuda(), eps=eps, idx=idx)
        tol = STEP_TOL[prec]
        for got, key in ((info["samples"], "mean"), (nobs, "next_obs"), (info["raw_reward"], "raw_reward"),
                         (info["penalty"], "penalty"), (rew, "reward")):
            want = ref[key].numpy()
            assert rel_err(got.cpu().numpy(), want) < tol, (prec, S, A, B, key, rel_err(got.cpu().numpy(), want))
            if prec != "fp16":
                assert rel_err_strict(got.cpu().numpy(), want) < 1e-4, (prec, S, A, B, key, rel_err_strict(got.cpu().numpy(), want))
        bad = np.flatnonzero(term[:, 0] != ref["terminal"][:, 0])
        assert all(_NEAR(ref["next_obs"][i].numpy()) for i in bad), (prec, S, A, B, bad)


@pytest.mark.parametrize("prec,S,A", [("bf16x2", 64, 16), ("bf16x2", 64, 1), ("bf16x2", 48, 1), ("bf16x2", 41, 16),
                                      ("fp16", 64, 16), ("fp16", 56, 1), ("fp16", 49, 16)])
def test_tensor_core_step_rejects_shapes_it_cannot_hold(prec, S, A):
    """Past 2S+A = 96 (bf16x2) / 112 (fp16) the reward model's [s, a, s'] plane does not fit in shared memory: the ABI
    rejects the shape as an argument error, and the automatic precision choice takes the fp32 kernel there."""
    from mobody_b200.dynamics import tc_step_supports
    assert not tc_step_supports(S, A, prec)
    dyn, _ = cuda_dynamics(S, A, 13, "walker2d", 1.0, precision=prec)
    x, a = torch.zeros(4, S, device="cuda"), torch.zeros(4, A, device="cuda")
    with pytest.raises(RuntimeError, match=r"mobody_b200 \[-1\]: mobody_step: tensor-core modes take"):
        dyn.step(x, a, eps=np.zeros((7, 4, S), np.float32), idx=np.zeros(4, np.int64))
    auto, _ = cuda_dynamics(S, A, 13, "walker2d", 1.0, precision=None)
    assert auto.precision == "fp32"
    auto.step(x, a, eps=np.zeros((7, 4, S), np.float32), idx=np.zeros(4, np.int64))
    assert tc_step_supports(40, 16, "bf16x2") and tc_step_supports(48, 16, "fp16") and not tc_step_supports(48, 16, "bf16x2")
    assert cuda_dynamics(40, 16, 13, "walker2d", 1.0, precision=None)[0].precision == "bf16x2"


def test_rollout_bf16x2_at_the_widest_tensor_core_shape():
    """A T = 3 bf16x2 rollout at (40, 16) -- 2S+A = 96, the widest reward-model input bf16x2 takes -- against M.rollout
    in float64 (injected noise and member picks)."""
    S, A, B, T = 40, 16, 300, 3
    dyn, p = cuda_dynamics(S, A, 17, "walker2d", 1.0, precision="bf16x2", h0=1.25)
    ag, st = cuda_agent(S, A, 17, env_filter=10.0)
    ag.dynamics = dyn
    rng = np.random.default_rng(64)
    obs = (np.r_[1.25, np.zeros(S - 1)][None] + 0.05 * rng.standard_normal((B, S))).astype(np.float32)
    eps = rng.standard_normal((T, 7, B, S)).astype(np.float32)
    idx = rng.integers(0, 7, (T, B))
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    want, winfo = M.rollout(p64, R.f64(st.policy), 1.0, torch.from_numpy(obs).double(), T,
                            [lambda n, t=t: torch.from_numpy(eps[t, :, :n]).double() for t in range(T)],
                            [lambda n, t=t: idx[t, :n] for t in range(T)], 3, 1.0)
    got, info = ag.rollout_device(torch.from_numpy(obs).cuda(), T, True, eps=eps, idx=idx)
    assert info["num_transitions"] == winfo["num_transitions"] and want["obss"].shape[0] > B
    for k in ("obss", "next_obss", "actions", "rewards", "penalty"):
        g, w = got[k].cpu().numpy(), want[k].numpy()
        assert g.shape == w.shape, k
        assert rel_err(g, w) < 1e-4 and rel_err_strict(g, w) < 1e-4, (k, rel_err(g, w), rel_err_strict(g, w))
    assert np.array_equal(got["terminals"].cpu().numpy(), want["terminals"].numpy())
