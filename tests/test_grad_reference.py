"""float64 reference gradients of the three update kernels (train step, classifier step, dynamics fit), the batch
conditioning that lets them be held to 1e-4 on every element, and CPU checks of that machinery on the oracle itself.

The update kernels are judged by the gradient they hand to Adam, recovered from the moments they write
(g_t = (m_t - 0.9 m_{t-1}) / 0.1), against torch.autograd of the oracle in float64 on the state read back before the
step.  Parameters after Adam cannot show a gradient error: at step 1 the update is lr * sign(g), and a constant factor on a
whole gradient tensor cancels in m / sqrt(v).

ReLU gates and the actor's min(q1, q2) have kinks.  A row whose pre-activation lies within rounding of 0 may take the
other branch in fp32 / 3xTF32 than in float64, which moves a gradient element by ~1/sqrt(N) of its tensor's scale.
Rather than letting a fraction of the elements escape, the batch is drawn from a larger candidate pool, keeping only the
rows whose every differentiated gate clears its kink by DELTA times the magnitude of its own dot product
sum_k |w_k x_k| (bias included).  Passes that are not differentiated (target critics, pi(s'), the BC weights) have no
kink in value and need no margin; the dynamics fit (swish, softplus, Gaussian terms) is smooth and needs none at all.
"""
from collections import OrderedDict

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import mobody_oracle as M

# Kink margin, relative to sum_k |w_k x_k| of the gate's own dot product.  The 3xTF32 tensor-core tiles are held to
# 5e-6 * sum |a||b| (test_gpu_umma.test_tf32x3_gemm_tiles) and typically land far inside it; 2^-18 = 3.8e-6 drops a few
# percent of the candidate rows and, on the B200, leaves every gradient element of every case inside the 1e-4 bound
# (test_gpu_grad_parity prints the share dropped and the worst err / bound per tensor).
DELTA = 2.0 ** -18
GRAD_TOL = 1e-4           # every element: |g - g_ref| <= GRAD_TOL * (|g_ref| + mean |g_ref|)
V_TOL = 2e-4              # exp_avg_sq, recovered by cancellation: against g_ref^2
B1, B2, ADAM_EPS = 0.9, 0.999, 1e-8
ULP4 = 2.0 ** -21         # four fp32 ulps (relative)


def f64(d):
    return OrderedDict((k, v.detach().to("cpu", torch.float64).clone()) for k, v in d.items())


# ---------------------------------------------------------------------------------------------------- kink margins
def mlp_margin(p, x, prefix, delta):
    """Forward of an oracle MLP (in -> 256 -> 256 -> out) -> (ok[N], out, mag): ok says every hidden ReLU pre-activation z
    of the row satisfies |z| > delta * sum_k |w_k x_k|; mag is that magnitude for the output layer."""
    ok, h = torch.ones(x.shape[0], dtype=torch.bool), x
    for li in (0, 2, 4):
        w, b = p[f"{prefix}network.{li}.weight"], p[f"{prefix}network.{li}.bias"]
        z, mag = F.linear(h, w, b), F.linear(h.abs(), w.abs(), b.abs())
        if li == 4:
            return ok, z, mag
        ok &= (z.abs() > delta * mag).all(1)
        h = F.relu(z)


def train_rows_ok(policy, q, s, a, max_action, delta=DELTA):
    """Rows on which every differentiated pass of the train step is clear of its kinks: the critics on (s, a), the policy
    on s, the critics on (s, pi(s)) and the actor's min(q1, q2) there.  float64 inputs."""
    x = torch.cat([s, a], 1)
    ok = mlp_margin(q, x, "network1.", delta)[0] & mlp_margin(q, x, "network2.", delta)[0]
    okp, pre, _ = mlp_margin(policy, s, "network.", delta)
    xa = torch.cat([s, torch.tanh(pre) * max_action], 1)
    ok1, q1, m1 = mlp_margin(q, xa, "network1.", delta)
    ok2, q2, m2 = mlp_margin(q, xa, "network2.", delta)
    return ok & okp & ok1 & ok2 & ((q1 - q2).abs() > delta * (m1 + m2))[:, 0]


def td_cancellation(policy, q, q_target, batch, gamma, max_action):
    """min over the two critics of |sum_i (q_i - y_i)| / sum_i |q_i - y_i|.  The critic's output bias has ONE gradient
    element, that sum: a batch on which it cancels to ~0 leaves the element ill-conditioned (fp32 summation error is
    relative to sum |q - y|), so such batches are drawn again rather than judged."""
    s, a, s2, r, nd = batch
    q1, q2 = M.double_q_forward(q, s, a)
    t1, t2 = M.double_q_forward(q_target, s2, M.policy_forward(policy, s2, max_action))
    y = r + nd * gamma * torch.min(t1, t2)
    return min(float((qk - y).sum().abs() / (qk - y).abs().sum()) for qk in (q1, q2))


TD_MIN_CANCELLATION = 2.0 ** -6


def classifier_rows_ok(params, s, a, s2, noise_sas, noise_sa, std, delta=DELTA):
    """Rows on which both classifiers' ReLU gates are clear of their kinks, on the noise-perturbed inputs."""
    sas = torch.cat([s, a, s2], 1) + noise_sas * std
    sa = torch.cat([s, a], 1) + noise_sa * std
    return mlp_margin(params, sas, "sas_classifier.", delta)[0] & mlp_margin(params, sa, "sa_classifier.", delta)[0]


def first_rows(ok, n):
    """Indices of the first n rows with ok set, in order."""
    idx = np.flatnonzero(np.asarray(ok))[:n]
    assert len(idx) == n, f"candidate pool too small: {int(np.asarray(ok).sum())} usable rows for {n}"
    return idx


# ---------------------------------------------------------------------------------------------------- references
def grad_from_moments(m_prev, m_new):
    """The gradient Adam consumed, recovered in float64 from its first moment before and after the step."""
    return (np.asarray(m_new, np.float64) - B1 * np.asarray(m_prev, np.float64)) / (1.0 - B1)


def sq_grad_from_moments(v_prev, v_new):
    return (np.asarray(v_new, np.float64) - B2 * np.asarray(v_prev, np.float64)) / (1.0 - B2)


def agent_state64(policy, q, q_target, m_q, v_q, m_pi, v_pi, t_q, t_pi):
    """An oracle AgentState holding the given tensors in float64 (t_q / t_pi: steps taken so far)."""
    st = M.AgentState.__new__(M.AgentState)
    st.policy, st.q, st.q_target = f64(policy), f64(q), f64(q_target)
    st.m_q, st.v_q, st.m_pi, st.v_pi = f64(m_q), f64(v_q), f64(m_pi), f64(v_pi)
    st.t_q, st.t_pi = int(t_q), int(t_pi)
    st.S, st.A = st.policy["network.network.0.weight"].shape[1], st.policy["network.network.4.bias"].shape[0]
    return st


def train_reference(st, batch, n_true, cfg):
    """M.train_step in float64 on ``st`` (mutated) -> (critic grads, actor grads, losses).  The actor's gradient is taken
    on the critics AFTER their Adam step, like the kernel; it equals the pre-step critics' when critic_lr = 0."""
    m_q0, m_pi0 = f64(st.m_q), f64(st.m_pi)
    losses = M.train_step(st, tuple(x.double() for x in batch), n_true, cfg)
    gq = {k: grad_from_moments(m_q0[k], st.m_q[k]) for k in st.q}
    gpi = {k: grad_from_moments(m_pi0[k], st.m_pi[k]) for k in st.policy}
    return gq, gpi, losses


def classifier_state64(params, m, v, t):
    cl = M.ClassifierState.__new__(M.ClassifierState)
    cl.params, cl.m, cl.v, cl.t = f64(params), f64(m), f64(v), int(t)
    return cl


def classifier_reference(cl, s, a, s2, label, noise_sas, noise_sa, std, lr):
    """M.classifier_update in float64 on ``cl`` (mutated) -> (grads, (loss_sa, loss_sas))."""
    m0 = f64(cl.m)
    losses = M.classifier_update(cl, s.double(), a.double(), s2.double(), label, noise_sas.double(), noise_sa.double(), std, lr)
    return {k: grad_from_moments(m0[k], cl.m[k]) for k in cl.params}, losses


def fit_reference(p, m, v, t_after, s, a, ns, r, eps_latent, eps_next, use_trg, lr):
    """M.fit_step in float64 (p, m, v: dicts of float64 tensors, mutated) -> (losses, grads)."""
    losses, grads = M.fit_step(p, m, v, t_after, *(x.double() for x in (s, a, ns, r, eps_latent, eps_next)), use_trg, lr)
    return losses, {k: g.numpy() for k, g in grads.items()}


# ---------------------------------------------------------------------------------------------------- checks
def strict_ratio(got, want, tol=GRAD_TOL):
    """max over elements of |got - want| / (tol * (|want| + mean |want|)): <= 1 passes."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    bound = tol * (np.abs(want) + np.abs(want).mean())
    return float(np.max(np.abs(got - want) / np.maximum(bound, 1e-300))) if want.size else 0.0


def where_bad(got, want, tol=GRAD_TOL):
    """Where the elements over the bound lie (count, and the distinct rows / columns of a 2-D or [E, in, out] tensor)."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    bad = np.abs(got - want) > tol * (np.abs(want) + np.abs(want).mean())
    out = {"n_bad": int(bad.sum()), "of": int(bad.size)}
    if bad.ndim >= 2 and bad.any():
        nz = np.nonzero(bad)
        out["rows"] = sorted(set(nz[-2].tolist()))[:16]
        out["cols"] = sorted(set(nz[-1].tolist()))[:16]
        if bad.ndim == 3:
            out["members"] = sorted(set(nz[0].tolist()))
    return out


def check_grads(got, want, tag, tol=GRAD_TOL):
    """Every element of every tensor inside the strict bound -> {name: worst err / bound}."""
    ratios = {}
    for k in want:
        ratios[k] = strict_ratio(got[k], want[k], tol)
        assert ratios[k] <= 1.0, (tag, k, ratios[k], where_bad(got[k], want[k], tol))
    return ratios


def adam_ratio(p_prev, p_new, m, v, t, lr):
    """Adam's arithmetic from the kernel's own moments: p_t = p_{t-1} - lr/bc1 * m_t / (sqrt(v_t)/sqrt(bc2) + eps),
    within four fp32 ulps of |p_{t-1}| and of the step -> worst err / bound."""
    p_prev, p_new, m, v = (np.asarray(x, np.float64) for x in (p_prev, p_new, m, v))
    bc1, bc2 = 1.0 - B1 ** t, 1.0 - B2 ** t
    step = lr / bc1 * m / (np.sqrt(v) / np.sqrt(bc2) + ADAM_EPS)
    bound = ULP4 * (np.abs(p_prev) + np.abs(step))
    return float(np.max(np.abs(p_new - (p_prev - step)) / np.maximum(bound, 1e-300)))


def polyak_ratio(qt_prev, qt_new, q_new, tau):
    """qt_t = tau * q_t + (1 - tau) * qt_{t-1} within four fp32 ulps -> worst err / bound."""
    qt_prev, qt_new, q_new = (np.asarray(x, np.float64) for x in (qt_prev, qt_new, q_new))
    bound = ULP4 * (tau * np.abs(q_new) + np.abs(qt_prev))
    return float(np.max(np.abs(qt_new - (tau * q_new + (1.0 - tau) * qt_prev)) / np.maximum(bound, 1e-300)))


# ---------------------------------------------------------------------------------------------------- CPU checks
CFG = dict(gamma=0.99, tau=0.005, actor_lr=3e-4, critic_lr=0.0, weight=2.5, bc_coef=1.0, max_action=1.0)


def _train_batch(S, A, n, seed):
    rng = np.random.default_rng(seed)
    s, s2, r = (torch.from_numpy(rng.standard_normal(sh)) for sh in ((n, S), (n, S), (n, 1)))
    a = torch.from_numpy(rng.uniform(-1, 1, (n, A)))
    nd = torch.from_numpy((rng.random((n, 1)) > 0.1).astype(np.float64))
    return s, a, s2, r, nd


def _oracle_train_step(S, A, N, n_true, seed=3):
    """One fp32 oracle step on a conditioned batch next to the float64 reference -> (fp32 grads, float64 grads, info)."""
    st32 = M.AgentState(S, A, seed)
    st32.q_target = M.AgentState(S, A, seed + 50).q                       # targets != critics: Polyak is not a no-op
    pool = _train_batch(S, A, N + N // 4 + 64, seed)
    ok = train_rows_ok(f64(st32.policy), f64(st32.q), pool[0], pool[1], CFG["max_action"])
    idx = first_rows(ok, N)
    batch = tuple(x[idx] for x in pool)
    st64 = agent_state64(st32.policy, st32.q, st32.q_target, st32.m_q, st32.v_q, st32.m_pi, st32.v_pi, 0, 0)
    gq_ref, gpi_ref, _ = train_reference(st64, batch, n_true, CFG)
    before = dict(q=f64(st32.q), qt=f64(st32.q_target), pi=f64(st32.policy))
    M.train_step(st32, tuple(x.float() for x in batch), n_true, CFG)
    gq = {k: grad_from_moments(0 * v, v) for k, v in f64(st32.m_q).items()}
    gpi = {k: grad_from_moments(0 * v, v) for k, v in f64(st32.m_pi).items()}
    return gq, gpi, gq_ref, gpi_ref, dict(st32=st32, before=before, dropped=len(pool[0]) - int(ok.sum()), pool=len(pool[0]))


def test_fp32_oracle_passes_the_strict_check_on_a_conditioned_batch():
    gq, gpi, gq_ref, gpi_ref, info = _oracle_train_step(17, 6, 600, 480)
    assert 0 < info["dropped"] < 0.5 * info["pool"]                       # the margin is active, the pool large enough
    check_grads(gq, gq_ref, "critic")
    check_grads(gpi, gpi_ref, "actor")
    st32, before = info["st32"], info["before"]
    for k in st32.q:                                                       # critic_lr = 0: critics bit-identical
        assert torch.equal(st32.q[k].double(), before["q"][k])
        assert polyak_ratio(before["qt"][k], st32.q_target[k], st32.q[k], CFG["tau"]) <= 1.0, k
        assert strict_ratio(sq_grad_from_moments(0 * st32.v_q[k].double(), st32.v_q[k]), gq_ref[k] ** 2, V_TOL) <= 1.0, k
    for k in st32.policy:
        assert adam_ratio(before["pi"][k], st32.policy[k], st32.m_pi[k], st32.v_pi[k], 1, CFG["actor_lr"]) <= 1.0, k
        assert strict_ratio(sq_grad_from_moments(0 * st32.v_pi[k].double(), st32.v_pi[k]), gpi_ref[k] ** 2, V_TOL) <= 1.0, k


def test_strict_check_catches_planted_defects():
    gq, gpi, gq_ref, gpi_ref, _ = _oracle_train_step(17, 6, 600, 480)
    k_b = "network1.network.0.bias"
    i = int(np.argmax(np.abs(gq_ref[k_b])))
    bad = dict(gq); bad[k_b] = gq[k_b].copy(); bad[k_b][i] *= 1 + 1e-3            # 1e-3 relative on one bias element
    with pytest.raises(AssertionError):
        check_grads(bad, gq_ref, "bias element")
    bad = dict(gpi); bad["network.network.2.weight"] = 2 * gpi["network.network.2.weight"]   # factor 2 on a whole tensor
    with pytest.raises(AssertionError):
        check_grads(bad, gpi_ref, "factor 2")
    k_w = "network2.network.2.weight"
    row = int(np.argmax(np.abs(gq_ref[k_w]).sum(1)))
    bad = dict(gq); bad[k_w] = gq[k_w].copy(); bad[k_w][row] = 0.0                   # one hidden unit's weight row zeroed
    with pytest.raises(AssertionError):
        check_grads(bad, gq_ref, "row zeroed")
    # Adam's own arithmetic: one ulp-scale slip passes, a wrong step does not
    p = np.float32([0.5, -0.25]); m = np.float32([1e-3, -2e-3]); v = np.float32([1e-6, 4e-6])
    want = p.astype(np.float64) - 3e-4 / 0.1 * m / (np.sqrt(v) / np.sqrt(0.001) + 1e-8)
    assert adam_ratio(p, want.astype(np.float32), m, v, 1, 3e-4) <= 1.0
    assert adam_ratio(p, (p - 2 * (p - want)).astype(np.float32), m, v, 1, 3e-4) > 1.0


def test_classifier_and_fit_references_agree_with_the_fp32_oracle():
    """The float64 classifier / dynamics-fit references against the fp32 oracle's own gradients (strict bound)."""
    S, A, N, std, lr = 17, 6, 400, 0.5, 3e-4
    rng = np.random.default_rng(9)
    cl32 = M.ClassifierState(S, A, 4)
    n = N + N // 4 + 64
    s, s2 = (torch.from_numpy(rng.standard_normal((n, S))) for _ in range(2))
    a = torch.from_numpy(rng.uniform(-1, 1, (n, A)))
    n_sas, n_sa = torch.from_numpy(rng.standard_normal((n, 2 * S + A))), torch.from_numpy(rng.standard_normal((n, S + A)))
    label = torch.from_numpy((rng.random(n) < 0.5).astype(np.int64))
    idx = first_rows(classifier_rows_ok(f64(cl32.params), s, a, s2, n_sas, n_sa, std), N)
    s, a, s2, n_sas, n_sa, label = (x[idx] for x in (s, a, s2, n_sas, n_sa, label))
    want, _ = classifier_reference(classifier_state64(cl32.params, cl32.m, cl32.v, 0), s, a, s2, label, n_sas, n_sa, std, lr)
    M.classifier_update(cl32, s.float(), a.float(), s2.float(), label, n_sas.float(), n_sa.float(), std, lr)
    check_grads({k: grad_from_moments(0 * v.double(), v) for k, v in cl32.m.items()}, want, "classifier")

    S, A, B = 17, 6, 40
    p32 = M.make_dynamics_params(S, A, 2)
    del p32["elites"]
    x = [torch.from_numpy(rng.standard_normal(sh).astype(np.float32)) for sh in ((7, B, S), (7, B, A), (7, B, S), (7, B, 1),
                                                                                 (6, 7, B, 16), (7, B, S))]
    names = [nm + sfx for nm in M.fit_trained_layers(False) for sfx in (".weight", ".bias")]
    zeros = lambda p: {k: torch.zeros_like(p[k]) for k in names}              # noqa: E731
    t = {nm: 1 for nm in M.fit_trained_layers(False)}
    p64 = f64(p32)
    _, got = M.fit_step(dict(p32), zeros(p32), zeros(p32), t, *x, False, 1e-3)
    _, want = fit_reference(p64, zeros(p64), zeros(p64), t, *x, False, 1e-3)
    check_grads({k: g.numpy() for k, g in got.items()}, want, "fit")
