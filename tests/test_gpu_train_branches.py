"""The fused train step's update branches (mobody_train_step_ex): advantage=1 (value step, V(s') TD target, V(s_t)
advantage weights), scale_Q=0 (p_w = 1) and q_weighted=0 (plain BC), on both tilings (mma.sync below 1 280 rows, tcgen05
from there) and ragged tiles.

Gradients are recovered from the Adam moments and held, element by element, to an fp64 autograd restatement of the
branch math on the state read back before the step (test_grad_reference's method: batches conditioned away from ReLU and
min kinks, critic_lr = 0 so the actor's and the TD target's networks are the pre-step ones).  Multi-step runs are held to
_train_torch_path, the torch autograd reference of every branch.
"""
import ctypes as C
import os
import subprocess
import sys
from collections import OrderedDict

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import test_grad_reference as R
from helpers import cuda_agent
from oracle import mobody_oracle as M
from test_gpu_grad_parity import _check_adam, _check_moments, _moments, _snap, _train_pool, _Worst, _report
from test_gpu_train import adam_close

pytestmark = pytest.mark.gpu
CFG = dict(gamma=0.99, tau=0.005, actor_lr=3e-4, critic_lr=3e-4, weight=2.5, bc_coef=1.0, max_action=1.0)
FLAGS = {"adv": dict(advantage=1), "noscale": dict(scale_Q=0), "plainbc": dict(q_weighted=0),
         "adv_plainbc": dict(advantage=1, q_weighted=0), "all": dict(advantage=1, scale_Q=0, q_weighted=0)}
SHAPES = [(17, 6, 320, 256), (11, 3, 77, 64), (111, 8, 96, 64), (27, 8, 1500, 1200), (27, 8, 10240, 8192)]


def _agent(S, A, seed, flags, **kw):
    ag, _ = cuda_agent(S, A, seed, **flags, **kw)
    ag.v_func.load_state_dict(OrderedDict(("network." + k, v) for k, v in M.make_mlp_params(S, 1, seed + 7).items()))
    return ag


def _rows(batch, RW):
    rows = torch.zeros(batch[0].shape[0], RW, dtype=torch.float32)
    c0 = 0
    for x in batch:
        rows[:, c0:c0 + x.shape[1]] = x.float()
        c0 += x.shape[1]
    return rows


def _random_rows(S, A, N, seed):
    from mobody_b200 import _ffi
    return _rows(_train_pool(S, A, N, np.random.default_rng(seed)), _ffi.lib().mobody_row_width(S, A)).cuda()


# ------------------------------------------------------------------------------------------- fp64 restatement
def branch_reference(pol, q, qt, vf, batch, n_true, cfg, flags):
    """Gradients and loss scalars of one update at the given (pre-step, float64) state, critic_lr = 0: the value function
    and critics the later phases read are the pre-step ones.  -> ({"v", "q", "pi": grads}, losses)"""
    s, a, s2, r, nd = batch
    ma, adv_on = cfg["max_action"], bool(flags.get("advantage", 0))
    grads, losses = {}, {}

    def grad(loss, p):
        return {k: g.numpy() for k, g in zip(p.keys(), torch.autograd.grad(loss, list(p.values())))}

    if adv_on:                                                                     # mobody.py:210-242
        vp = OrderedDict((k, v.clone().requires_grad_(True)) for k, v in vf.items())
        qtv = torch.min(*M.double_q_forward(qt, s, a))
        v = M.mlp_forward(vp, s, "network.")
        adv = qtv - v
        v_loss = torch.mean(torch.abs(0.7 - (adv < 0).double()) * adv ** 2)
        grads["v"] = grad(v_loss, vp)
        losses.update(v_loss=float(v_loss.detach()), adv_mean=float(adv.detach().mean()), v_mean=float(v.detach().mean()))
    with torch.no_grad():
        boot = M.mlp_forward(vf, s2, "network.") if adv_on else torch.min(*M.double_q_forward(qt, s2, M.policy_forward(pol, s2, ma)))
        y = r + nd * cfg["gamma"] * boot
    qp = OrderedDict((k, v.clone().requires_grad_(True)) for k, v in q.items())
    q1, q2 = M.double_q_forward(qp, s, a)
    q_loss = F.mse_loss(q1, y) + F.mse_loss(q2, y)
    grads["q"] = grad(q_loss, qp)
    pp = OrderedDict((k, v.clone().requires_grad_(True)) for k, v in pol.items())
    qv = torch.min(*M.double_q_forward(q, s, M.policy_forward(pp, s, ma)))
    p_w = cfg["weight"] / qv.abs().mean().detach() if flags.get("scale_Q", 1) else 1.0
    st, at = s[:n_true], a[:n_true]
    pred = M.policy_forward(pp, st, ma)
    with torch.no_grad():
        qb = torch.min(*M.double_q_forward(q, st, at))
        adv_t = qb - M.mlp_forward(vf, st, "network.") if adv_on else qb / qb.abs().mean()
        w = torch.exp(3 * adv_t).clamp(max=100.0) if flags.get("q_weighted", 1) else torch.ones_like(qb)
        q_beh = torch.min(*M.double_q_forward(q, s, a)).mean()
    bc = torch.mean(w * (pred - at) ** 2)
    loss = p_w * (-qv).mean() + cfg["bc_coef"] * bc
    grads["pi"] = grad(loss, pp)
    losses.update(q_loss=float(q_loss), q1_mean=float(q1.mean()), pi_loss=float(loss), bc_loss=float(bc),
                  q_policy=float(qv.mean()), w_mean=float(w.mean()), p_w=float(p_w), q_behavior=float(q_beh))
    return grads, losses, (y, q1, q2, adv if adv_on else None)


def _cancellation(d):
    """|sum d| / sum |d|: an output bias's gradient element is sum d, ill-conditioned when it cancels."""
    return float(d.sum().abs() / d.abs().sum())


@pytest.mark.parametrize("flags", list(FLAGS), ids=list(FLAGS))
@pytest.mark.parametrize("S,A,N,n_true", SHAPES)
def test_branch_gradients(S, A, N, n_true, flags):
    fl = FLAGS[flags]
    adv_on = bool(fl.get("advantage", 0))
    cfg = dict(CFG, critic_lr=0.0)
    ag = _agent(S, A, 5, fl, critic_lr=0.0)
    ag.target_q_funcs.load_state_dict(M.AgentState(S, A, 55).q)                    # targets != critics
    rng = np.random.default_rng(N * 13 + S)
    from mobody_b200 import _ffi
    RW = _ffi.lib().mobody_row_width(S, A)
    worst, dropped = _Worst(), []
    v0_all = _snap(ag.v_func)
    for it in range(2):
        pol, q, qt, vf = _snap(ag.policy), _snap(ag.q_funcs), _snap(ag.target_q_funcs), _snap(ag.v_func)
        (mq, vq), (mpi, vpi), (mv, vv) = _moments(ag._opts["q"], ag.q_funcs), _moments(ag._opts["pi"], ag.policy), _moments(ag._opts["v"], ag.v_func)
        t_pi, t_v = ag._t_pi, ag._t_v
        P = {k: R.f64(x) for k, x in (("pi", pol), ("q", q), ("qt", qt), ("v", vf))}
        for _ in range(16):
            pool = _train_pool(S, A, N + N // 4 + 64, rng)
            ok = R.train_rows_ok(P["pi"], P["q"], pool[0], pool[1], cfg["max_action"])
            if adv_on:
                ok &= R.mlp_margin(P["v"], pool[0], "network.", R.DELTA)[0]
            idx = R.first_rows(ok, N)
            batch = tuple(x[idx] for x in pool)
            _, _, (y, q1r, q2r, adv) = branch_reference(P["pi"], P["q"], P["qt"], P["v"], batch, n_true, cfg, fl)
            cancel = [_cancellation(qk - y) for qk in (q1r, q2r)]
            if adv_on:
                cancel.append(_cancellation(torch.abs(0.7 - (adv < 0).double()) * adv))
            if min(cancel) >= R.TD_MIN_CANCELLATION:
                break
        dropped.append(1.0 - float(ok[:idx[-1] + 1].double().mean()))
        g_ref, want, _ = branch_reference(P["pi"], P["q"], P["qt"], P["v"], batch, n_true, cfg, fl)
        ag.train_on_rows(_rows(batch, RW).cuda(), n_true)
        got = ag.loss_scalars()
        tag = (S, A, N, n_true, flags, it)
        assert ("v_loss" in got) == adv_on, tag
        got["q_behavior"] = float(ag._scalars[14])
        for k in ("q_loss", "pi_loss", "bc_loss", "q1_mean", "q_policy", "w_mean", "p_w", "q_behavior") + (("v_loss", "adv_mean", "v_mean") if adv_on else ()):
            assert abs(got[k] - want[k]) <= 1e-4 * (abs(want[k]) + 1e-2), (tag, k, got[k], want[k])
        (mq1, vq1), (mpi1, vpi1), (mv1, vv1) = _moments(ag._opts["q"], ag.q_funcs), _moments(ag._opts["pi"], ag.policy), _moments(ag._opts["v"], ag.v_func)
        _check_moments(worst, "critic", mq, mq1, vq, vq1, g_ref["q"], tag)
        _check_moments(worst, "actor", mpi, mpi1, vpi, vpi1, g_ref["pi"], tag)
        _check_adam(worst, "adam", pol, _snap(ag.policy), mpi1, vpi1, t_pi + 1, cfg["actor_lr"], tag)
        if adv_on:
            assert ag._t_v == t_v + 1, tag
            _check_moments(worst, "value", mv, mv1, vv, vv1, g_ref["v"], tag)
        else:
            assert ag._t_v == 0, tag
            for k in mv:
                assert torch.equal(mv[k], mv1[k]) and torch.equal(vv[k], vv1[k]), (tag, k)
        for k, x in _snap(ag.v_func).items():
            assert torch.equal(x, v0_all[k]), (tag, k)                             # critic_lr = 0, or no value step at all
    _report("branch-grad", (S, A, N, n_true, flags), worst, round(max(dropped), 4))


# ------------------------------------------------------------------------------------------- against the torch path
_NETS = ("policy", "q_funcs", "target_q_funcs", "v_func")


def _adopt(dst, src):
    """dst takes src's parameters, target critics, value function and Adam moments (same step counts)."""
    with torch.no_grad():
        for name in _NETS:
            for x, y in zip(getattr(dst, name).parameters(), getattr(src, name).parameters()):
                x.copy_(y)
        for opt in ("q", "v", "pi"):
            sd, ss = dst._opts[opt], src._opts[opt]
            for pd, ps in zip((p for g in sd.param_groups for p in g["params"]), (p for g in ss.param_groups for p in g["params"])):
                sd.state[pd]["exp_avg"].copy_(ss.state[ps]["exp_avg"])
                sd.state[pd]["exp_avg_sq"].copy_(ss.state[ps]["exp_avg_sq"])


@pytest.mark.parametrize("flags", list(FLAGS), ids=list(FLAGS))
@pytest.mark.parametrize("S,A,N,n_true", SHAPES)
def test_three_steps_match_the_torch_path(S, A, N, n_true, flags):
    """Three consecutive updates (Adam step counts 1..3, moments carried), each compared with _train_torch_path taken
    from the same state: the torch agent adopts the fused agent's tensors before every step, so the comparison holds
    each update to the reference instead of measuring how two runs drift apart (Adam's first steps are lr * sign(g))."""
    fl = FLAGS[flags]
    rows = _random_rows(S, A, N, 3 * N + S)
    a1, a2 = _agent(S, A, 9, fl), _agent(S, A, 9, fl)
    v0 = _snap(a1.v_func)
    for step in range(3):
        _adopt(a2, a1)
        a1.train_on_rows(rows, n_true)
        a2._train_torch_path(rows, n_true, None, None)
        torch.cuda.synchronize()
        for name in _NETS:
            for (k, x1), x2 in zip(getattr(a1, name).state_dict().items(), getattr(a2, name).state_dict().values()):
                adam_close(x1.cpu().numpy(), x2.cpu().numpy(), 3e-4, 1, (flags, step, name, k))
        got = a1.loss_scalars()
        for k, idx in (("q_loss", 0), ("pi_loss", 2)):
            want = float(a2._scalars[idx])
            assert abs(got[k] - want) <= 1e-4 * (abs(want) + 1e-2), (flags, step, k, got[k], want)
    n_v = 3 * int(bool(fl.get("advantage")))
    assert a1._t_q == a2._t_q == 3 and a1._t_pi == a2._t_pi == 3 and a1._t_v == a2._t_v == n_v
    if not n_v:
        for k, x in _snap(a1.v_func).items():
            assert torch.equal(x, v0[k]), k


@pytest.mark.parametrize("S,A,N,n_true", [(17, 6, 320, 256), (27, 8, 1500, 1200)])
def test_default_flags_through_ex_are_bit_identical(S, A, N, n_true, monkeypatch):
    from mobody_b200 import _ffi
    L = _ffi.lib()
    rows = _random_rows(S, A, N, 17)

    def run():
        ag = _agent(S, A, 4, {})
        for _ in range(3):
            ag.train_on_rows(rows, n_true)
        torch.cuda.synchronize()
        return [x.cpu() for m in (ag.policy, ag.q_funcs, ag.target_q_funcs) for x in m.state_dict().values()] + [ag._scalars[:11].cpu()]

    base = run()
    calls = []

    def via_ex(dref, stream):
        x = _ffi.TrainExDesc()
        x.base, x.advantage, x.scale_q, x.q_weighted = dref._obj, 0, 1, 1
        calls.append(1)
        return L.mobody_train_step_ex(C.byref(x), stream)

    monkeypatch.setattr(L, "mobody_train_step", via_ex)
    ex = run()
    assert len(calls) == 3
    for x, y in zip(base, ex):
        assert torch.equal(x, y)


@pytest.mark.parametrize("flags", ["adv", "all"])
@pytest.mark.parametrize("S,A,N,n_true", [(17, 6, 320, 256), (27, 8, 1500, 1200)])
def test_row_splits_reproducible_and_agree(S, A, N, n_true, flags):
    rows = _random_rows(S, A, N, 5 * N)

    def run(nsplit):
        ag = _agent(S, A, 6, FLAGS[flags])
        for _ in range(2):
            ag.train_on_rows(rows, n_true, nsplit=nsplit)
        torch.cuda.synchronize()
        return {f"{g}.{k}": v.cpu().numpy().copy() for g, m in (("pi", ag.policy), ("q", ag.q_funcs), ("qt", ag.target_q_funcs), ("v", ag.v_func))
                for k, v in m.state_dict().items()}, ag._scalars.cpu().numpy()

    for nsplit in (1, 3, 64):
        a, sa = run(nsplit)
        b, sb = run(nsplit)
        assert all(np.array_equal(a[k], b[k]) for k in a) and np.array_equal(sa[:15], sb[:15]), nsplit
        if nsplit == 1:
            base = a
        else:
            for k in base:
                adam_close(a[k], base[k], 3e-4, 2, (nsplit, k))


_DIGEST = r"""
import hashlib, sys, os
sys.path.insert(0, os.path.join(os.getcwd(), "tests"))
import numpy as np, torch
from test_gpu_train_branches import FLAGS, _agent, _random_rows
h = hashlib.sha256()
for flags in ("adv", "all"):
    for S, A, N, n_true, steps in ((17, 6, 320, 256, 10), (27, 8, 5120, 4096, 3)):
        rows = _random_rows(S, A, N, N)
        ag = _agent(S, A, 9, FLAGS[flags])
        for _ in range(steps):
            ag.train_on_rows(rows, n_true)
        torch.cuda.synchronize()
        for m in (ag.policy, ag.q_funcs, ag.target_q_funcs, ag.v_func):
            for v in m.state_dict().values():
                h.update(v.detach().cpu().numpy().tobytes())
        h.update(ag._scalars[:15].cpu().numpy().tobytes())
print("DIGEST", h.hexdigest())
"""


def test_launch_modes_give_identical_bits_in_subprocess():
    """PDL on / off and the large-batch side stream on / off do not change a bit of the branch updates."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def digest(**env):
        r = subprocess.run([sys.executable, "-c", _DIGEST], env=dict(os.environ, **env), capture_output=True, text=True,
                           timeout=300, cwd=root)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return [ln.split()[1] for ln in r.stdout.splitlines() if ln.startswith("DIGEST")][0]

    base = digest(MOBODY_PDL="1", MOBODY_TRAIN_SIDE="1")
    assert base == digest(MOBODY_PDL="0")
    assert base == digest(MOBODY_TRAIN_SIDE="0")


# ------------------------------------------------------------------------------------------- train()
class _Writer:
    def __init__(self):
        self.calls = []

    def add_scalar(self, name, value, global_step=None):
        self.calls.append((name, float(value), int(global_step)))


class _Wandb:
    def __init__(self):
        self.calls = []

    def log(self, d, step=None, commit=True):
        self.calls.append((sorted(d), int(step), commit))


def _buffers(ag, S, A):
    import mobody_b200 as mb
    rng = np.random.default_rng(3)

    def ds(n):
        return dict(observations=rng.standard_normal((n, S)).astype(np.float32), actions=rng.uniform(-1, 1, (n, A)).astype(np.float32),
                    next_observations=rng.standard_normal((n, S)).astype(np.float32), rewards=rng.standard_normal(n).astype(np.float32),
                    terminals=(rng.random(n) < 0.1))
    src, tar = mb.ReplayBuffer(S, A, "cuda"), mb.ReplayBuffer(S, A, "cuda")
    src.convert_D4RL(ds(3000)); tar.convert_D4RL(ds(500)); ag.fake_replay_buffer.convert_D4RL(ds(800))
    return src, tar


@pytest.mark.parametrize("flags", list(FLAGS), ids=list(FLAGS))
def test_train_runs_every_branch_fused_and_logs_the_torch_path_keys(flags, monkeypatch):
    S, A, B = 11, 3, 64
    fl = FLAGS[flags]
    ag = _agent(S, A, 21, fl)
    src, tar = _buffers(ag, S, A)
    ref = _agent(S, A, 21, fl)
    ref.fake_replay_buffer = ag.fake_replay_buffer

    def refuse(*a, **k):
        raise AssertionError("train() entered _train_torch_path")

    monkeypatch.setattr(ag, "_train_torch_path", refuse)
    ag.total_it = ref.total_it = 4997                                    # the third step logs (total_it % 5000 == 0)
    w, wb = _Writer(), _Wandb()
    for _ in range(2):
        ag.train(src, tar, B, w, wb)
    assert w.calls == [] and wb.calls == []
    ag.train(src, tar, B, w, wb)
    torch.cuda.synchronize()
    n_v = 3 * int(bool(fl.get("advantage")))
    assert ag._t_q == ag._t_pi == 3 and ag._t_v == n_v
    assert float(ag.v_optimizer.state_dict()["state"][0]["step"]) == n_v
    # the torch path's keys, order and wandb calls on the same batch rows
    rows = src.sample_rows(B, np.arange(B))
    ref.total_it = 5000
    w_ref, wb_ref = _Writer(), _Wandb()
    ref._train_torch_path(torch.cat([rows, rows]), B, w_ref, wb_ref)
    assert [c[0] for c in w.calls] == [c[0] for c in w_ref.calls]
    assert all(c[2] == 5000 and np.isfinite(c[1]) for c in w.calls)
    assert [c[0] for c in wb.calls] == [c[0] for c in wb_ref.calls] and [c[2] for c in wb.calls] == [c[2] for c in wb_ref.calls]
    exp_adv = dict((c[0], c[1]) for c in w.calls)["train/exp_adv"]
    assert (exp_adv == 1.0) == (not fl.get("q_weighted", 1))
