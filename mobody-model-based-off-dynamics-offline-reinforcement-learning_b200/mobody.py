"""MOBODY agent: fused model rollout + Q-weighted behaviour-cloning update.

Mirror of algo/offline_offline/mobody.py (``MLPNetwork``, ``Policy``, ``DoubleQFunc``,
``ValueFunc``, ``MOBODY.select_action / rollout / train / save / load``).  The nn.Modules keep
the reference's names so ``_actor`` / ``_critic`` checkpoints (mobody.py:584-594) load unchanged;
they only own parameters — the hot path hands their device pointers to the CUDA kernels.
"""
import copy
import ctypes as C

import numpy as np
import torch
import torch.nn as nn

from . import _ffi
from .buffer import ReplayBuffer
from .dynamics import StepWorkspace


class MLPNetwork(nn.Module):                                   # mobody.py:35-48
    def __init__(self, input_dim, output_dim, hidden_size=256):
        super().__init__()
        self.network = nn.Sequential(nn.Linear(input_dim, hidden_size), nn.ReLU(),
                                     nn.Linear(hidden_size, hidden_size), nn.ReLU(),
                                     nn.Linear(hidden_size, output_dim))

    def forward(self, x):
        return self.network(x)


class ValueFunc(nn.Module):                                    # mobody.py:50-57
    def __init__(self, state_dim, action_dim, hidden_size=256):
        super().__init__()
        self.network = MLPNetwork(state_dim, 1, hidden_size)

    def forward(self, state):
        return self.network(state)


class Policy(nn.Module):                                       # mobody.py:60-72
    def __init__(self, state_dim, action_dim, max_action, hidden_size=256):
        super().__init__()
        self.action_dim, self.max_action = action_dim, max_action
        self.network = MLPNetwork(state_dim, action_dim, hidden_size)

    def forward(self, x):
        """tanh(MLP(x)) * max_action through the CUDA policy kernel (no autograd; training uses the
        fused actor update)."""
        x = x.contiguous().float()
        out = torch.empty(x.shape[0], self.action_dim, dtype=torch.float32, device=x.device)
        mp, _keep = _ffi.mlp_params(self.network)
        _ffi.check(_ffi.lib().mobody_policy_forward(_ffi.ptr(x), x.shape[0], x.shape[1], self.action_dim, C.byref(mp),
                                                    float(self.max_action), _ffi.ptr(out), _ffi.stream_ptr(x.device)))
        return out

    def forward_autograd(self, x):
        """Same function through torch ops (differentiable): used only by the torch reference update (_train_torch_path)."""
        return torch.tanh(self.network(x)) * self.max_action


class DoubleQFunc(nn.Module):                                  # mobody.py:74-83
    def __init__(self, state_dim, action_dim, hidden_size=256):
        super().__init__()
        self.network1 = MLPNetwork(state_dim + action_dim, 1, hidden_size)
        self.network2 = MLPNetwork(state_dim + action_dim, 1, hidden_size)

    def forward(self, state, action):                          # torch ops: the torch reference update only
        x = torch.cat((state, action), dim=1)
        return self.network1(x), self.network2(x)


class Classifier(nn.Module):                                   # mobody.py:11-33 (domain classifier of DARA / DARC)
    def __init__(self, state_dim, action_dim, hidden_size=256, gaussian_noise_std=1.0):
        super().__init__()
        self.action_dim, self.gaussian_noise_std = action_dim, gaussian_noise_std
        self.sa_classifier = MLPNetwork(state_dim + action_dim, 2, hidden_size)
        self.sas_classifier = MLPNetwork(2 * state_dim + action_dim, 2, hidden_size)



_SM_COUNT = {}


def _sm_count(device):
    key = str(device)
    if key not in _SM_COUNT:
        _SM_COUNT[key] = torch.cuda.get_device_properties(device).multi_processor_count
    return _SM_COUNT[key]


def _adam(params, lr):
    """torch.optim.Adam with its per-parameter state created up front (mobody.py:127-135).  The fused kernels update
    ``exp_avg`` / ``exp_avg_sq`` of this state IN PLACE, so ``state_dict()`` is the reference's optimizer checkpoint and the
    torch-path branches continue from the same moments."""
    opt = torch.optim.Adam(params, lr=lr)
    for g in opt.param_groups:
        for prm in g["params"]:
            opt.state[prm] = {"step": torch.tensor(0.0), "exp_avg": torch.zeros_like(prm), "exp_avg_sq": torch.zeros_like(prm)}
    return opt


def _storage_idle(t):
    """True when nothing but ``t`` itself references its storage (no view handed out earlier is still alive)."""
    try:
        return torch._C._storage_Use_Count(t.untyped_storage()._cdata) <= 2
    except Exception:       # no such hook in this torch build: treat the slab as busy (allocate a fresh one)
        return False


def _wgrad_splits(n_rows, tiles_per_launch, device, sm_count=None, ctas_per_sm=2, cta_overhead=0.0, per_split=0.0):
    """Row splits of the weight-gradient launches.  A launch runs ``tiles * nsplit`` CTAs of 128 x 64 outputs, two per
    SM, each walking its rows in chunks of 32: pick the split count (<= 64) that minimises rounds x chunks per CTA
    summed over the launches of an update (tiles: critic 2 x (8 + 2), actor 8 + 2), i.e. avoid a nearly empty last
    round.  Any value gives the same result up to fp32 summation order; the order is fixed for a given value.
    ``cta_overhead`` (a CTA's fixed cost -- set-up, epilogue of a whole output tile -- in units of one 32-row chunk) and
    ``per_split`` (what one more partial costs the Adam launches, same unit) make the model prefer fewer, longer splits:
    used for the tcgen05 tiles, where they are measured (batch 4096: 27 splits 2 343, 54 splits 2 269, 16 splits 2 195 updates/s)."""
    if sm_count is None:
        sm_count = _sm_count(device)
    slots, chunks = ctas_per_sm * sm_count, (n_rows + 31) // 32
    best, best_cost = 1, None
    for n in range(1, min(64, chunks) + 1):
        per = (chunks + n - 1) // n
        cost = sum(((t * n + slots - 1) // slots) for t in tiles_per_launch) * (per + cta_overhead) + per_split * n
        if best_cost is None or cost < best_cost:
            best, best_cost = n, cost
    return best

def pipe_bounds(B, wave, first=None, rows=None):
    """Chunk boundaries of a pipelined one-step rollout of B start states on a device whose full wave is ``wave`` rows
    (SM count x 128-row tiles): a one-wave first chunk (little H2D exposed before the first kernel), two-wave chunks after
    it, and the sub-wave remainder as its own last chunk (little D2H exposed after the last kernel).  Whole waves per
    chunk: chunking adds no partially filled round to the step kernel."""
    first = wave if first is None else first
    rows = 2 * wave if rows is None else rows
    bounds, lo = [0], min(first, B)
    while lo < B:
        bounds.append(lo)
        lo += rows
    bounds.append(B)
    tail = (B - bounds[-2]) % wave
    if 0 < tail < B - bounds[-2] and tail <= wave // 2:
        bounds.insert(-1, B - tail)                           # split the sub-wave remainder off the last chunk
    return bounds


class MOBODY(object):
    def __init__(self, config, device, target_entropy=None):   # mobody.py:91-135
        self.config, self.device = config, torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("mobody_b200.MOBODY needs a CUDA device (there is no CPU path)")
        if config.get("hidden_sizes", 256) != 256:
            raise NotImplementedError("mobody_b200 kernels are built for hidden_sizes=256")
        self.discount, self.tau = config["gamma"], config["tau"]
        self.update_interval = config.get("update_interval", 2)   # read but unused by the reference too
        S, A = config["state_dim"], config["action_dim"]
        self.seed = int(config.get("seed", 0))
        self.fake_replay_buffer = ReplayBuffer(S, A, self.device, seed=ReplayBuffer.stream_seed(self.seed, "fake"))
        self.penalty_type = config.get("penalty_type", "par")
        self.total_it = 0
        self.q_funcs = DoubleQFunc(S, A).to(self.device)
        self.target_q_funcs = copy.deepcopy(self.q_funcs)
        for p in self.target_q_funcs.parameters():
            p.requires_grad = False
        self.v_func = ValueFunc(S, A).to(self.device)
        self.policy = Policy(S, A, config["max_action"]).to(self.device)
        self.classifier = Classifier(S, A, 256, config.get("gaussian_noise_std", 1.0)).to(self.device)   # :134
        self.dynamics = None                                     # injected by the caller (train_mobody.py:888)
        # the reference's four optimizers (mobody.py:127-135).  The fused kernels own the Adam arithmetic; these objects
        # own the moments (updated in place by the kernels) and serve the checkpoint files and the torch-path branches.
        self._opts = {"q": _adam(self.q_funcs.parameters(), config["critic_lr"]),
                      "v": _adam(self.v_func.parameters(), config["critic_lr"]),
                      "pi": _adam(self.policy.parameters(), config["actor_lr"]),
                      "cls": _adam(self.classifier.parameters(), config["actor_lr"])}
        self._t_q = self._t_pi = self._t_cls = self._t_v = 0     # steps taken by the fused kernels (host counters) ...
        self._steps_dirty = set()                                # ... flushed into the optimizers' ``step`` tensors on access
        self._moment_cache = {}
        self._cls_ws, self._cls_scalars = None, torch.zeros(2, dtype=torch.float32, device=self.device)
        self._train_ws = None
        self._scalars = torch.zeros(16, dtype=torch.float32, device=self.device)
        self._par_mean = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._par_ws = None
        self._roll_ws = {}                                       # (T, B, S, A) -> rollout scratch
        self._eval_ws = {}                                       # (B, S, A, slot) -> evaluate_in_model scratch
        self._eval_draw = 0                                      # Philox step counter of evaluate_in_model
        self._host_slabs = []                                    # pinned staging slabs of rollout() results (reused when idle)
        self._pipe_streams, self._pipe_hdr = None, None          # side streams / pinned header of the pipelined rollout()
        self._pipe_plan_cache = None                             # (key, per-chunk launch plan)
        sm = _sm_count(self.device)
        self.PIPE_FIRST = sm * 128      # first chunk of a pipelined rollout(): one wave of 128-row tiles, so the first kernel starts after a short H2D
        self.PIPE_ROWS = 2 * sm * 128   # later chunks: two full waves
        self._wave = sm * 128

    # ------------------------------------------------------------------ optimizers (mobody.py:127-135)
    _OPT_COUNTER = {"q": "_t_q", "v": "_t_v", "pi": "_t_pi", "cls": "_t_cls"}

    def _optimizer(self, name):
        """The torch optimizer ``name`` with its ``step`` tensors brought up to date with the fused kernels' counters."""
        opt = self._opts[name]
        if name in self._steps_dirty:
            t = float(getattr(self, self._OPT_COUNTER[name]))
            for st in opt.state.values():
                st["step"].fill_(t)
            self._steps_dirty.discard(name)
        return opt

    q_optimizer = property(lambda self: self._optimizer("q"))
    v_optimizer = property(lambda self: self._optimizer("v"))
    policy_optimizer = property(lambda self: self._optimizer("pi"))
    classifier_optimizer = property(lambda self: self._optimizer("cls"))

    def _pull_steps(self, name):
        """After torch stepped (or loaded) optimizer ``name``: adopt its step count and its (possibly new) moment tensors."""
        opt = self._opts[name]
        steps = [int(st["step"]) for st in opt.state.values()]
        setattr(self, self._OPT_COUNTER[name], max(steps) if steps else 0)
        self._steps_dirty.discard(name)
        self._moment_cache.pop(name, None)

    def _moments(self, name, modules):
        """[(exp_avg list, exp_avg_sq list) per MLP] of optimizer ``name`` in mlp_tensors order (the kernels' operand order)."""
        ent = self._moment_cache.get(name)
        if ent is None:
            opt = self._opts[name]
            ent = []
            for mlp in modules:
                prm = [t for li in (0, 2, 4) for t in (mlp.network[li].weight, mlp.network[li].bias)]
                ent.append(([opt.state[q]["exp_avg"] for q in prm], [opt.state[q]["exp_avg_sq"] for q in prm]))
            for m_list, v_list in ent:
                for t in m_list + v_list:
                    if not (t.is_cuda and t.is_contiguous() and t.dtype == torch.float32):
                        raise RuntimeError("mobody_b200: Adam moments must be contiguous fp32 CUDA tensors")
            self._moment_cache[name] = ent
        return ent

    def select_action(self, state, policy, cuda=False):          # mobody.py:138-144
        with torch.no_grad():
            s = _ffi.f32(state, self.device).view(-1, self.config["state_dim"])
            action = policy(s)
            return action.squeeze() if cuda else action.squeeze().cpu().numpy()

    # ------------------------------------------------------------------ rollout
    def _rollout_workspace(self, T, B, S, A, slot=0):
        """Device scratch of mobody_rollout for (T, B): allocated once and reused (the result slab is not part of it).
        ``slot`` separates workspaces of rollouts that are in flight at the same time on different streams."""
        key = (T, B, S, A, slot)
        ws = self._roll_ws.get(key)
        if ws is None:
            dev, f = self.device, dict(dtype=torch.float32, device=self.device)
            ws = dict(obss=torch.empty(T, B, S, **f), acts=torch.empty(T, B, A, **f), nexts=torch.empty(T, B, S, **f),
                      rews=torch.empty(T, B, 1, **f), pens=torch.empty(T, B, 1, **f), raw=torch.empty(B, 1, **f),
                      terms=torch.empty(T, B, dtype=torch.uint8, device=dev), mean=torch.empty(7, B, S, **f),
                      row_ids=torch.empty(T, B, dtype=torch.int64, device=dev),
                      counts=torch.zeros(T + 2, dtype=torch.int32, device=dev),
                      pos=torch.empty(max(T * B, 1), dtype=torch.int32, device=dev),
                      scratch=torch.empty(int(_ffi.lib().mobody_compact_scratch_ints(T * B)), dtype=torch.int32, device=dev),
                      stats=torch.zeros(int(_ffi.lib().mobody_rollout_stats_doubles()), dtype=torch.float64, device=dev),
                      ticket=torch.zeros(1, dtype=torch.int32, device=dev))
            if len(self._roll_ws) >= 8:                       # a handful of shapes per run (50 000 / 2 000 starts)
                self._roll_ws.pop(next(iter(self._roll_ws)))
            self._roll_ws[key] = ws
        return ws

    @torch.no_grad()
    def _take_draws(self, T, step0=None):
        """Philox step counters of a T-step rollout: by default the dynamics object's monotonically increasing draw
        counter (every rollout / step call consumes fresh noise and member picks, like the reference's torch.normal /
        np.random.choice), or an explicit base ``step0`` (tests, replays) that leaves the counter alone."""
        if step0 is not None:
            return int(step0)
        base = self.dynamics._draw
        self.dynamics._draw += int(T)
        return base

    def _rollout_desc(self, init_obss, T, use_trg, ws, packed, eps=None, idx=None, row0=0, step0=None, verify_images=True):
        """A filled mobody_rollout_desc for start states ``init_obss`` [B,S] (device, contiguous) on workspace ``ws``.
        ``packed``: destination of the pack stage (multi-GPU: this rank's slot of its receive buffer).  Returns (desc, keep-alive)."""
        B, S = init_obss.shape
        d = _ffi.RolloutDesc()
        keep = self.dynamics.fill_step_desc(d.step, B, S, self.device, policy=self.policy.network, max_action=self.policy.max_action,
                                            use_trg=use_trg, verify_images=verify_images)
        d.step.obs, d.step.mean, d.step.raw_reward = _ffi.ptr(init_obss), _ffi.ptr(ws["mean"]), _ffi.ptr(ws["raw"])
        d.step.step, d.step.row0 = self._take_draws(T, step0), int(row0)
        d.T, d.filter_bad_rollout = T, int(bool(self.config.get("filter_bad_rollout", 1)))
        d.env_filter = float(self.config.get("env_filter", 0.0))
        d.eps_all, d.idx_all = _ffi.ptr(eps), _ffi.ptr(idx)
        for k in ("obss", "acts", "nexts", "rews", "pens", "terms", "row_ids", "counts", "pos", "scratch", "stats", "ticket"):
            setattr(d, k, _ffi.ptr(ws[k]))
        if T == 1:
            d.obss = d.step.obs            # one step: the start states ARE obss[0] (aliasing skips the copy, include/mobody_b200.h)
        d.packed = _ffi.ptr(packed)
        return d, (keep, init_obss, eps, idx, ws, packed)

    def verify_images(self, use_trg=True):
        """Bring the packed tensor-core weight images up to date on the CURRENT stream (device-side checksum, re-pack when the
        parameters changed).  Call once before enqueueing several rollouts with ``verify_images=False`` on other streams."""
        probe = _ffi.StepDesc()
        return self.dynamics.fill_step_desc(probe, 1, self.config["state_dim"], self.device, policy=self.policy.network,
                                            max_action=self.policy.max_action, use_trg=use_trg)

    def rollout_streams(self):
        """Two side streams for INDEPENDENT rollouts.  A rollout of B start states is ceil(B / 128) tiles on the device's SMs
        (100 000 states on 148 SMs: 5.28 rounds, the sixth 72 % idle); enqueued on alternating streams -- each with its own
        ``ws_slot``, after one verify_images() on the stream they fork from -- the tail round of one rollout runs beside the
        first round of the next.  The refresh block uses them for its three independent dynamics calls."""
        if getattr(self, "_roll_streams", None) is None:
            self._roll_streams = (torch.cuda.Stream(self.device), torch.cuda.Stream(self.device))
        return self._roll_streams

    def rollout_device(self, init_obss, rollout_length, use_trg=True, *, eps=None, idx=None, row0=0, out_packed=None,
                       sync=True, ws_slot=0, step0=None, verify_images=True):
        """T-step imagined rollout entirely on the device (mobody.py:596-657 without its per-step D2H copies and
        host masks): ONE C-ABI call (mobody_rollout) enqueues the T fused steps, the compactions between them, the
        concatenation + penalty filter and the packing of the kept transitions.

        eps: optional [T,7,B,S] / idx: optional [T,B] injected draws (step t uses the first B_t rows, exactly what
        the reference consumes when fed the same arrays).
        step0: explicit Philox step counter of the first step (default: the dynamics' running draw counter, advanced by T).
        out_packed: optional preallocated [>= T*B, 2S+A+3] CUDA tensor receiving the kept transitions as rows
        [obs | act | next_obs | reward | terminal | penalty] (the slab the multi-GPU all-gather ships).
        sync=True: one host read at the end (row counts + reward sum); the returned dict holds [M, .] column views of
        the slab.  sync=False: nothing is read back; the dict holds capacity-sized views (rows >= kept are
        unspecified) and info carries device tensors only (``kept_dev``, ``counts_dev``, ``stats_dev`` — views of the
        cached workspace: consume them on the stream before the next rollout of the same shape overwrites them).
        Returns (dict of CUDA tensors, info) or (None, None) when rollout_length == 0."""
        if rollout_length == 0:
            return None, None                                    # mobody.py:602-603
        dyn, dev, T = self.dynamics, self.device, int(rollout_length)
        init_obss = _ffi.f32(init_obss, dev)
        B, S = init_obss.shape
        A = self.config["action_dim"]
        W = 2 * S + A + 3
        ws = self._rollout_workspace(T, B, S, A, ws_slot)
        packed = out_packed if out_packed is not None else torch.empty(max(T * B, 1), W, dtype=torch.float32, device=dev)
        assert packed.shape[1] == W and packed.shape[0] >= T * B and packed.is_contiguous()
        if eps is not None:
            eps = _ffi.f32(eps, dev); assert tuple(eps.shape) == (T, 7, B, S)
        if idx is not None:
            idx = torch.as_tensor(np.asarray(idx) if not torch.is_tensor(idx) else idx).to(device=dev, dtype=torch.int64).contiguous()
        counts = ws["counts"]
        if B > 0:
            d, keep = self._rollout_desc(init_obss, T, use_trg, ws, packed, eps, idx, row0, step0, verify_images)   # noqa: F841
            _ffi.check(_ffi.lib().mobody_rollout(C.byref(d), _ffi.stream_ptr(dev)))
        else:
            counts.zero_(); ws["stats"][:2].zero_()
        mdev = counts[T + 1:T + 2]
        if sync:
            host = torch.cat([counts.double(), ws["stats"][:2]]).cpu()       # the single host read
            n_per_step = [int(v) for v in host[:T]]
            M, num_transitions, rew_sum = int(host[T + 1]), int(host[T + 3]), float(host[T + 2])
            info = {"num_transitions": num_transitions, "reward_mean": rew_sum / max(num_transitions, 1),
                    "rows_per_step": n_per_step, "kept": M, "kept_dev": mdev}
        else:
            M = T * B
            info = {"kept_dev": mdev, "counts_dev": counts, "stats_dev": ws["stats"][:2], "capacity": T * B}
        out, c0 = {}, 0
        for name, w in (("obss", S), ("actions", A), ("next_obss", S), ("rewards", 1), ("terminals", 1), ("penalty", 1)):
            out[name] = packed[:M, c0:c0 + w]
            c0 += w
        info["packed"] = packed
        return out, info

    # ------------------------------------------------------------------ policy evaluation in the learned model
    @property
    def eval_seed(self):
        """Philox key of evaluate_in_model: a stream of its own under the dynamics seed, so evaluations never reuse the
        training rollouts' draws."""
        return ReplayBuffer.stream_seed(self.dynamics.seed, "eval")

    def _eval_workspace(self, B, S, A, slot=0):
        """Device scratch of mobody_model_eval for B start states (its size does not depend on the horizon).  ``slot``
        separates workspaces of evaluations in flight at the same time on different streams."""
        key = (B, S, A, slot)
        ws = self._eval_ws.get(key)
        if ws is None:
            ws = torch.empty(int(_ffi.lib().mobody_model_eval_workspace_bytes(B, S, A)), dtype=torch.uint8, device=self.device)
            if len(self._eval_ws) >= 4:
                self._eval_ws.pop(next(iter(self._eval_ws)))
            self._eval_ws[key] = ws
        return ws

    def _launch_model_eval(self, init_obss, H, gamma, penalized, use_trg, row0, step0, ws_slot=0, verify_images=True):
        """Enqueue one mobody_model_eval on the current stream; no host synchronisation.  Returns (outputs, counts[H+1])."""
        dev = self.device
        B, S = init_obss.shape
        out = {"returns": torch.empty(B, dtype=torch.float64, device=dev),                  # (the library zeroes them)
               "discounted_returns": torch.empty(B, dtype=torch.float64, device=dev),
               "lengths": torch.empty(B, dtype=torch.int32, device=dev)}
        counts = torch.zeros(H + 1, dtype=torch.int32, device=dev)
        if B > 0:
            d = _ffi.ModelEvalDesc()
            keep = self.dynamics.fill_step_desc(d.step, B, S, dev, policy=self.policy.network, max_action=self.policy.max_action,  # noqa: F841
                                                use_penalty=penalized, use_trg=use_trg, verify_images=verify_images)
            ws = self._eval_workspace(B, S, self.config["action_dim"], ws_slot)
            d.step.obs, d.step.seed, d.step.step, d.step.row0 = _ffi.ptr(init_obss), self.eval_seed, int(step0), int(row0)
            d.H, d.gamma, d.workspace, d.workspace_bytes = H, float(gamma), _ffi.ptr(ws), ws.numel()
            d.ret, d.ret_disc = _ffi.ptr(out["returns"]), _ffi.ptr(out["discounted_returns"])
            d.length, d.counts = _ffi.ptr(out["lengths"]), _ffi.ptr(counts)
            _ffi.check(_ffi.lib().mobody_model_eval(C.byref(d), _ffi.stream_ptr(dev)))
        return out, counts

    @torch.no_grad()
    def evaluate_in_model(self, init_obss, horizon=1000, *, gamma=None, penalized=False, use_trg=True, row0=0, step0=None):
        """Score the policy without a simulator: one episode per start state in the learned dynamics (the target-domain model
        with ``use_trg``), driven by the deterministic policy, up to ``horizon`` steps.  An episode's return sums the step
        rewards up to and including its first terminal step, the quantity eval_policy prints (train_mobody.py:53-205); with
        ``penalized`` the reward is the rollout's uncertainty-penalized reward.  ONE C-ABI call (mobody_model_eval) runs
        the whole horizon on the device in memory independent of the horizon.

        Draws: Philox keyed on (eval_seed, step0 + t, row0 + i), so a start state's episode does not depend on how the
        start states are batched or sharded (give each shard its global ``row0``).  ``step0`` defaults to this object's
        evaluation counter, advanced by ``horizon`` per call; the training draw counter (dynamics._draw) is never touched,
        so evaluations interleaved with training change no training result.
        Returns ({returns, discounted_returns (float64), lengths (int32)}: CUDA tensors [B], info) with info holding
        ``return_mean``, ``length_mean`` and ``live_per_step`` (live rows entering each step, then the rows still live after
        the last), read back with one host read."""
        H = int(horizon)
        init_obss = _ffi.f32(init_obss, self.device)
        gamma = self.config["gamma"] if gamma is None else gamma
        out, counts = self._launch_model_eval(init_obss, H, gamma, penalized, use_trg, row0,
                                              self._eval_draw if step0 is None else step0)
        if step0 is None:
            self._eval_draw += H
        host = torch.cat([counts.double(), out["returns"].mean()[None], out["lengths"].double().mean()[None]]).cpu()   # the single host read
        info = {"return_mean": float(host[H + 1]), "length_mean": float(host[H + 2]),
                "live_per_step": [int(v) for v in host[:H + 1]]}
        return out, info

    def _host_slab(self, rows, W):
        """Pinned staging slab for a rollout() result.  The CPU tensors rollout() returns are views of the slab and own it
        for as long as any of them is alive (like the reference's fresh tensors, mobody.py:641-657): a slab is reused only
        when its storage is referenced by nobody else; otherwise a new one is allocated and the busy one is left to its
        holder.  A caller that drops each result before the second-next call (train()'s add_batch copies immediately)
        cycles through two slabs with no allocation."""
        for slab in self._host_slabs:
            if slab.shape[1] == W and slab.shape[0] >= rows and _storage_idle(slab):
                return slab
        slab = torch.empty(max(rows, 1), W, dtype=torch.float32, pin_memory=True)
        self._slab_allocs = getattr(self, "_slab_allocs", 0) + 1
        self._host_slabs = [t for t in self._host_slabs if not _storage_idle(t)][-3:] + [slab]   # idle leftovers are too small: drop them
        return slab

    def rollout(self, init_obss, rollout_length, use_trg=True, **kw):
        """Reference signature and return convention (mobody.py:596-657): dict of CPU tensors + info.
        The kept rows are copied D2H once, into a pinned staging slab; the dict values are column views of it.
        One-step rollouts of many start states are pipelined in chunks on two side streams (H2D of chunk c+1 and D2H
        of chunk c-1 overlap the kernels of chunk c); rows are independent and Philox is keyed on the global row id,
        so the result is identical to the unchunked call (row order included)."""
        T = int(rollout_length)
        if T == 0:
            return None, None
        S, A = self.config["state_dim"], self.config["action_dim"]
        W = 2 * S + A + 3
        B = int(init_obss.shape[0])
        if T == 1 and B >= 2 * self.PIPE_ROWS and not kw:
            res_host, n_tr, rsum, M = self._rollout_pipelined(init_obss, use_trg, S, A, W)
        else:
            out, info = self.rollout_device(init_obss, T, use_trg, **kw)
            M, packed = info["kept"], info["packed"]
            res_host = self._host_slab(M, W)[:M]
            res_host.copy_(packed[:M], non_blocking=True)
            torch.cuda.current_stream(self.device).synchronize()
            n_tr, rsum = info["num_transitions"], info["reward_mean"] * info["num_transitions"]
        if self.config.get("filter_bad_rollout", 1):
            print("filtered rollout", M, n_tr)                                   # mobody.py:653
        res, c0 = {}, 0
        for name, w in (("obss", S), ("actions", A), ("next_obss", S), ("rewards", 1), ("terminals", 1), ("penalty", 1)):
            res[name] = res_host[:, c0:c0 + w]
            c0 += w
        return res, {"num_transitions": n_tr, "reward_mean": rsum / max(n_tr, 1)}

    def _pipe_bounds(self, B):
        return pipe_bounds(B, self._wave, self.PIPE_FIRST, self.PIPE_ROWS)

    def _pipe_plan(self, B, S, A, W, use_trg, bounds):
        """Per-chunk launch plan of the pipelined rollout (device input / output buffers, workspace, a filled
        mobody_rollout_desc, an event), cached while nothing it points to changes: a chunk then costs one H2D
        enqueue, ONE C-ABI call and two 8-byte D2H enqueues of host time."""
        dev, dyn = self.device, self.dynamics
        probe = _ffi.StepDesc()
        # also (re)builds the packed weight images on the caller's stream, before the side streams fork from it
        keep0 = dyn.fill_step_desc(probe, 1, S, dev, policy=self.policy.network, max_action=self.policy.max_action, use_trg=use_trg)
        filt, env_filter = int(bool(self.config.get("filter_bad_rollout", 1))), float(self.config.get("env_filter", 0.0))
        key = (tuple(bounds), S, A, bool(use_trg), probe.precision, probe.dyn_pack, probe.policy_pack,
               C.addressof(probe.dyn.contents), C.addressof(probe.policy.contents), probe.elites, probe.n_elites,
               probe.penalty_coef, probe.term_kind, probe.seed, probe.max_action, filt, env_filter, self._wave)
        if self._pipe_plan_cache is not None and self._pipe_plan_cache[0] == key:
            return self._pipe_plan_cache[1]
        plan = []
        for c in range(len(bounds) - 1):
            lo, hi = bounds[c], bounds[c + 1]
            n = hi - lo
            ws = self._rollout_workspace(1, n, S, A, 1 + (c & 1))
            x = torch.empty(n, S, dtype=torch.float32, device=dev)
            packed = torch.empty(n, W, dtype=torch.float32, device=dev)
            d = _ffi.RolloutDesc()
            keep = dyn.fill_step_desc(d.step, n, S, dev, policy=self.policy.network, max_action=self.policy.max_action, use_trg=use_trg)
            d.step.obs, d.step.mean, d.step.raw_reward = _ffi.ptr(x), _ffi.ptr(ws["mean"]), _ffi.ptr(ws["raw"])
            d.step.step, d.step.row0 = 0, int(lo)                 # .step is patched per call (fresh Philox draws)
            d.T, d.filter_bad_rollout, d.env_filter = 1, filt, env_filter
            d.eps_all, d.idx_all = None, None
            for k in ("obss", "acts", "nexts", "rews", "pens", "terms", "row_ids", "counts", "pos", "scratch", "stats", "ticket"):
                setattr(d, k, _ffi.ptr(ws[k]))
            d.obss = d.step.obs                                   # T == 1: no copy of the start states
            d.packed = _ffi.ptr(packed)
            plan.append(dict(lo=lo, hi=hi, x=x, packed=packed, desc=d, ref=C.byref(d), keep=(keep, keep0, ws),
                             kept_dev=ws["counts"][2:3], stats_dev=ws["stats"][:2], ev=torch.cuda.Event()))
        self._pipe_plan_cache = (key, plan)
        return plan

    def _rollout_pipelined(self, init_obss, use_trg, S, A, W):
        dev, lib = self.device, _ffi.lib()
        if not torch.is_tensor(init_obss):
            init_obss = torch.as_tensor(np.asarray(init_obss, dtype=np.float32))
        B = init_obss.shape[0]
        bounds = self._pipe_bounds(B)
        n = len(bounds) - 1
        if self._pipe_streams is None:
            self._pipe_streams = [torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)]   # 2 compute + 1 D2H
        if self._pipe_hdr is None or self._pipe_hdr[0].shape[0] < n:
            self._pipe_hdr = (torch.zeros(max(n, 8), 1, dtype=torch.int32).pin_memory(),      # kept rows per chunk
                              torch.zeros(max(n, 8), 2, dtype=torch.float64).pin_memory())    # [reward sum, produced]
        hdr_kept, hdr_stats = self._pipe_hdr
        cur = torch.cuda.current_stream(dev)
        plan = self._pipe_plan(B, S, A, W, use_trg, bounds)
        draw = self._take_draws(1)
        ready = torch.cuda.Event(); ready.record(cur)
        host = self._host_slab(B, W)
        for c, ch in enumerate(plan):
            st = self._pipe_streams[c & 1]
            with torch.cuda.stream(st):
                st.wait_event(ready)
                ch["x"].copy_(init_obss[ch["lo"]:ch["hi"]], non_blocking=True)
                ch["desc"].step.step = draw
                _ffi.check(lib.mobody_rollout(ch["ref"], C.c_void_p(st.cuda_stream)))
                # [kept | reward sum, produced] of this chunk -> pinned header rows (stream-ordered 4- and 16-byte D2H)
                hdr_kept[c].copy_(ch["kept_dev"], non_blocking=True)
                hdr_stats[c].copy_(ch["stats_dev"], non_blocking=True)
                ch["ev"].record(st)
        off, n_tr, rsum = 0, 0, 0.0
        copy_stream = self._pipe_streams[2]                       # dedicated copy stream: never queued behind a later chunk's kernels
        for c, ch in enumerate(plan):
            ch["ev"].synchronize()                                # chunk c is done; later chunks keep the GPU busy
            m = int(hdr_kept[c, 0]); rsum += float(hdr_stats[c, 0]); n_tr += int(hdr_stats[c, 1])
            with torch.cuda.stream(copy_stream):
                host[off:off + m].copy_(ch["packed"][:m], non_blocking=True)
            off += m
        copy_stream.synchronize()
        return host[:off], n_tr, rsum, off

    # ------------------------------------------------------------------ DARA domain classifier
    def classifier_step_on_rows(self, rows, label, *, noise_sas=None, noise_sa=None):
        """One fused classifier update (forward on noise-perturbed inputs, cross-entropy on the softmaxed outputs,
        backward, Adam) on packed batch rows [N, RW] with int32 domain labels [N].  Asynchronous; the two losses land
        in ``self._cls_scalars`` = [loss_sa, loss_sas] (device).  mobody.py:11-33, 146-181."""
        cfg = self.config
        S, A = cfg["state_dim"], cfg["action_dim"]
        N = rows.shape[0]
        nsplit = _wgrad_splits(N, (16 + 2 * ((2 * S + A + 63) // 64) + 2 * ((S + A + 63) // 64),), self.device)
        lib = _ffi.lib()
        need = int(lib.mobody_classifier_workspace_bytes(N, S, A, nsplit))
        if self._cls_ws is None or self._cls_ws.numel() < need:
            self._cls_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        self._t_cls += 1; self._steps_dirty.add("cls")
        d = _ffi.ClassifierDesc()
        d.rows, d.N, d.S, d.A, d.row_width = _ffi.ptr(rows), N, S, A, rows.shape[1]
        d.label = _ffi.ptr(label)
        # injected draws: the device copies must stay referenced until the launch is enqueued (a dropped temporary's block
        # is handed to the very next allocation by the caching allocator)
        noise_sas = None if noise_sas is None else _ffi.f32(noise_sas, self.device)
        noise_sa = None if noise_sa is None else _ffi.f32(noise_sa, self.device)
        d.noise_sas, d.noise_sa = _ffi.ptr(noise_sas), _ffi.ptr(noise_sa)
        d.noise_std, d.seed, d.draw = float(self.classifier.gaussian_noise_std), int(cfg.get("seed", 0)), self._t_cls
        cl = self.classifier
        d.sas, d.sa = _ffi.mlp_state(_ffi.mlp_tensors(cl.sas_classifier)), _ffi.mlp_state(_ffi.mlp_tensors(cl.sa_classifier))
        (sa_m, sa_v), (sas_m, sas_v) = self._moments("cls", (cl.sa_classifier, cl.sas_classifier))
        d.sas_m, d.sas_v = _ffi.mlp_state(sas_m), _ffi.mlp_state(sas_v)
        d.sa_m, d.sa_v = _ffi.mlp_state(sa_m), _ffi.mlp_state(sa_v)
        d.t, d.lr, d.nsplit = self._t_cls, float(cfg["actor_lr"]), nsplit           # Adam(lr=actor_lr), mobody.py:135
        d.workspace, d.workspace_bytes, d.scalars_out = _ffi.ptr(self._cls_ws), self._cls_ws.numel(), _ffi.ptr(self._cls_scalars)
        _ffi.check(lib.mobody_classifier_step(C.byref(d), _ffi.stream_ptr(self.device)))
        return self._cls_scalars

    def update_classifier(self, src_replay_buffer, tar_replay_buffer, batch_size, writer=None, *, _inject=None):
        """Reference signature (mobody.py:146-181) -> (loss_sa, loss_sas) as 0-d device tensors.
        ``_inject`` optionally scripts the draws of np.random.randint / torch.randperm / torch.randn_like:
        {src, tar, perm, noise_sas, noise_sa}."""
        if self.config.get("penalize_fake", 0):
            raise NotImplementedError("penalize_fake=1 mixes batch sizes the reference's own labels do not cover (mobody.py:149-162)")
        inj = _inject or {}
        B = int(batch_size)
        RW = src_replay_buffer.RW
        rows = torch.empty(2 * B, RW, dtype=torch.float32, device=self.device)
        src_replay_buffer.sample_rows(B, inj.get("src"), out=rows[:B])
        tar_replay_buffer.sample_rows(B, inj.get("tar"), out=rows[B:])
        perm = inj.get("perm")
        perm = torch.randperm(2 * B, device=self.device) if perm is None else torch.as_tensor(np.asarray(perm)).to(self.device)
        rows = rows[perm]                                                            # :164-166
        label = (perm >= B).to(torch.int32).contiguous()                             # zeros for src, ones for tar (:162)
        sc = self.classifier_step_on_rows(rows, label, noise_sas=inj.get("noise_sas"), noise_sa=inj.get("noise_sa"))
        if writer is not None and self.total_it % 5000 == 0:                         # :176-179
            v = sc.cpu().tolist()
            writer.add_scalar("train/sas classifier loss", v[1], global_step=self.total_it)
            writer.add_scalar("train/sa classifier loss", v[0], global_step=self.total_it)
        return sc[0], sc[1]

    @torch.no_grad()
    def dara_relabel(self, src_replay_buffer, penalty_out=None):
        """One-off relabel of the source rewards with the trained classifier (mobody.py:364-378), in place on the
        device-resident buffer rows: reward += penalty_coef * clamp(log-ratio, -10, 10)."""
        cl = self.classifier
        sas, k0 = _ffi.mlp_params(cl.sas_classifier)
        sa, k1 = _ffi.mlp_params(cl.sa_classifier)
        buf = src_replay_buffer
        _ffi.check(_ffi.lib().mobody_dara_relabel(_ffi.ptr(buf._rows), buf.size, buf.S, buf.A, buf.RW, C.byref(sas), C.byref(sa),
                                                  float(self.config["penalty_coef"]), _ffi.ptr(penalty_out),
                                                  _ffi.stream_ptr(self.device)))
        del k0, k1

    # ------------------------------------------------------------------ train step
    def train_on_rows(self, rows, n_true, *, nsplit=None):
        """One fused critic + Polyak + actor update on packed batch rows [N, RW] (device, rows ordered
        src, tar, fake; the first ``n_true`` rows are the src+tar rows of the BC term).  Asynchronous:
        losses land in ``self._scalars`` (device).  mobody.py:533-573.  The config flags select the update's branches:
        ``advantage`` (value step first, V(s') TD target, V(s_t) advantage weights), ``scale_Q`` and ``q_weighted``;
        the default flags take mobody_train_step, every other combination mobody_train_step_ex.
        ``nsplit`` overrides the row-split count of the weight-gradient GEMMs (1..64; tests)."""
        cfg = self.config
        default = self._default_update()
        advantage = bool(cfg.get("advantage", 0))
        S, A = cfg["state_dim"], cfg["action_dim"]
        N = rows.shape[0]
        if nsplit is None:
            # row splits of the weight-gradient GEMMs (partials summed in Adam, fixed order); 128 x 64 tiles per split:
            # critic 2 x (256 x 256 -> 8, 256 x (S+A) -> 2 per 64 columns), actor 8 + 2 per 64 columns of S
            if N >= _ffi.TC_TRAIN_MIN_ROWS:   # tcgen05 path: 128 x 256 GEMM tiles, two CTAs per SM; critic launch 4 x 2 + 2 x 1 tiles, actor 2 x 2 + 1
                nsplit = _wgrad_splits(N, (10, 5), self.device, ctas_per_sm=2, cta_overhead=4.0, per_split=0.36)
            else:
                nsplit = _wgrad_splits(N, (2 * (8 + 2 * ((S + A + 63) // 64)), 8 + 2 * ((S + 63) // 64)), self.device)
        lib = _ffi.lib()
        need = int(lib.mobody_train_workspace_bytes(N, S, A, nsplit) if default else lib.mobody_train_ex_workspace_bytes(N, S, A, nsplit))
        if self._train_ws is None or self._train_ws.numel() < need:
            self._train_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        self._t_q += 1; self._t_pi += 1
        self._steps_dirty.update(("q", "pi"))
        x = _ffi.TrainExDesc()
        d = x.base
        d.rows, d.N, d.n_true, d.S, d.A, d.row_width = _ffi.ptr(rows), N, int(n_true), S, A, rows.shape[1]
        qt = self.target_q_funcs
        d.policy = _ffi.mlp_state(_ffi.mlp_tensors(self.policy.network))
        d.q1, d.q2 = _ffi.mlp_state(_ffi.mlp_tensors(self.q_funcs.network1)), _ffi.mlp_state(_ffi.mlp_tensors(self.q_funcs.network2))
        d.q1_target, d.q2_target = _ffi.mlp_state(_ffi.mlp_tensors(qt.network1)), _ffi.mlp_state(_ffi.mlp_tensors(qt.network2))
        ((pi_m, pi_v),) = self._moments("pi", (self.policy.network,))
        (q1_m, q1_v), (q2_m, q2_v) = self._moments("q", (self.q_funcs.network1, self.q_funcs.network2))
        d.policy_m, d.policy_v = _ffi.mlp_state(pi_m), _ffi.mlp_state(pi_v)
        d.q1_m, d.q1_v = _ffi.mlp_state(q1_m), _ffi.mlp_state(q1_v)
        d.q2_m, d.q2_v = _ffi.mlp_state(q2_m), _ffi.mlp_state(q2_v)
        d.t_q, d.t_pi = self._t_q, self._t_pi
        d.gamma, d.tau = float(self.discount), float(self.tau)
        d.critic_lr, d.actor_lr = float(cfg["critic_lr"]), float(cfg["actor_lr"])
        d.weight, d.bc_coef, d.max_action = float(cfg["weight"]), float(cfg.get("bc_coef", 1.0)), float(cfg["max_action"])
        d.nsplit, d.workspace, d.workspace_bytes = nsplit, _ffi.ptr(self._train_ws), self._train_ws.numel()
        d.scalars_out = _ffi.ptr(self._scalars)
        if default:
            _ffi.check(lib.mobody_train_step(C.byref(d), _ffi.stream_ptr(self.device)))
            return self._scalars
        x.advantage, x.scale_q, x.q_weighted = int(advantage), int(bool(cfg.get("scale_Q", 1))), int(bool(cfg.get("q_weighted", 1)))
        if advantage:
            self._t_v += 1
            self._steps_dirty.add("v")
            ((v_m, v_v),) = self._moments("v", (self.v_func.network,))
            x.value = _ffi.mlp_state(_ffi.mlp_tensors(self.v_func.network))
            x.value_m, x.value_v, x.t_v = _ffi.mlp_state(v_m), _ffi.mlp_state(v_v), self._t_v
        _ffi.check(lib.mobody_train_step_ex(C.byref(x), _ffi.stream_ptr(self.device)))
        # (parameters were updated in place behind autograd's version counters; the packed tensor-core image of the
        # policy follows them through the library's device-side checksum, dynamics._packed_image)
        return self._scalars

    def loss_scalars(self):
        """Host copy of the last step's diagnostics (one D2H sync; call sparingly).  With advantage=1 it adds the value
        step's loss, mean advantage and mean V(s)."""
        v = self._scalars.cpu().tolist()
        out = dict(q_loss=v[0], q1_mean=v[1], pi_loss=v[2], bc_loss=v[3], q_policy=v[4], q_abs_mean=v[5],
                   w_mean=v[6], w_min=v[7], w_max=v[8], p_w=v[9])
        if self.config.get("advantage", 0):
            out.update(v_loss=v[11], adv_mean=v[12], v_mean=v[13])
        return out

    def _default_update(self):
        cfg = self.config
        return not cfg.get("advantage", 0) and bool(cfg.get("scale_Q", 1)) and bool(cfg.get("q_weighted", 1))

    def _par_penalty(self, rows, n_src, writer, eps=None, idx=None):
        """``penalty_type == 'par'`` (mobody.py:428-434): src_reward -= penalty_coef * mean((s' - s'_model)^2, 1), where
        s'_model is a dynamics step on the batch's (s, a).  Two launches, no host synchronisation: the fused step reads the
        state / action columns of the packed batch rows in place, and ``mobody_par_penalty`` rewrites the reward column."""
        if n_src <= 0:
            return
        cfg, dyn = self.config, self.dynamics
        S, A = cfg["state_dim"], cfg["action_dim"]
        if self._par_ws is None or self._par_ws.next_obs.shape[0] != n_src:
            self._par_ws = StepWorkspace(n_src, S, A, self.device)
        if eps is not None:
            eps = _ffi.f32(eps, self.device)
        if idx is not None:
            idx = torch.as_tensor(np.asarray(idx) if not torch.is_tensor(idx) else idx).to(device=self.device, dtype=torch.int64).contiguous()
        dyn.launch_step(rows[:n_src, :S], rows[:n_src, S:S + A], self._par_ws, eps=eps, idx=idx, step=dyn._draw)
        dyn._draw += 1
        _ffi.check(_ffi.lib().mobody_par_penalty(_ffi.ptr(rows), n_src, S, A, rows.shape[1], _ffi.ptr(self._par_ws.next_obs),
                                                 float(cfg["penalty_coef"]), _ffi.ptr(self._par_mean), _ffi.stream_ptr(self.device)))
        if writer is not None and self.total_it % 100 == 0:                                           # :432-433
            writer.add_scalar("train/reward_penalty_par", float(self._par_mean), global_step=self.total_it)

    def train(self, src_replay_buffer, tar_replay_buffer, batch_size=128, writer=None, wandbrun=None, *, _inject=None):
        """Reference signature (mobody.py:347-578).  ``_inject`` optionally scripts the draws the reference would make
        (parity tests): buffer indices {src, tar, fake, src_init, tar_init} (np.random.randint) and the noise / member
        indices of its dynamics calls {par_eps, par_idx, src_eps, src_idx, tar_eps, tar_idx, sa_eps, sa_idx}."""
        cfg = self.config
        self.total_it += 1
        self.src_replay_buffer, self.tar_replay_buffer = src_replay_buffer, tar_replay_buffer
        if self.penalty_type == "dara" and self.total_it == 1:                                        # :354-378
            for it in range(10 * 500):
                loss_sa, loss_sas = self.update_classifier(src_replay_buffer, tar_replay_buffer, batch_size, writer)
                if it % 2000 == 0:
                    print(loss_sa, loss_sas)
            self.dara_relabel(src_replay_buffer)
        inj = _inject or {}
        n_src, n_tar = int(cfg["src_ratio"] * batch_size), int(cfg["trg_ratio"] * batch_size)
        n_fake = int(cfg["fake_batch_scale"] * batch_size) if cfg["fake_batch_scale"] != 0 else 0
        RW = src_replay_buffer.RW
        rows = torch.empty(n_src + n_tar + n_fake, RW, dtype=torch.float32, device=self.device)
        refresh = (self.total_it - 1) % 5000 == 0
        par = self.penalty_type == "par"
        one_launch = (not inj and not refresh and n_fake and
                      all(b.index_source == "philox" and b.size > 0 for b in (src_replay_buffer, tar_replay_buffer, self.fake_replay_buffer)))
        if one_launch:   # the three buffer samples of this step (:399, 400, 524) as ONE launch: Philox draw + 128-bit row gather
            jobs = (_ffi.SampleJob * 3)()
            for jb, (b, n, lo) in zip(jobs, ((src_replay_buffer, n_src, 0), (tar_replay_buffer, n_tar, n_src),
                                             (self.fake_replay_buffer, n_fake, n_src + n_tar))):
                jb.rows, jb.n, jb.size, jb.draw, jb.seed = _ffi.ptr(b._rows), n, b.size, b._draw, b.seed
                jb.out = rows.data_ptr() + 4 * RW * lo
                b._draw += 1
            _ffi.check(_ffi.lib().mobody_sample_rows(jobs, 3, RW, _ffi.stream_ptr(self.device)))
            if par:
                self._par_penalty(rows, n_src, writer)                                                # :428-434
        else:
            src_replay_buffer.sample_rows(n_src, inj.get("src"), out=rows[:n_src])                    # :399
            tar_replay_buffer.sample_rows(n_tar, inj.get("tar"), out=rows[n_src:n_src + n_tar])       # :400
            if par:
                self._par_penalty(rows, n_src, writer, inj.get("par_eps"), inj.get("par_idx"))
            if refresh:                                                                               # :441-513
                self.refresh_fake_buffer(src_replay_buffer, tar_replay_buffer, inj, batch_size)
            if n_fake:
                self.fake_replay_buffer.sample_rows(n_fake, inj.get("fake"), out=rows[n_src + n_tar:])   # :524
        self.train_on_rows(rows, n_src + n_tar)
        self._train_side_effects(writer, wandbrun)

    def _train_torch_path(self, rows, n_true, writer, wandbrun):
        """The reference update as torch autograd, every branch -- ``advantage=1`` (value-function baseline, mobody.py:210-242,
        533-539), ``scale_Q=0`` (update_policy_1, :278-310), ``q_weighted=0`` (:262-263) and the default flags -- on the same
        device-resident batch rows and the same torch.optim.Adam objects (whose moments the fused kernels share).  train()
        runs the fused kernels for every flag combination; this path is the reference the tests compare them against.  Not a
        performance path."""
        cfg = self.config
        S, A = cfg["state_dim"], cfg["action_dim"]
        state, action, next_state = rows[:, :S], rows[:, S:S + A], rows[:, S + A:2 * S + A]
        reward, not_done = rows[:, 2 * S + A:2 * S + A + 1], rows[:, 2 * S + A + 1:2 * S + A + 2]
        t_state, t_action = state[:n_true], action[:n_true]
        log = writer is not None and self.total_it % 5000 == 0
        q_opt, pi_opt = self.q_optimizer, self.policy_optimizer        # (properties: step tensors flushed)
        if cfg.get("advantage", 0):                                                                   # :210-242, 533-537
            with torch.no_grad():
                qt = torch.min(*self.target_q_funcs(state, action))
            v = self.v_func(state)
            adv = qt - v
            if log:
                writer.add_scalar("train/adv", adv.mean(), self.total_it)
                writer.add_scalar("train/value", v.mean(), self.total_it)
            v_loss = torch.mean(torch.abs(0.7 - (adv < 0).float()) * adv ** 2)                        # asymmetric_l2_loss(adv, 0.7), :85-86
            self.v_optimizer.zero_grad(); v_loss.backward(); self.v_optimizer.step()
            self._pull_steps("v")
        with torch.no_grad():                                                                         # :189-195 / :210-216
            if cfg.get("advantage", 0):
                q_target = self.v_func(next_state)
            else:
                q_target = torch.min(*self.target_q_funcs(next_state, self.policy.forward_autograd(next_state)))
            y = reward + not_done * self.discount * q_target
        q1, q2 = self.q_funcs(state, action)
        if log:
            writer.add_scalar("train/q1", q1.mean(), self.total_it)
            if wandbrun is not None:
                wandbrun.log({"train/q1": q1.mean()}, step=self.total_it, commit=False)
        q_loss = torch.nn.functional.mse_loss(q1, y) + torch.nn.functional.mse_loss(q2, y)
        q_opt.zero_grad(); q_loss.backward(); q_opt.step()                                           # :546-548
        with torch.no_grad():                                                                         # update_target, :183-187
            for tp, qp in zip(self.target_q_funcs.parameters(), self.q_funcs.parameters()):
                tp.data.copy_(self.tau * qp.data + (1.0 - self.tau) * tp.data)
        for prm in self.q_funcs.parameters():
            prm.requires_grad = False
        qv = torch.min(*self.q_funcs(state, self.policy.forward_autograd(state)))                    # :279-281 / :315-317
        p_w = cfg["weight"] / qv.abs().mean().detach() if cfg.get("scale_Q", 1) else 1.0
        pi_loss = p_w * (-qv).mean()
        pred = self.policy.forward_autograd(t_state)                                                  # bc_loss, :246-276
        with torch.no_grad():
            qb = torch.min(*self.q_funcs(t_state, t_action))
            adv = qb - self.v_func(t_state) if cfg.get("advantage", 0) else qb / qb.abs().mean()
            exp_adv = torch.exp(3 * adv).clamp(max=100.0)
        if cfg.get("q_weighted", 1):
            if self.total_it % 1000 == 0:
                print(torch.mean(exp_adv), torch.min(exp_adv), torch.max(exp_adv))
            bc = torch.mean(exp_adv * (pred - t_action) ** 2)
        else:
            bc = torch.mean((pred - t_action) ** 2)
        if log:
            writer.add_scalar("train/exp_adv", exp_adv.mean() if cfg.get("q_weighted", 1) else 1.0, self.total_it)
            writer.add_scalar("train/bc_loss", bc, self.total_it)
        pi_loss = pi_loss + cfg.get("bc_coef", 1.0) * bc
        if log:
            with torch.no_grad():
                q_beh = torch.min(*self.q_funcs(state, action))
            writer.add_scalar("train/q_behavior", q_beh.mean(), self.total_it)
            writer.add_scalar("train/q_policy", qv.mean(), self.total_it)
            writer.add_scalar("train/policy_loss", pi_loss, self.total_it)
            if wandbrun is not None:
                wandbrun.log({"train/q_behavior": q_beh.mean(), "train/q_policy": qv.mean(), "train/policy_loss": pi_loss}, step=self.total_it)
        pi_opt.zero_grad(); pi_loss.backward(); pi_opt.step()                                         # :571-573
        for prm in self.q_funcs.parameters():
            prm.requires_grad = True
        self._pull_steps("q"); self._pull_steps("pi")
        self._scalars[0], self._scalars[2] = q_loss.detach(), pi_loss.detach()

    def _train_side_effects(self, writer, wandbrun):
        cfg = self.config
        if self.total_it % 1000 == 0 and cfg.get("q_weighted", 1):                                    # :269-270
            v = self.loss_scalars()
            print(v["w_mean"], v["w_min"], v["w_max"])
        if not self._default_update():
            self._branch_side_effects(writer, wandbrun)
        elif writer is not None and self.total_it % 5000 == 0:                                        # :203-205, 272-274, 332-344
            v = self.loss_scalars()
            writer.add_scalar("train/q1", v["q1_mean"], self.total_it)
            writer.add_scalar("train/exp_adv", v["w_mean"], self.total_it)
            writer.add_scalar("train/bc_loss", v["bc_loss"], self.total_it)
            writer.add_scalar("train/q_policy", v["q_policy"], self.total_it)
            writer.add_scalar("train/policy_loss", v["pi_loss"], self.total_it)
            if wandbrun is not None:
                wandbrun.log({"train/q1": v["q1_mean"], "train/q_policy": v["q_policy"], "train/policy_loss": v["pi_loss"]},
                             step=self.total_it)

    def _branch_side_effects(self, writer, wandbrun):
        """The writer / wandb keys of the update branches, in _train_torch_path's order (:217-218, 203-205, 272-274, 332-344)."""
        if writer is None or self.total_it % 5000 != 0:
            return
        cfg, it = self.config, self.total_it
        v = self.loss_scalars()
        q_beh = float(self._scalars[14])
        if cfg.get("advantage", 0):
            writer.add_scalar("train/adv", v["adv_mean"], it)
            writer.add_scalar("train/value", v["v_mean"], it)
        writer.add_scalar("train/q1", v["q1_mean"], it)
        if wandbrun is not None:
            wandbrun.log({"train/q1": v["q1_mean"]}, step=it, commit=False)
        writer.add_scalar("train/exp_adv", v["w_mean"] if cfg.get("q_weighted", 1) else 1.0, it)
        writer.add_scalar("train/bc_loss", v["bc_loss"], it)
        writer.add_scalar("train/q_behavior", q_beh, it)
        writer.add_scalar("train/q_policy", v["q_policy"], it)
        writer.add_scalar("train/policy_loss", v["pi_loss"], it)
        if wandbrun is not None:
            wandbrun.log({"train/q_behavior": q_beh, "train/q_policy": v["q_policy"], "train/policy_loss": v["pi_loss"]}, step=it)

    def refresh_fake_buffer(self, src_buf, tar_buf, inj=None, batch_size=128):
        """Synthetic-data refresh (mobody.py:441-475): two policy rollouts through the learned target dynamics and one
        dynamics step on dataset (s, a) pairs, all inserted into the fake buffer without leaving the device.  Every
        dynamics call takes fresh Philox draws (the dynamics' running draw counter) unless ``inj`` scripts them."""
        cfg, inj = self.config, inj or {}
        S, A = cfg["state_dim"], cfg["action_dim"]
        lib, dev, fake = _ffi.lib(), self.device, self.fake_replay_buffer
        src_rows = src_buf.sample_rows(50000, inj.get("src_init"))                                    # :442 (sizes hard-coded there)
        tar_rows = tar_buf.sample_rows(2000, inj.get("tar_init"))                                     # :443
        # The three dynamics calls of the block are independent: they run on two side streams (the tail round of one
        # overlaps the first round of the next, rollout_streams()); the inserts follow in the reference's order.
        cur = torch.cuda.current_stream(dev)
        self.verify_images()
        fork = torch.cuda.Event(); fork.record(cur)
        s0, s1 = self.rollout_streams()
        runs = {}
        for tag, st, rows_, T, slot in (("src", s0, src_rows, cfg["src_rollout_length"], 8), ("tar", s1, tar_rows, cfg["trg_rollout_length"], 9)):
            with torch.cuda.stream(st):
                st.wait_event(fork)
                runs[tag] = self.rollout_device(rows_[:, :S].contiguous(), T, eps=inj.get(tag + "_eps"), idx=inj.get(tag + "_idx"),
                                                sync=False, ws_slot=slot, verify_images=False)                # :444, 453
        sa = None
        if cfg.get("use_src_sa_to_get_target_next_state", 1):                                         # :460-475
            with torch.cuda.stream(s1):
                n = src_rows.shape[0]
                ws = StepWorkspace(n, S, A, dev)
                eps, idx = inj.get("sa_eps"), inj.get("sa_idx")
                if eps is not None:
                    eps = _ffi.f32(eps, dev)
                if idx is not None:
                    idx = torch.as_tensor(np.asarray(idx) if not torch.is_tensor(idx) else idx).to(device=dev, dtype=torch.int64).contiguous()
                self.dynamics.launch_step(src_rows[:, :S], src_rows[:, S:S + A], ws, eps=eps, idx=idx, step=self.dynamics._draw,
                                          verify_images=False)
                self.dynamics._draw += 1
                # keep rows with penalty < env_filter (strict `<` here, `<=` in rollout(): mobody.py:468 vs :649) -- stable device
                # compaction, then one gather of the kept rows into buffer layout [s | a | s'_model | r_model | 1 - terminal]
                pos = torch.empty(n, dtype=torch.int32, device=dev)
                cnt = torch.zeros(1, dtype=torch.int32, device=dev)
                scratch = torch.empty(int(lib.mobody_compact_scratch_ints(n)), dtype=torch.int32, device=dev)
                _ffi.check(lib.mobody_compact(_ffi.KEEP_F32_LT, None, _ffi.ptr(ws.penalty), float(cfg["env_filter"]), n, None,
                                              _ffi.ptr(scratch), _ffi.ptr(pos), _ffi.ptr(cnt), _ffi.stream_ptr(dev)))
                rows = fake._pack(src_rows[:, :S], src_rows[:, S:S + A], ws.next_obs, ws.reward, ws.terminal.float(), True)
                kept = torch.empty_like(rows)
                _ffi.check(lib.mobody_gather_pos(_ffi.ptr(rows), fake.RW, fake.RW, _ffi.ptr(pos), _ffi.ptr(cnt), n, _ffi.ptr(kept), fake.RW,
                                                 _ffi.stream_ptr(dev)))
                sa = (kept, cnt, (ws, pos, scratch, rows, eps, idx))
        cur.wait_stream(s0); cur.wait_stream(s1)
        for tag in ("src", "tar"):
            out, info = runs[tag]
            if out is None:
                continue
            info["packed"].record_stream(cur)
            T = int(cfg["src_rollout_length"] if tag == "src" else cfg["trg_rollout_length"])
            host = torch.cat([info["counts_dev"].double(), info["stats_dev"]]).cpu()                  # one small read per rollout
            kept_n, produced = int(host[T + 1]), int(host[T + 3])
            if cfg.get("filter_bad_rollout", 1):
                print("filtered rollout", kept_n, produced)                                           # :653
            fake.add_rollout_slab(info["packed"], kept_n)                                             # add_batch, :445, 454
        if sa is not None:
            sa[0].record_stream(cur)
            fake.add_packed(sa[0], int(sa[1].item()))         # the host owns ptr / size (utils.py:68-92): one count read
        if cfg.get("rollout_from_src", 0):                                                            # :477-510
            if self.penalty_type != "dara":
                self.update_classifier(src_buf, tar_buf, batch_size)
            starts = torch.cat([src_buf.sample_rows(50000, inj.get("src_init2"))[:, :S],
                                tar_buf.sample_rows(100, inj.get("tar_init2"))[:, :S]], 0).contiguous()
            out, info = self.rollout_device(starts, cfg["rollout_from_src_length"], use_trg=False)   # source-dynamics heads
            if out is not None:
                if cfg.get("filter_bad_rollout", 1):
                    print("filtered rollout", info["kept"], info["num_transitions"])
                rows = self.fake_replay_buffer._pack(out["obss"], out["actions"], out["next_obss"], out["rewards"],
                                                     out["terminals"], True)
                cl = self.classifier                                                                  # :498-505 reward penalty
                sas, k0 = _ffi.mlp_params(cl.sas_classifier)
                sa, k1 = _ffi.mlp_params(cl.sa_classifier)
                _ffi.check(_ffi.lib().mobody_dara_relabel(_ffi.ptr(rows), rows.shape[0], S, A, rows.shape[1], C.byref(sas),
                                                          C.byref(sa), float(cfg["penalty_coef"]), None, _ffi.stream_ptr(self.device)))
                self.fake_replay_buffer.add_packed(rows, rows.shape[0])

    # ------------------------------------------------------------------ checkpoints
    def save(self, filename):                                    # mobody.py:584-588: the reference's four files
        torch.save(self.q_funcs.state_dict(), filename + "_critic")
        torch.save(self.q_optimizer.state_dict(), filename + "_critic_optimizer")
        torch.save(self.policy.state_dict(), filename + "_actor")
        torch.save(self.policy_optimizer.state_dict(), filename + "_actor_optimizer")

    def load(self, filename):                                    # mobody.py:590-594
        self.q_funcs.load_state_dict(torch.load(filename + "_critic"))
        self._opts["q"].load_state_dict(torch.load(filename + "_critic_optimizer"))
        self.policy.load_state_dict(torch.load(filename + "_actor"))
        self._opts["pi"].load_state_dict(torch.load(filename + "_actor_optimizer"))
        for name in ("q", "pi"):
            self._adopt_loaded_state(name)

    def _adopt_loaded_state(self, name):
        """load_state_dict replaced the optimizer's state tensors: make sure every parameter has fused-kernel-ready
        moments (a checkpoint written before the first step holds none) and adopt the step count."""
        opt = self._opts[name]
        for g in opt.param_groups:
            for prm in g["params"]:
                st = opt.state[prm]
                if "exp_avg" not in st:
                    st.update({"step": torch.tensor(0.0), "exp_avg": torch.zeros_like(prm), "exp_avg_sq": torch.zeros_like(prm)})
                st["exp_avg"], st["exp_avg_sq"] = st["exp_avg"].contiguous().float(), st["exp_avg_sq"].contiguous().float()
                if not torch.is_tensor(st["step"]):
                    st["step"] = torch.tensor(float(st["step"]))
        self._pull_steps(name)
