"""MOBODYEnsembleDynamics.step as one fused CUDA launch.

Mirror of algo/dynamics/mobody_dynamics.py:83-265 (identity StandardScaler + ``step``).  The model
fitting half of that class (``learn`` / ``validate`` / ``select_elites`` / ``train``, :300-1156) lives in
dynamics_fit.py (one C-ABI call per mini-batch).
"""
import ctypes as C
from typing import Callable, Dict, Optional, Tuple

import numpy as np
import torch

from . import _ffi
from .dynamics_fit import DynamicsFitting
from .terminal_funs import TerminationFn


class StandardScaler(object):
    """Identity scaler: the reference's transform/inverse_transform return their input
    (mobody_dynamics.py:111-131) and load_scaler ends with mu=0, std=1 (:153-154)."""

    def __init__(self, mu=None, std=None):
        self.mu, self.std = mu, std

    def transform(self, data):
        return data

    def inverse_transform(self, data):
        return data

    def transform_tensor(self, data):
        return data


    # checkpoint side files of the reference (mobody_dynamics.py:133-154): mu.npy / std.npy are written and read,
    # and the loaded values are then overwritten by mu = 0, std = 1 — i.e. an identity scaler either way
    def save_scaler(self, save_path):
        import os
        np.save(os.path.join(save_path, "mu.npy"), np.asarray(0.0 if self.mu is None else self.mu))
        np.save(os.path.join(save_path, "std.npy"), np.asarray(1.0 if self.std is None else self.std))

    def load_scaler(self, load_path):
        import os
        np.load(os.path.join(load_path, "mu.npy"), allow_pickle=True)
        np.load(os.path.join(load_path, "std.npy"), allow_pickle=True)
        self.mu, self.std = 0, 1


class StepWorkspace:
    """Output tensors of one step; torch owns the memory, the C side only fills it."""

    def __init__(self, B, S, A, device, want_act=False):
        f = dict(dtype=torch.float32, device=device)
        self.next_obs = torch.empty(B, S, **f)
        self.reward = torch.empty(B, 1, **f)
        self.raw_reward = torch.empty(B, 1, **f)
        self.penalty = torch.empty(B, 1, **f)
        self.terminal = torch.empty(B, dtype=torch.uint8, device=device)
        self.mean = torch.empty(7, B, S, **f)
        self.act = torch.empty(B, A, **f) if want_act else None


def tc_step_supports(S, A, precision):
    """Whether the tensor-core step kernels take observation / action widths (S, A) in ``precision`` (mobody_step's check)."""
    if precision == "bf16x2_wide":
        return _ffi.TC_WIDE_MIN_S <= S <= _ffi.TC_WIDE_MAX_S and 1 <= A <= _ffi.TC_WIDE_MAX_A
    if precision == "bf16x2_t64":
        return (2 <= S <= _ffi.TC_T64_MAX_S and 1 <= A <= _ffi.TC_T64_MAX_A) and not tc_step_supports(S, A, "bf16x2")
    if precision == "fp16_t64":
        return (2 <= S <= _ffi.TC_WIDE_MAX_S and 1 <= A <= _ffi.TC_WIDE_MAX_A) and not tc_step_supports(S, A, "fp16")
    return 2 <= S <= _ffi.TC_MAX_S and 1 <= A <= _ffi.TC_MAX_A and 2 * S + A <= _ffi.TC_MAX_SAS[precision]


class MOBODYEnsembleDynamics(DynamicsFitting):
    def __init__(self, config, model, optim=None, scaler=None,
                 terminal_fn: Optional[Callable] = None, penalty_coef: float = 0.0,
                 uncertainty_mode: str = "pairwise-diff", precision: Optional[str] = None, seed: int = 0) -> None:
        if uncertainty_mode != "pairwise-diff":
            # 'aleatoric' / 'ensemble_std' (mobody_dynamics.py:241-252) are unreachable from train_mobody.py
            raise NotImplementedError("mobody_b200 implements the default 'pairwise-diff' uncertainty mode")
        if not isinstance(terminal_fn, TerminationFn):
            raise TypeError("terminal_fn must come from mobody_b200.get_termination_fn (device predicate)")
        self.model, self.optim = model, optim
        self.terminal_fn = terminal_fn
        self._penalty_coef = penalty_coef
        self._uncertainty_mode = uncertainty_mode
        self.obs_scaler, self.action_scaler = StandardScaler(), StandardScaler()
        self.config = config
        self.encoder_loss_coef = config.get("encoder_loss_coef", 1) if config else 1
        self.domain_loss_coef = config.get("domain_loss_coef", 0) if config else 0
        self.cycle_loss_coef = config.get("cycle_loss_coef", 0) if config else 0
        self.encode_trg_diff = getattr(model, "encode_trg_diff", 0)
        # 'auto' (default): the tcgen05 kernel in its fp32-parity mode (bf16 hi+lo split, inside the 1e-4 bound) whenever
        # it supports the shapes, else the fp32 CUDA-core kernel (any S <= 128).  "bf16x2_wide" (S > 64),
        # "bf16x2_t64" (the S <= 64 shapes bf16x2 refuses) and "fp16_t64" (the shapes fp16 refuses) are opt-in.
        self.precision = precision or (config or {}).get("b200_precision", "auto")
        if self.precision == "auto":
            S_, A_ = getattr(model, "obs_dim", 0), getattr(model, "action_dim", 0)
            self.precision = "bf16x2" if tc_step_supports(S_, A_, "bf16x2") else "fp32"
        if self.precision not in _ffi.PREC:
            raise ValueError(f"precision {self.precision!r}: choose one of {tuple(_ffi.PREC)} (single-pass bf16 is outside "
                             "the stated error bounds and is not a product mode)")
        self.seed = int(seed)
        self._draw = 0        # Philox step counter for stand-alone step() calls in production mode
        self._packs = {}       # image slot -> (blob, device-side change-detector state) of a tensor-core weight image
        self._param_cache = {}  # (kind, id(module)) -> (parameters, data_ptrs, pointer struct, keep-alive list)

    # ------------------------------------------------------------------
    def _packed_image(self, slot, n_bytes, dev):
        """(blob, state) of a packed tensor-core weight image.  ``state`` is the library's device-side change detector
        (u64[4], zeroed once): mobody_*_pack checksums the live parameters on the device and re-packs only when they
        differ from what the image was built from, so the image follows ANY write to the parameters -- an optimiser
        step, load_state_dict, or a ``.data.copy_()`` that bumps no autograd version counter (MOBODYModule.load_save,
        mobody_module.py:407-408) -- with no host synchronisation."""
        ent = self._packs.get(slot)
        if ent is None or ent[0].numel() != n_bytes or ent[0].device != dev:
            ent = (torch.empty(n_bytes, dtype=torch.uint8, device=dev), torch.zeros(4, dtype=torch.int64, device=dev))
            if len(self._packs) >= 16:
                self._packs.pop(next(iter(self._packs)))
            self._packs[slot] = ent
        return ent

    def _packed_dynamics(self, dp, keep, verify=True):
        S, A, prec = self.model.obs_dim, self.model.action_dim, _ffi.PREC[self.precision]
        dev = keep[0].device
        blob, state = self._packed_image(("dyn", self.precision), int(_ffi.lib().mobody_dyn_pack_bytes(S, A, prec)), dev)
        if verify:
            _ffi.check(_ffi.lib().mobody_dyn_pack(C.byref(dp), S, A, prec, _ffi.ptr(blob), _ffi.ptr(state), _ffi.stream_ptr(dev)))
        return blob

    def _packed_policy(self, policy, mp, keep, verify=True):
        S, A, prec = self.model.obs_dim, self.model.action_dim, _ffi.PREC[self.precision]
        dev = keep[0].device
        blob, state = self._packed_image(("pol", id(policy), self.precision), int(_ffi.lib().mobody_mlp_pack_bytes(S, A, prec)), dev)
        if verify:
            _ffi.check(_ffi.lib().mobody_mlp_pack(C.byref(mp), S, A, prec, _ffi.ptr(blob), _ffi.ptr(state), _ffi.stream_ptr(dev)))
        return blob

    # ------------------------------------------------------------------
    def _cached_params(self, kind, module, build):
        """Pointer struct of a module's live parameters, rebuilt only when a parameter's storage moved (building it
        costs ~0.1 ms of host time for the 26 ensemble tensors; the check costs a few microseconds)."""
        ent = self._param_cache.get((kind, id(module)))
        if ent is not None:
            ent[4] += 1
            # walking the module tree costs more than everything else in a launch: the parameter list itself is re-read
            # only every 64th call (a Parameter object replaced by hand is picked up then; .to() / load_state_dict / in-place
            # optimiser steps keep the objects and are caught by the pointer comparison below on every call)
            params = ent[3] if ent[4] & 63 else list(module.parameters())
            if [p.data_ptr() for p in params] == ent[0]:
                ent[3] = params
                return ent[1], ent[2]
        struct, keep = build(module)
        params = list(module.parameters())
        self._param_cache[(kind, id(module))] = [[p.data_ptr() for p in params], struct, keep, params, 0]
        return struct, keep

    def fill_step_desc(self, d, B, S, dev, *, policy=None, max_action=1.0, use_penalty=True, use_trg=True, verify_images=True):
        """Fill the call-invariant half of a mobody_step_desc (shapes, parameter pointers, packed weight images,
        penalty/termination/elite settings).  Returns the tensors/structs that must outlive the launch.
        ``verify_images=False`` skips the device-side check / re-pack of the packed weight images: for calls that run
        CONCURRENTLY on several streams (the check is stateful), after one verified call on the stream they forked from."""
        A = self.model.action_dim
        d.precision = _ffi.PREC[self.precision]
        d.B, d.S, d.A = B, S, A
        keep = []
        tensor_core = self.precision != "fp32"
        if policy is not None:
            mp, k = self._cached_params("pol", policy, _ffi.mlp_params); keep += k; keep.append(mp)
            d.policy = C.pointer(mp)
            if tensor_core:
                d.policy_pack = _ffi.ptr(self._packed_policy(policy, mp, k, verify_images))
        d.max_action = float(max_action)
        dp, k = self._cached_params("dyn", self.model, _ffi.dyn_params); keep += k; keep.append(dp)
        d.dyn = C.pointer(dp)
        if tensor_core:
            d.dyn_pack = _ffi.ptr(self._packed_dynamics(dp, k, verify_images))
        d.use_trg, d.use_penalty = int(bool(use_trg)), int(bool(use_penalty))
        d.penalty_coef = float(self._penalty_coef)
        d.term_kind = self.terminal_fn.kind
        elites = self.model.elites.data
        if elites.dtype != torch.int64 or not elites.is_cuda:
            elites = elites.to(device=dev, dtype=torch.int64)
        keep.append(elites)
        d.elites, d.n_elites = _ffi.ptr(elites), elites.numel()
        d.seed = self.seed
        return keep

    def launch_step(self, obs, act, ws: StepWorkspace, *, policy=None, max_action=1.0, use_penalty=True,
                    use_trg=True, eps=None, idx=None, n_rows_dev=None, row_ids=None, step=0, row0=0, verify_images=True):
        """Enqueue the fused step on the current stream; no host synchronisation.
        obs [B,S] (B = capacity), act [B,A] or None with ``policy`` (an MLPNetwork-like module).  obs / act may be
        column views of wider rows (e.g. the state / action columns of packed replay-buffer rows): the row stride is
        passed to the kernel, nothing is copied."""
        dev = obs.device
        B, S = obs.shape
        A = self.model.action_dim
        for t in (obs, act):
            if t is not None and (t.dtype != torch.float32 or not t.is_cuda or (t.shape[0] > 1 and t.stride(1) != 1) or t.shape[1] < 1):
                raise RuntimeError("mobody_b200: step inputs must be fp32 CUDA tensors with unit column stride")
        d = _ffi.StepDesc()
        keep = self.fill_step_desc(d, B, S, dev, policy=policy, max_action=max_action, use_penalty=use_penalty, use_trg=use_trg,  # noqa: F841
                                   verify_images=verify_images)
        if policy is not None and ws.act is None:
            ws.act = torch.empty(B, A, dtype=torch.float32, device=dev)
        d.n_rows_dev, d.row_ids = _ffi.ptr(n_rows_dev), _ffi.ptr(row_ids)
        d.obs, d.act = obs.data_ptr(), (None if act is None else act.data_ptr())
        d.obs_ld = obs.stride(0) if B > 1 else S
        d.act_ld = (act.stride(0) if B > 1 else A) if act is not None else A
        d.eps, d.idx = _ffi.ptr(eps), _ffi.ptr(idx)
        d.step, d.row0 = int(step), int(row0)
        d.act_out = _ffi.ptr(ws.act)
        d.next_obs, d.reward, d.raw_reward = _ffi.ptr(ws.next_obs), _ffi.ptr(ws.reward), _ffi.ptr(ws.raw_reward)
        d.penalty, d.terminal, d.mean = _ffi.ptr(ws.penalty), _ffi.ptr(ws.terminal), _ffi.ptr(ws.mean)
        _ffi.check(_ffi.lib().mobody_step(C.byref(d), _ffi.stream_ptr(dev)))
        return ws

    # ------------------------------------------------------------------ checkpoints (mobody_dynamics.py:1158-1166)
    def save(self, save_path: str) -> None:
        import os
        torch.save(self.model.state_dict(), os.path.join(save_path, "dynamics.pth"))
        self.obs_scaler.save_scaler(save_path)

    def load(self, load_path: str) -> None:
        import os
        self.model.load_state_dict(torch.load(os.path.join(load_path, "dynamics.pth"), map_location=self.model.elites.device))
        self.obs_scaler.load_scaler(load_path)                   # (the packed tensor-core image follows by checksum)

    @torch.no_grad()
    def step(self, obs, action, use_penalty=True, use_trg=True, *, eps=None, idx=None
             ) -> Tuple[torch.Tensor, torch.Tensor, np.ndarray, Dict]:
        """Reference signature (mobody_dynamics.py:193-265):
        -> (next_obs Tensor[B,S], reward Tensor[B,1], terminal np.bool_[B,1] on host, info).
        ``eps`` [7,B,S] / ``idx`` [B] inject the noise and member indices the reference would draw
        from torch.normal / np.random.choice; when omitted they come from Philox (seed, draw)."""
        self.model.inference()
        dev = self.model.elites.device
        obs = _ffi.f32(obs, dev)
        action = _ffi.f32(action, dev).reshape(obs.shape[0], self.model.action_dim)
        B, S = obs.shape
        if eps is not None:
            eps = _ffi.f32(eps, dev)
            assert tuple(eps.shape) == (7, B, S)
        if idx is not None:
            idx = torch.as_tensor(np.asarray(idx) if not torch.is_tensor(idx) else idx).to(device=dev, dtype=torch.int64).contiguous()
        ws = StepWorkspace(B, S, action.shape[1], dev)
        if B > 0:
            self.launch_step(obs, action, ws, use_penalty=use_penalty, use_trg=use_trg, eps=eps, idx=idx, step=self._draw)
        self._draw += 1
        info = {"samples": ws.mean, "raw_reward": ws.raw_reward, "penalty": ws.penalty}
        terminal = ws.terminal.bool()[:, None].cpu().numpy()      # the one D2H the reference API demands (:237)
        return ws.next_obs, ws.reward, terminal, info
