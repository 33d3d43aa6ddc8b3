#!/usr/bin/env python
"""Benchmark of the MOBODY model-rollout hot path (BASELINE.json metric: model-rollout transitions/sec).

Workload at N=1: BASELINE.json configs[1] — halfcheetah-gravity shaped (obs 17 / act 6), 100 000 start
states, rollout_length=1, 7-member ensemble, policy forward fused in.  At N>1 every rank rolls its own
100 000 start states (weak scaling) and the pack stage of each rank's rollout pushes its transitions into
every rank's receive buffer over peer memory (csrc/peer.cu; NCCL padded all-gather as the fallback).  The
same run also reports a STRONG-scaling arm (BASELINE configs[2]: hopper, 1 000 000 start states,
rollout_length=5, split over the N ranks) and, at N=1, one line per BASELINE config with its termination rate.
Before the timed region every N>1 run verifies the exchange: the gathered transitions of a 10 007-row problem
must equal, bit for bit, the single-GPU result (parallel.self_check) — reported as `exchange_check`.

One "step" = one full rollout of the start states (policy + 7-member dynamics + reward ensemble +
penalty + termination + penalty filter), exactly what MOBODY.rollout does per refresh.

  value   : transitions/s with the start states already in HBM (CUDA events around each rollout,
            inputs rotate over a pool of buffers larger than L2, max over ranks)
  e2e     : the same through the public API MOBODY.rollout() with HOST buffers: pinned-host -> device
            copy of the start states and device -> host copy of the returned transition dict inside
            the timed region
  roofline: tensor-core roofline of the fused step kernel (algorithmic FLOP / measured kernel time) in the headline
            fp32-parity mode (bf16 hi+lo split); the single-pass fp16 / bf16 modes (looser stated bounds) are timed too
  cpu_baseline: the oracle (CPU restatement of the reference, torch CPU) timed on this box's host cores

`--impl reference` times the reference's CPU path (oracle port; the reference is Python and does not
travel to the GPU box) with all host threads on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the source tree as it found it (it may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

S, A, B_PER_GPU, T = 17, 6, 100_000, 1
ENV, TASK, COEF, ENV_FILTER = "halfcheetah", "halfcheetah-medium-v2", 5.0, 10.0
METRIC, UNIT = "model-rollout transitions/sec", "transitions/s"


def flop_per_transition(S, A, H=256, E=7):
    """SURVEY.md §8d: 2*[E*(dyn+rew)+policy] with dead columns counted (not credited as skipped)."""
    dyn = S * H + H * H + 32 * H + (16 + A) * 32 + 32 * 32 + 16 * H + H * H + H * S
    rew = (2 * S + A) * H + H * H + 2 * H
    pol = S * H + H * H + H * A
    return 2 * (E * (dyn + rew) + pol)


def synth_obs(n, seed):
    rng = np.random.default_rng(seed)
    return (0.3 * rng.standard_normal((n, S))).astype(np.float32)   # halfcheetah healthy set: |x| < 100


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons sampled DURING the timed regions (NVML every 5 ms; nvidia-smi as a fallback)."""
    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.sm, self.mx, self.reasons, self._halt, self.n = gpu, [], [], set(), threading.Event(), 0
        self.period = 0.005         # seconds between samples
        self.nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _nvml(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4)):
            if r & bit:
                self.reasons.add(name)

    def _smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        r = [x.strip() for x in out.split(",")]
        self.sm.append(float(r[0])); self.mx.append(float(r[1]))
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if r[2 + i].lower().startswith("active"):
                self.reasons.add(name)

    def run(self):
        while not self._halt.is_set():
            try:
                self._nvml() if self.nv else self._smi()
                self.n += 1
            except Exception:
                pass
            self._halt.wait(self.period if self.nv else max(self.period, 0.1))

    def stop(self):
        self._halt.set(); self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                "reasons": sorted(self.reasons), "samples": self.n, "source": "nvml" if self.nv else "nvidia-smi"}


AGENT_CFG = dict(max_action=1.0, hidden_sizes=256, gamma=0.99, tau=0.005, update_interval=2, actor_lr=3e-4, critic_lr=3e-4,
                 gaussian_noise_std=1.0, weight=2.5, penalty_type="none", penalty_coef=0.1, mopo=0, latent_reward=0, advantage=0,
                 q_weighted=1, scale_Q=1, bc_coef=1.0, fake_batch_scale=0.5, src_ratio=1, trg_ratio=1, filter_bad_rollout=1,
                 env_filter=ENV_FILTER, src_rollout_length=1, trg_rollout_length=1, use_src_sa_to_get_target_next_state=1,
                 rollout_from_src=0)


def build_dynamics(mb, s_dim, a_dim, precision, dev, seed=1):
    """Random-init ensemble of the reference architecture (MOBODYModule's own initialiser) behind the product API.
    The GPU arm never touches oracle/: that package is test infrastructure (CPU-baseline legs only)."""
    torch.manual_seed(seed)
    model = mb.MOBODYModule(s_dim, a_dim, 256, 7, 5, device=dev, config={"mopo": 0, "latent_reward": 0})
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if name.endswith(".bias"):
                prm.normal_(0.0, 0.1)                 # biases randomised so they matter (the reference zero-initialises them)
    return mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, model, None, None,
                                     mb.get_termination_fn(TASK), penalty_coef=COEF, precision=precision)


def build_config_dynamics(mb, env, s_dim, a_dim, dev, h0, gain, coef=1.0, precision="bf16x2", seed=3):
    """Random-init ensemble (the reference module's own initialiser) whose decoder bias sits in the env's healthy set and
    whose decoder weights are scaled so that a real share of the rows terminates at every step (SURVEY 8d recipe)."""
    torch.manual_seed(seed)
    model = mb.MOBODYModule(s_dim, a_dim, 256, 7, 5, device=dev, config={"mopo": 0, "latent_reward": 0})
    with torch.no_grad():
        for name, prm in model.named_parameters():
            if name.endswith(".bias"):
                prm.normal_(0.0, 0.1)
        model.transition3.weight.mul_(gain)
        model.transition3.bias.mul_(0.1)
        model.transition3.bias[:, :, 0] += h0
    task = {"hopper": "hopper-medium-v2", "ant": "ant-medium-v2", "walker2d": "walker2d-medium-v2", "halfcheetah": "halfcheetah-medium-v2"}[env]
    return mb.MOBODYEnsembleDynamics({"encoder_loss_coef": 1, "domain_loss_coef": 0, "cycle_loss_coef": 0}, model, None, None,
                                     mb.get_termination_fn(task), penalty_coef=coef, precision=precision)


def config_obs(env, n, s_dim, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    x = 0.2 * torch.randn(n, s_dim, generator=g, device=dev)
    x[:, 0] += {"hopper": 1.25, "walker2d": 1.25, "ant": 0.6, "halfcheetah": 0.0}[env]
    return x


def timed_rollouts(fn, reps):
    """CUDA-event time of ``reps`` calls of ``fn`` (after one warm-up call) in seconds per call."""
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3 / reps


def baseline_config_lines(mb, dev):
    """One entry per BASELINE.json config at its size (single GPU): transitions/s of the whole rollout (device timed), the
    live rows entering every step and the share of rows that terminated -- compaction on shrinking batches is timed, not
    assumed away."""
    out = {}
    cases = [("C1 walker2d-friction S17/A6 50k+2k starts T=1", "walker2d", 17, 6, [52_000], [1], 1.0, 4.0, 5.0),
             ("C3 hopper-kinematic S11/A3 1M starts T=5", "hopper", 11, 3, [1_000_000], [5], 0.8, 4.0, 1.0),
             ("C4 ant-friction S27/A8 50k starts T=5", "ant", 27, 8, [50_000], [5], 0.4, 4.0, 1.0),
             ("C5 antmaze-umaze-style S29/A8 sweep", "ant", 29, 8, [10_000, 100_000, 1_000_000, 4_000_000], [1, 5], 0.35, 6.0, 1.0),
             # observations wider than the tensor-core kernel's 64 (Ant-v3's 111 dims): the fp32 CUDA-core step kernel
             ("wide observations S111/A8 (Ant-v3) 100k starts T=1, fp32 CUDA-core step kernel", "ant", 111, 8, [100_000], [1], 0.6, 4.0, 1.0)]
    for name, env, sd, ad, sizes, Ts, h0, gain, coef in cases:
        dyn = build_config_dynamics(mb, env, sd, ad, dev, h0, gain, coef, precision="bf16x2" if sd <= 64 else "fp32")
        ag = build_agent(mb, sd, ad, dev, env_filter=1e9)
        ag.dynamics = dyn
        rows = []
        for n in sizes:
            obs = config_obs(env, n, sd, n, dev)
            for T_ in Ts:
                _, info = ag.rollout_device(obs, T_)
                per = timed_rollouts(lambda: ag.rollout_device(obs, T_, sync=False), 3 if n * T_ >= 1_000_000 else 10)
                cnt = info["rows_per_step"]
                term = [round(1.0 - cnt[t + 1] / max(cnt[t], 1), 4) for t in range(len(cnt) - 1)]
                rows.append({"start_states": n, "rollout_length": T_, "transitions": info["num_transitions"], "ms": per * 1e3,
                             "transitions_per_s": info["num_transitions"] / per, "rows_per_step": cnt, "terminated_share_per_step": term})
                ag._roll_ws.clear()
            del obs
        out[name] = rows if len(rows) > 1 else rows[0]
        del ag, dyn
        torch.cuda.empty_cache()
    return out


def step_kernel_traffic():
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the step kernel from an `ncu --set full`
    capture of this bench command (profiles/step_kernel_traffic.json, written by scripts/ncu_traffic.py).  The record names
    the sha256 of the kernel sources it was captured from; if the sources changed since, the number is stale -> None."""
    import hashlib
    try:
        with open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json")) as f:
            rec = json.load(f)
        h = hashlib.sha256()
        csrc = os.path.join(ROOT, "mobody-model-based-off-dynamics-offline-reinforcement-learning_b200", "csrc")
        for fn in rec["sources"]:
            with open(os.path.join(csrc, fn), "rb") as f:
                h.update(f.read())
        if h.hexdigest() != rec["sources_sha256"]:
            return None, "stale (kernel sources changed since the ncu capture)"
        return int(rec["dram_bytes_read"]) + int(rec["dram_bytes_write"]), rec.get("capture", "profiles/")
    except Exception:
        return None, "no ncu capture on record"


def build_agent(mb, s_dim, a_dim, dev, seed=1, **overrides):
    torch.manual_seed(seed + 100)
    cfg = dict(AGENT_CFG, state_dim=s_dim, action_dim=a_dim); cfg.update(overrides)
    return mb.MOBODY(cfg, dev)


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_rollout_rate(n_rows, threads, repeats=1):
    """Oracle (CPU restatement of MOBODY.rollout, proven equal to the reference) on host cores."""
    from oracle import mobody_oracle as M
    torch.set_num_threads(threads)
    p = M.make_dynamics_params(S, A, 1)
    ag = M.AgentState(S, A, 1)
    obs = torch.from_numpy(synth_obs(n_rows, 0))
    g = torch.Generator().manual_seed(0)
    elites = p["elites"].numpy()
    best = None
    for _ in range(repeats + 1):            # first pass is warm-up
        t0 = time.perf_counter()
        eps = [lambda n: torch.randn(7, n, S, generator=g)]
        idx = [lambda n: elites[np.random.randint(0, len(elites), n)]]
        _, info = M.rollout(p, ag.policy, 1.0, obs, T, eps, idx, M.termination_kind(TASK), COEF, ENV_FILTER, True)
        dt = time.perf_counter() - t0
        best = dt if best is None or _ == 0 else min(best, dt)
        if _ == 0:
            best = None
    return info["num_transitions"] / best, best


def synth_buffer_dict(n, seed, s_dim=None, a_dim=None):
    s_dim, a_dim = s_dim or S, a_dim or A
    rng = np.random.default_rng(seed)
    obs = lambda sd: (0.3 * np.random.default_rng(sd).standard_normal((n, s_dim))).astype(np.float32)   # noqa: E731
    return dict(observations=obs(seed), actions=rng.uniform(-1, 1, (n, a_dim)).astype(np.float32),
                next_observations=obs(seed + 1), rewards=rng.standard_normal(n).astype(np.float32),
                terminals=np.zeros(n, bool))


def cpu_train_rate(batch, threads, steps=5):
    """Oracle steady-state MOBODY.train step (3 buffer gathers + critic + Polyak + actor) on host cores."""
    from oracle import mobody_oracle as M
    torch.set_num_threads(threads)
    ag = M.AgentState(S, A, 1)
    bufs = []
    for n, sd in ((200_000, 1), (20_000, 2), (50_000, 3)):
        d = synth_buffer_dict(n, sd)
        b = M.RingBuffer(S, A, n)
        b.state[:] = torch.from_numpy(d["observations"]); b.action[:] = torch.from_numpy(d["actions"])
        b.next_state[:] = torch.from_numpy(d["next_observations"]); b.reward[:, 0] = torch.from_numpy(d["rewards"]); b.not_done[:] = 1.0
        b.size = n; bufs.append(b)
    cfg = dict(gamma=0.99, tau=0.005, actor_lr=3e-4, critic_lr=3e-4, weight=2.5, bc_coef=1.0, max_action=1.0)
    ns = (batch, batch, batch // 2)
    t0 = None
    for it in range(steps + 2):
        if it == 2:
            t0 = time.perf_counter()
        parts = [b.gather(np.random.randint(0, b.size, n)) for b, n in zip(bufs, ns)]
        M.train_step(ag, tuple(torch.cat([p[c] for p in parts], 0) for c in range(5)), 2 * batch, cfg)
    return steps / (time.perf_counter() - t0)


def gpu_train_rate(mb, dev, batch, steps=300, s_dim=None, a_dim=None, penalty_type="none", dynamics=None):
    """MOBODY.train steady state through the public API: device-resident buffers, Philox indices, fused step."""
    s_dim, a_dim = s_dim or S, a_dim or A
    ag = build_agent(mb, s_dim, a_dim, dev, seed=2, penalty_type=penalty_type)
    ag.dynamics = dynamics
    src, tar = mb.ReplayBuffer(s_dim, a_dim, dev), mb.ReplayBuffer(s_dim, a_dim, dev)
    src.convert_D4RL(synth_buffer_dict(200_000, 1, s_dim, a_dim)); tar.convert_D4RL(synth_buffer_dict(20_000, 2, s_dim, a_dim))
    ag.fake_replay_buffer.convert_D4RL(synth_buffer_dict(50_000, 3, s_dim, a_dim))
    ag.total_it = 1                               # steady state: the 5000-step refresh is measured by the rollout metric
    for _ in range(20):
        ag.train(src, tar, batch)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        ag.train(src, tar, batch)
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return steps / (e0.elapsed_time(e1) * 1e-3), steps / wall


def fit_batch_data(B, seed=5):
    rng = np.random.default_rng(seed)
    s = (0.3 * rng.standard_normal((7, B, S))).astype(np.float32)
    return [s, rng.uniform(-1, 1, (7, B, A)).astype(np.float32), (s + 0.1 * rng.standard_normal((7, B, S))).astype(np.float32),
            rng.standard_normal((7, B, 1)).astype(np.float32)]


def gpu_fit_rate(mb, dev, dyn, B=256, n_batches=40, epochs=5):
    """Dynamics fitting (MOBODYEnsembleDynamics.learn, 7 x B rows per mini-batch): optimiser steps/s through learn() on
    device-resident epoch tensors (one scalar read-back per learn() call)."""
    data = [torch.from_numpy(np.concatenate([x] * n_batches, 1)).to(dev) for x in fit_batch_data(B)]
    dyn.learn(True, *data, B, 0.01)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter(); e0.record()
    for _ in range(epochs):
        dyn.learn(True, *data, B, 0.01)
    e1.record(); torch.cuda.synchronize()
    return epochs * n_batches / (e0.elapsed_time(e1) * 1e-3), epochs * n_batches / (time.perf_counter() - t0)


def cpu_fit_rate(threads, B=256, steps=3):
    """Oracle fitting step (autograd restatement of learn(), proven equal to the reference) on host cores."""
    from oracle import mobody_oracle as M
    torch.set_num_threads(threads)
    p = M.make_dynamics_params(S, A, 1)
    names = [n + sfx for n in M.fit_trained_layers(True) for sfx in (".weight", ".bias")]
    m = {k: torch.zeros_like(p[k]) for k in names}; v = {k: torch.zeros_like(p[k]) for k in names}
    data = [torch.from_numpy(x) for x in fit_batch_data(B)]
    t0 = None
    for it in range(steps + 1):
        if it == 1:
            t0 = time.perf_counter()
        M.fit_step(p, m, v, {n: it + 1 for n in M.fit_trained_layers(True)}, *data, torch.randn(6, 7, B, 16), torch.randn(7, B, S), True)
    return steps / (time.perf_counter() - t0)


def hbm_stage_rates(mb, dev, hbm_peak, n=2_000_000):
    """Achieved HBM GB/s of the byte-moving stages of the path at a size well beyond L2 (2 M rows x 176 B): replay-buffer
    sampling (Philox draw + random row gather), ring insert, and the row packing of convert_D4RL / add_batch."""
    from mobody_b200 import _ffi
    buf = mb.ReplayBuffer(S, A, dev, max_size=n)
    buf.size = n
    RW, lib, st = buf.RW, _ffi.lib(), _ffi.stream_ptr(dev)
    out = torch.empty(n, RW, dtype=torch.float32, device=dev)
    cols = [torch.randn(n, w, device=dev) for w in (S, A, S)] + [torch.randn(n, device=dev), torch.zeros(n, device=dev)]

    def timed(fn, reps=5):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps * 1e-3
    row_bytes = RW * 4
    res = {}
    t = timed(lambda: buf.sample_rows(n, out=out))
    res["sample_rows (Philox draw + random gather)"] = (n * (2 * row_bytes + 16)) / t / 1e9      # rows read + written, int64 index written + read
    t = timed(lambda: buf.add_packed(out, n))
    res["ring_insert"] = (n * 2 * row_bytes) / t / 1e9
    t = timed(lambda: _ffi.check(lib.mobody_pack_rows(*[_ffi.ptr(c) for c in cols], n, S, A, 1, _ffi.ptr(out), st)))
    res["pack_rows"] = (n * ((2 * S + A + 2) * 4 + row_bytes)) / t / 1e9
    return {k: {"GB/s": round(v, 1), "frac_of_hbm_peak": round(v / hbm_peak, 3)} for k, v in res.items()}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, out, info):
    """Write what the last timed rollout returned as ``out_dir/<name>.npy``: the kept transitions (the dict MOBODY.rollout
    hands its caller, float32) and the info scalars (float64).  The inputs are seeded, so two builds run with the same
    arguments can be compared file for file.  Transitions above DUMP_BYTES are replaced by a fixed, seeded sample of rows
    (``row_index.npy`` holds their positions)."""
    os.makedirs(out_dir, exist_ok=True)
    M = int(info["kept_dev"].item())
    counts, stats = info["counts_dev"].cpu().numpy(), info["stats_dev"].cpu().numpy()
    rows = {k: v[:M] for k, v in out.items()}
    row_bytes = sum(v.shape[1] for v in rows.values()) * 4
    budget = DUMP_BYTES - (1 << 20)                  # headroom for the info arrays and the .npy headers
    if M * row_bytes > budget:
        idx = np.sort(np.random.default_rng(0).choice(M, budget // (row_bytes + 8), replace=False))
        sel = torch.from_numpy(idx).to(next(iter(rows.values())).device)
        rows = {k: v[sel] for k, v in rows.items()}
        np.save(os.path.join(out_dir, "row_index.npy"), idx.astype(np.float64))
    for k, v in rows.items():
        np.save(os.path.join(out_dir, k + ".npy"), v.cpu().numpy().astype(np.float32))
    T = len(counts) - 2
    np.save(os.path.join(out_dir, "rows_per_step.npy"), counts[:T].astype(np.float64))
    np.save(os.path.join(out_dir, "num_transitions.npy"), np.float64(stats[1]))
    np.save(os.path.join(out_dir, "reward_mean.npy"), np.float64(stats[0] / max(stats[1], 1.0)))


def run_reference(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    n = B_PER_GPU                            # one full rollout of the workload per step: ~1.3 s on 16 cores
    rate, dt = cpu_rollout_rate(n, cores, repeats=max(args.steps, 1))   # includes one warm-up pass
    val = rate
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"halfcheetah-gravity S{S}/A{A} rollout_length={T}, {B_PER_GPU} start states (BASELINE configs[1])",
                       "sample": f"{n} of {B_PER_GPU} start states per step (the full workload)"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"oracle.rollout on {n} start states, best of {max(args.steps, 1)} after 1 warm-up, torch threads={cores}"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def strong_scaling_arm(mb, P, dev, dist, rank, world, steps):
    """BASELINE configs[2]: hopper-kinematic, 1 000 000 start states, rollout_length 5, split over the ranks (strong scaling:
    total work fixed).  Device-timed, max over ranks; transitions = what all ranks produced."""
    env, sd, ad, total, T_ = "hopper", 11, 3, 1_000_000, 5
    dyn = build_config_dynamics(mb, env, sd, ad, dev, 0.8, 4.0, 1.0)
    ag = build_agent(mb, sd, ad, dev, env_filter=1e9)
    ag.dynamics = dyn
    lo, hi = P.shard_range(total, rank, world)
    obs = config_obs(env, total, sd, 99, dev)[lo:hi].contiguous()          # same global states on every rank, this rank's range
    produced = torch.zeros(1, dtype=torch.float64, device=dev)
    pend = []

    def one():
        if dist is None:
            _, info = ag.rollout_device(obs, T_, row0=lo, sync=False)
            produced.add_(info["stats_dev"][1:2])
        else:
            h = P.p2p_rollout(ag, obs, T_, True, lo, P.shard_range(total, 0, world)[1] * T_)
            produced.add_(h.info["stats_dev"][1:2])
            pend.append(h)
            if len(pend) > 1:
                pend.pop(0).wait()
    for _ in range(2):
        one()
    while pend:
        pend.pop(0).wait()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    produced.zero_()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        one()
    while pend:
        pend.pop(0).wait()
    e1.record(); torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1), float(produced.item())], dtype=torch.float64, device=dev)
    if dist is not None:
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        ms, n = float(mx[0]), float(sm[1])
    else:
        ms, n = float(t[0]), float(t[1])
    return {"scaling": "strong", "workload": f"hopper-kinematic S{sd}/A{ad} rollout_length={T_}, {total} start states split over {world} GPU(s) (BASELINE configs[2])",
            "value": n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps, "steps": steps, "transitions_per_step": n / steps,
            "start_states_per_gpu": hi - lo}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("MOBODY_PRECISION", "auto"))
    ap.add_argument("--rows", type=int, default=B_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the updates/sec measurement (short ncu runs)")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-config lines and the strong-scaling arm (short ncu runs)")
    ap.add_argument("--exchange", default=os.environ.get("MOBODY_EXCHANGE", "p2p"), choices=["p2p", "nccl"],
                    help="N>1: peer-memory push (default) or the NCCL padded all-gather")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the transitions of the last timed rollout as DIR/<name>.npy (single GPU)")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and world > 1:
        ap.error("--dump-outputs writes a single-GPU rollout: run it without torchrun")
    if args.impl == "reference":
        return run_reference(args, rank)
    W = max(args.warmup, 3)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as G
    if rank == 0 or not os.path.exists(os.path.join(G.PKG, "libmobody_b200.so")):
        G.build()
    if dist is not None:
        dist.barrier()
    import mobody_b200 as mb
    from mobody_b200 import _ffi, parallel as P
    enabled = list(getattr(_ffi, "ENABLED_PRECISIONS", ("fp32",)))
    prec = args.precision if args.precision != "auto" else ("bf16x2" if "bf16x2" in enabled else "fp32")
    dyn = build_dynamics(mb, S, A, prec, dev)
    ag = build_agent(mb, S, A, dev)
    ag.dynamics = dyn
    Bn = args.rows
    obs_host = torch.from_numpy(synth_obs(Bn, 100 + rank)).pin_memory()
    obs_dev = obs_host.to(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2 (kernel-only timings)
    # whole-rollout timing: the start states rotate over a pool of distinct buffers larger than L2, so every rollout reads
    # its inputs from HBM (the 6.5 MB weight image is L2 resident by design: all 782 CTAs of a launch share it)
    n_pool = max(2, -(-160 * 1024 * 1024 // (Bn * S * 4)))
    obs_pool = [obs_dev] + [obs_dev.clone() for _ in range(n_pool - 1)]
    pool_i = [0]

    # ---- N > 1: prove the exchange before timing it (gathered transitions == the single-GPU result, bit for bit) ----
    exchange, check = "none", None
    if dist is not None:
        exchange = args.exchange
        try:
            check = P.self_check(ag, 10_007, rounds=4)
            if exchange == "p2p" and not check["p2p"]:
                exchange = "nccl"                                  # fall back, and say so in the line
        except Exception as e:                                     # noqa: BLE001
            check = {"ok": False, "error": repr(e)}
            exchange = "nccl"
    if os.environ.get("MOBODY_PROBE_LATE"):        # timing experiments only (parallel.p2p_rollout): takes effect after the self-check
        os.environ["MOBODY_PROBE"] = os.environ["MOBODY_PROBE_LATE"]
    pending = []

    def wait_on_own_stream(h):
        # a p2p handle is waited for on the stream its rollout ran on: the ack of epoch e - 2 (enqueued with rollout e on
        # that same stream) is then ordered after it
        if isinstance(h, tuple):
            with torch.cuda.stream(h[1]):
                h[0].wait()
        else:
            h.wait()

    def drain():
        while pending:
            wait_on_own_stream(pending.pop(0))

    produced = torch.zeros(1, dtype=torch.float64, device=dev)   # transitions produced by this rank (device accumulator)
    # Consecutive rollouts are independent, so they alternate between the agent's two rollout streams (own workspace
    # each): the last, 72 %-idle round of one step kernel (782 tiles on 148 SMs) runs beside the first round of the next.
    # N > 1 (peer-memory exchange): epoch parity = stream, see parallel.p2p_rollout.
    two_streams = (dist is None or exchange == "p2p") and os.environ.get("MOBODY_BENCH_STREAMS", "2") != "1"
    side = ag.rollout_streams() if two_streams else None
    produced_side = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(2)]
    last_handle = [None]
    last_rollout = [None]   # N = 1: (transitions dict, info) of the latest rollout, for --dump-outputs
    last_epoch = [None]     # (epoch parity) xor (stream index) of the first two-stream exchange: constant afterwards

    def fork_streams():
        if side:
            ag.verify_images()
            for st in side:
                st.wait_stream(torch.cuda.current_stream(dev))

    def join_streams():
        if side:
            for st in side:
                torch.cuda.current_stream(dev).wait_stream(st)
            produced.add_(produced_side[0]).add_(produced_side[1])
            produced_side[0].zero_(); produced_side[1].zero_()

    def one_rollout_device():
        """One rollout with nothing read back by the host (counts stay on the device; read once after the timed region)."""
        i = pool_i[0]
        x = obs_pool[i % n_pool]; pool_i[0] += 1
        if side and dist is None:
            with torch.cuda.stream(side[i & 1]):
                o, info = ag.rollout_device(x, T, row0=rank * Bn, sync=False, ws_slot=10 + (i & 1), verify_images=False)
                produced_side[i & 1].add_(info["stats_dev"][1:2])
                last_rollout[0] = o, info
            return
        if side:
            st = side[i & 1]
            with torch.cuda.stream(st):
                h = P.sharded_rollout(ag, x, T, sharded_input=True, gather="p2p", verify_images=False)
                if last_epoch[0] is None:
                    last_epoch[0] = (h.epoch ^ i) & 1
                assert ((h.epoch ^ i) & 1) == last_epoch[0], "exchange epoch parity and stream fell out of step"
                produced_side[i & 1].add_(h.info["stats_dev"][1:2])
            last_handle[0] = h
            pending.append((h, st))
            if len(pending) > 1:
                wait_on_own_stream(pending.pop(0))
            return
        if dist is None:
            o, info = ag.rollout_device(x, T, row0=rank * Bn, sync=False)
            last_rollout[0] = o, info
        elif exchange == "p2p":
            # shard = this rank's start states; the pack stage pushes the kept transitions into every rank's receive buffer
            h = P.sharded_rollout(ag, x, T, sharded_input=True, gather="p2p")
            info = h.info
            pending.append(h)
            if len(pending) > 1:
                pending.pop(0).wait()                     # the exchange of step t-1 overlapped this step's rollout
        else:
            (o, counts_dev, widths, work), info = P.sharded_rollout(ag, x, T, sharded_input=True, gather="padded_async")
            pending.append(work)
            if len(pending) > 1:
                pending.pop(0).wait()
        produced.add_(info["stats_dev"][1:2])

    # ---- device-resident timing ----
    fork_streams()
    for _ in range(W):
        one_rollout_device()
    drain()
    join_streams()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    torch.cuda.synchronize()
    produced.zero_()
    wall0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fork_streams()
    for _ in range(args.steps):
        one_rollout_device()
    drain()                                               # every rank's rows of every step have landed before the closing event
    join_streams()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    wall = time.perf_counter() - wall0
    dev_ms = e0.elapsed_time(e1)
    n_trans = float(produced.item())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *last_rollout[0])
    last_rollout[0] = None
    if last_handle[0] is not None and check is not None and not os.environ.get("MOBODY_PROBE"):
        # the last timed step, as every rank received it: the headers in MY receive buffer must add up to what the ranks
        # say they produced (device counters, all-reduced) -- the two-stream pipeline delivered complete results
        h = last_handle[0]
        kept_r, produced_all, _ = h.counts()
        mine = torch.stack([h.info["stats_dev"][1], h.info["kept_dev"][0].double()])
        dist.all_reduce(mine)
        check["timed_last_step"] = {"produced": produced_all, "kept": int(sum(kept_r)),
                                    "ok": bool(int(mine[0].item()) == produced_all and int(mine[1].item()) == sum(kept_r))}

    # ---- step-kernel-only timing for the roofline (same stream, events directly around the launch) ----
    from mobody_b200.dynamics import StepWorkspace
    ws = StepWorkspace(Bn, S, A, dev, want_act=True)
    dyn.launch_step(obs_dev, None, ws, policy=ag.policy.network, max_action=1.0, step=0, row0=rank * Bn)   # (packs the weight images)
    kt = []
    for it in range(W + args.steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d = _ffi.StepDesc()
        keep = dyn.fill_step_desc(d, Bn, S, dev, policy=ag.policy.network, max_action=1.0)     # noqa: F841 (image checksum passes run here, outside the events)
        d.obs, d.step, d.row0, d.act_out = _ffi.ptr(obs_dev), it, rank * Bn, _ffi.ptr(ws.act)
        d.next_obs, d.reward, d.raw_reward = _ffi.ptr(ws.next_obs), _ffi.ptr(ws.reward), _ffi.ptr(ws.raw_reward)
        d.penalty, d.terminal, d.mean = _ffi.ptr(ws.penalty), _ffi.ptr(ws.terminal), _ffi.ptr(ws.mean)
        e0.record()
        _ffi.check(_ffi.lib().mobody_step(d, _ffi.stream_ptr(dev)))
        e1.record()
        kt.append((e0, e1))
    torch.cuda.synchronize()
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in kt[W:]]))

    # ---- end-to-end through the public API with host buffers ----
    sampler.period = 0.02
    def one_rollout_e2e():
        import contextlib, io
        with contextlib.redirect_stdout(io.StringIO()):
            if dist is None:
                return ag.rollout(obs_host, T)      # pinned HOST start states in, CPU tensors out (H2D + D2H inside)
            # N > 1: this rank's shard from HOST memory in, the transitions of ALL ranks out as CPU tensors (H2D + rollout +
            # peer-memory exchange + D2H of the gathered rows inside)
            return P.sharded_rollout_host(ag, obs_host, T) if exchange == "p2p" else e2e_nccl()

    def e2e_nccl():
        x = obs_host.to(dev, non_blocking=True)
        out, info = P.sharded_rollout(ag, x, T, sharded_input=True, gather=True)
        return {k: v.cpu() for k, v in out.items()}, info
    for _ in range(3):                 # held like the timed loop holds them: both pinned result slabs exist before timing
        tr, info = one_rollout_e2e()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter(); e2e_trans = 0; d2h = 0
    for _ in range(args.steps):
        tr, info = one_rollout_e2e(); e2e_trans += info["num_transitions"]
        d2h = sum(v.numel() * v.element_size() for v in tr.values())
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
        d2h *= world if exchange == "p2p" else 1      # whole-job bytes: every rank copies its own shard
    e2e_s = time.perf_counter() - t0           # (at N > 1 every rank's info already counts the whole job's transitions)

    # ---- single-pass fp16 mode of the same step (stated looser bound), reported next to the headline mode ----
    loose = {}
    for lp in ("fp16",):
        if lp == prec or lp not in enabled:
            continue
        dyn_l = build_dynamics(mb, S, A, lp, dev)
        dyn_l.launch_step(obs_dev, None, ws, policy=ag.policy.network, max_action=1.0, step=0, row0=rank * Bn)
        lt = []
        for it in range(W + args.steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dyn_l.launch_step(obs_dev, None, ws, policy=ag.policy.network, max_action=1.0, step=it, row0=rank * Bn)
            e1.record()
            lt.append((e0, e1))
        torch.cuda.synchronize()
        loose[lp] = float(np.mean([a.elapsed_time(b) for a, b in lt[W:]]))
    clocks = sampler.stop()
    # ---- strong-scaling arm (BASELINE configs[2]) and, at N = 1, one line per BASELINE config ----
    strong = cfg_lines = None
    if not args.no_extras:
        strong = strong_scaling_arm(mb, P, dev, dist, rank, world, min(args.steps, 5))
        if world == 1:
            cfg_lines = baseline_config_lines(mb, dev)
    # second BASELINE metric: Q-weighted BC updates/sec (one update = one steady-state MOBODY.train step)
    upd_dev = upd_wall = None
    big_dev = big_wall = None
    par_dev = par_wall = None
    if rank == 0 and not args.no_train:
        upd_dev, upd_wall = gpu_train_rate(mb, dev, 128)
        par_dev, par_wall = gpu_train_rate(mb, dev, 128, penalty_type="par", dynamics=dyn)     # the CLI default penalty: + one 128-row dynamics step per update
        big_dev, big_wall = gpu_train_rate(mb, dev, 4096, steps=40, s_dim=27, a_dim=8)     # BASELINE configs[3]: ant-shaped, batch 4096

    t = torch.tensor([dev_ms, e2e_s, float(n_trans), float(e2e_trans), k_ms], dtype=torch.float64, device=dev)
    per_rank = None
    if dist is not None:
        allt = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(allt, t)
        per_rank = {"ms_per_step": [round(float(x[0]) / args.steps, 4) for x in allt], "step_kernel_ms": [round(float(x[4]), 4) for x in allt]}
        mx = t.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = t.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        dev_ms, e2e_s, k_ms = float(mx[0]), float(mx[1]), float(mx[4])
        n_trans, e2e_trans = float(sm[2]), float(mx[3])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    pk, pk_src = peaks()
    flop = flop_per_transition(S, A)
    split = {"fp32": 1, "fp16": 1, "bf16x2": 3}[prec]
    ach = flop * Bn / (k_ms * 1e-3) / 1e12
    peak = pk["bf16_tflops"]                               # kernel timed alone -> burst figure
    value = n_trans / (dev_ms * 1e-3)
    traffic, traffic_src = step_kernel_traffic() if (Bn == 100_000 and prec == "bf16x2") else (None, "not captured for this workload")
    # kernels launched per rollout: init, T steps (+2 image checksum/pack passes each), (T-1) x (3 compact + advance), 3 compact, pack (or pack+push), stats
    launches_per_rollout = 1 + T * 1 + 4 + (T - 1) * 4 + 3 + 1 + 1 + (2 if world > 1 else 0)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": W,
        "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32", "bf16x2": "bf16x2 (hi+lo split, fp32-parity)", "fp16": "f16"}[prec], "data": "synthetic",
        "config": {"workload": f"halfcheetah-gravity S{S}/A{A} rollout_length={T}, {Bn} start states per GPU, 7-member ensemble, hidden 256 "
                               f"(BASELINE configs[1])",
                   "precision": prec, "l2": f"inputs larger than L2: start states rotate over {n_pool} distinct buffers ({n_pool * Bn * S * 4 >> 20} MiB > 126 MB L2); "
                         "kernel-only timings flush L2 with a 256 MiB memset before each launch",
                   "streams": "consecutive (independent) rollouts alternate between two CUDA streams: one step kernel's partial last round overlaps the next one's first"
                              if two_streams else "one stream",
                   "parallelism": (f"dp{world} (start states sharded; transitions assembled in every rank's buffer by "
                                   f"{'peer-memory stores from the pack kernel' if exchange == 'p2p' else 'an NCCL all-gather of padded slabs'})")
                                  if world > 1 else "single GPU"},
        "e2e": {"value": e2e_trans / e2e_s, "unit": UNIT, "h2d_bytes_per_step": Bn * S * 4 * world, "d2h_bytes_per_step": int(d2h),
                "path": "MOBODY.rollout(host tensor)" if world == 1 else
                        "parallel.sharded_rollout_host: host shard in -> rollout -> peer-memory exchange (every rank's device buffer then holds all ranks' transitions) -> "
                        "this rank's transitions out as CPU tensors; the job's gathered output reaches the host once, in parallel over the ranks"},
        "gpu_launches": args.steps * launches_per_rollout,
        "roofline": {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": "fused rollout step", "kernel_ms": k_ms, "peak_source": pk_src + " bf16 burst",
                     "mma_passes_per_gemm": split, "frac_of_mma_issued": ach * split / peak,
                     "flop_per_transition": flop, "algorithmic_io_bytes": Bn * (3 * S + A + 3) * 4,
                     # the same algorithmic work over the whole timed loop (this rank's transitions / loop time): with two
                     # streams the partial last round of one launch is filled by the next launch, which the single-launch
                     # timing above cannot show
                     "per_rollout_in_loop": {"ms": dev_ms / args.steps, "achieved": flop * (n_trans / world) / (dev_ms * 1e-3) / 1e12,
                                             "frac": flop * (n_trans / world) / (dev_ms * 1e-3) / 1e12 / peak}},
        "clocks": clocks, "wall_s": wall,
    }
    if world > 1:
        line["exchange"] = {"mode": exchange, "peer_memory": P._exchange_mode(ag), "check": check}
        line["per_rank"] = per_rank
    if strong is not None:
        line["strong_scaling"] = strong
    if cfg_lines is not None:
        line["baseline_configs"] = cfg_lines
    for lp, ms in loose.items():
        la = flop * Bn / (ms * 1e-3) / 1e12
        line["roofline"][lp + "_single_pass"] = {
            "kernel_ms": ms, "achieved": la, "frac": la / peak, "transitions_per_s": Bn / (ms * 1e-3),
            "tolerance": "5e-3 relative (the stated looser bound of north_star for reduced-precision GEMMs; measured <= 4.6e-3)"}
    if not args.no_train:
        line["hbm_stages"] = hbm_stage_rates(mb, dev, pk["hbm_gbs"])
    if upd_wall is not None:
        line["train"] = {"metric": "Q-weighted BC updates/sec", "value": upd_wall, "unit": "updates/s", "device_only": upd_dev,
                         "config": {"workload": f"MOBODY.train steady state, batch 128 (128 src + 128 tar + 64 fake rows), S{S}/A{A}",
                                    "launches_per_update": 10, "dtype": "f32 (3xTF32 tensor-core MMA for the 256-wide layers, fp32 elsewhere)"},
                         "penalty_type_par": {"value": par_wall, "device_only": par_dev, "unit": "updates/s",
                                              "workload": "same with penalty_type='par' (the CLI default): + one fused 128-row dynamics step and the reward shift per update, no host sync"},
                         "batch4096_S27A8": {"value": big_wall, "device_only": big_dev, "unit": "updates/s",
                                             "workload": "MOBODY.train steady state, batch 4096 (4096 src + 4096 tar + 2048 fake rows), S27/A8 (BASELINE configs[3])"}}
    if upd_wall is not None:
        fit_dev, fit_wall = gpu_fit_rate(mb, dev, dyn)
        line["train"]["dynamics_fit"] = {"metric": "dynamics fitting steps/sec", "value": fit_wall, "device_only": fit_dev, "unit": "steps/s",
                                         "workload": f"MOBODYEnsembleDynamics.learn, 7 members x 256 rows per mini-batch, S{S}/A{A} "
                                                     "(3 losses + backward + Adam = one C-ABI call, 43 launches, weight gradients on a side stream)"}
    if not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        if upd_wall is not None:
            line["train"]["dynamics_fit"]["cpu_baseline"] = {"value": cpu_fit_rate(cores), "unit": "steps/s", "cores": cores, "kind": "port",
                                                             "sample": "oracle.fit_step (autograd + Adam), 3 steps after 1 warm-up"}
            line["train"]["cpu_baseline"] = {"value": cpu_train_rate(128, cores), "unit": "updates/s", "cores": cores, "kind": "port",
                                             "sample": "oracle.train_step incl. 3 buffer gathers, 5 steps after 2 warm-up"}
        n = min(Bn, 100_000)                   # the whole workload (~1.3 s per pass on 16 cores), best of 3 after a warm-up
        rate, dt = cpu_rollout_rate(n, cores, repeats=3)
        rate1, _ = cpu_rollout_rate(10_000, 1, repeats=1)      # the reference pins torch to ONE thread (train_mobody.py:3-5, 50-51)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"oracle.rollout (CPU restatement of MOBODY.rollout) on {n} of {Bn} start states, "
                                          f"best of 3 after 1 warm-up, torch threads={cores}",
                                "single_thread": {"value": rate1, "unit": UNIT, "cores": 1,
                                                  "sample": "same, 10000 start states, torch threads=1 (the reference's own setting)"},
                                "cpu_model": cpu_model()}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
