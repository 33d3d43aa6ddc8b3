"""CPU-side checks of policy evaluation in the learned model: the C ABI of mobody_model_eval (layout, argument checks,
workspace size) and the CPU reference model_return against the oracle's rollout."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

from model_eval_oracle import model_return
from oracle import mobody_oracle as M
from oracle.make_golden import healthy
from oracle.philox import rollout_elite_slot, rollout_noise

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mobody_b200.h")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from mobody_b200 import _ffi
    return _ffi.lib()


def test_model_eval_desc_layout_matches_header_via_gcc(lib, tmp_path):
    from mobody_b200 import _ffi
    ct, cname = _ffi.ModelEvalDesc, "mobody_model_eval_desc"
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             f'printf("{cname} %zu\\n", sizeof({cname}));']
    lines += [f'printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));' for f, _ in ct._fields_]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines + ["return 0;}"]))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got[cname]) == ctypes.sizeof(ct)
    for f, _ in ct._fields_:
        assert int(got[f"{cname}.{f}"]) == getattr(ct, f).offset, f


def test_workspace_size_has_no_horizon_and_grows_with_rows(lib):
    ws = lib.mobody_model_eval_workspace_bytes
    assert ws(0, 17, 6) == 0 and ws(10, 0, 6) == 0 and ws(10, 17, 0) == 0
    assert ws(2000, 17, 6) > ws(1000, 17, 6) > ws(1, 17, 6) > 0
    assert ws(1000, 17, 6) > ws(1000, 11, 3)
    # O(B): the start-state ping-pong, next state, action, 7 member means and per-row scalars, nothing per step
    assert ws(100_000, 17, 6) < 100_000 * 4 * (10 * 17 + 6 + 16)


def _valid_desc():
    """A descriptor that passes every check before the first launch (fake device pointers; nothing is dereferenced on the
    host).  Each rejection test breaks one field."""
    from mobody_b200 import _ffi
    keep = [_ffi.MlpParams(), _ffi.DynParams()]
    for i in range(3):
        keep[0].w[i] = keep[0].b[i] = 0x1000
    for i in range(13):
        keep[1].w[i] = keep[1].b[i] = 0x1000
    d = _ffi.ModelEvalDesc()
    s = d.step
    s.precision, s.B, s.S, s.A = _ffi.PREC["bf16x2"], 300, 17, 6
    s.obs, s.policy, s.dyn, s.dyn_pack, s.policy_pack = 0x1000, ctypes.pointer(keep[0]), ctypes.pointer(keep[1]), 0x1000, 0x1000
    s.elites, s.n_elites, s.step = 0x1000, 5, 0
    d.H, d.gamma = 1000, 0.99
    d.workspace, d.workspace_bytes = 0x1000, 1 << 40
    d.ret, d.ret_disc, d.length, d.counts = 0x1000, 0x1000, 0x1000, 0x1000
    return d, keep


def _breakers():
    def tc_shape(d):
        d.step.S, d.step.A = 64, 16                              # 2S+A = 144 > 96: bf16x2 cannot take it
    return [
        ("H=0", lambda d: setattr(d, "H", 0), b"bad H"),
        ("H too long", lambda d: setattr(d, "H", 100_001), b"bad H"),
        ("step word overflow", lambda d: setattr(d.step, "step", 2 ** 32 - 999), b"overflows"),
        ("eps", lambda d: setattr(d.step, "eps", 0x1000), b"Philox draws only"),
        ("idx", lambda d: setattr(d.step, "idx", 0x1000), b"Philox draws only"),
        ("policy", lambda d: setattr(d.step, "policy", None), b"policy"),
        ("strided start states", lambda d: setattr(d.step, "obs_ld", 44), b"dense"),
        ("ret", lambda d: setattr(d, "ret", None), b"null output"),
        ("ret_disc", lambda d: setattr(d, "ret_disc", None), b"null output"),
        ("length", lambda d: setattr(d, "length", None), b"null output"),
        ("counts", lambda d: setattr(d, "counts", None), b"null output"),
        ("no workspace", lambda d: setattr(d, "workspace", None), b"workspace"),
        ("small workspace", lambda d: setattr(d, "workspace_bytes", 1000), b"workspace"),
        ("precision shape", tc_shape, b"tensor-core modes take"),
    ]


@pytest.mark.parametrize("name,brk,msg", _breakers(), ids=[b[0] for b in _breakers()])
def test_model_eval_rejects_bad_arguments(lib, name, brk, msg):
    d, keep = _valid_desc()
    brk(d)
    assert lib.mobody_model_eval(ctypes.byref(d), None) == -1, name
    assert msg in lib.mobody_last_error(), (name, lib.mobody_last_error())


def test_model_eval_null_descriptor_and_last_step_word(lib):
    assert lib.mobody_model_eval(None, None) == -1 and b"null descriptor" in lib.mobody_last_error()
    d, keep = _valid_desc()
    d.step.step = 2 ** 32 - 1000                                 # step words up to 2^32 - 1: accepted, fails later at the shape
    d.step.S, d.step.A = 64, 16
    assert lib.mobody_model_eval(ctypes.byref(d), None) == -1 and b"tensor-core modes take" in lib.mobody_last_error()


def _hopper(S=11, A=3, seed=3):
    p = M.make_dynamics_params(S, A, seed, healthy_state=healthy("hopper", S, 0.8), t3_gain=2.0)
    st = M.AgentState(S, A, seed)
    obs = (healthy("hopper", S, 0.8)[None] + 0.1 * np.random.default_rng(1).standard_normal((40, S))).astype(np.float32)
    return p, st.policy, obs


def test_model_return_equals_per_start_sums_of_the_oracle_rollout():
    """model_return against M.rollout (no filter) fed the same Philox draws: the rollout's callables receive only the live
    row count, so the live global ids of each step are found by iterating to a fixed point (pass k fixes step k)."""
    p, pol, obs = _hopper()
    S, H, seed, step0, row0, gamma, coef = obs.shape[1], 6, 21, 9, 500, 0.97, 5.0
    B = len(obs)
    elites = p["elites"].numpy()
    ids = [np.arange(B)] * H

    def draws(t, n):
        rows = ids[t] if len(ids[t]) == n else np.arange(n)       # a wrong guess of step t's live rows: fixed in a later pass
        g = (row0 + rows).astype(np.uint64)
        members = elites[rollout_elite_slot(seed, step0 + t, g, len(elites))]
        eps = np.zeros((7, n, S), np.float32)
        eps[members, np.arange(n)] = rollout_noise(seed, step0 + t, g, S)
        return torch.from_numpy(eps), members

    for _ in range(H + 1):
        eps_l = [lambda n, t=t: draws(t, n)[0] for t in range(H)]
        idx_l = [lambda n, t=t: draws(t, n)[1] for t in range(H)]
        tr, _ = M.rollout(p, pol, 1.0, torch.from_numpy(obs), H, eps_l, idx_l, 2, coef, filter_bad=False)
        term = tr["terminals"].numpy()[:, 0] != 0
        new, off, cur = [], 0, np.arange(B)
        for t in range(H):                                       # step-major output, live rows in ascending order
            new.append(cur)
            n = len(cur)
            cur = cur[~term[off:off + n]]
            off += n
        if all(np.array_equal(a, b) for a, b in zip(new, ids)):
            break
        ids = new
    rew = tr["rewards"].numpy()[:, 0].astype(np.float64)
    ret, ret_disc, length = np.zeros(B), np.zeros(B), np.zeros(B, np.int32)
    off, disc = 0, 1.0
    for t in range(H):
        n = len(ids[t])
        ret[ids[t]] += rew[off:off + n]
        ret_disc[ids[t]] += disc * rew[off:off + n]
        length[ids[t]] = t + 1
        off, disc = off + n, disc * gamma
    assert off == len(rew)
    ref = model_return(p, pol, 1.0, obs, H, gamma, seed, step0, row0, 2, coef, use_penalty=True)
    assert 0 < ref["counts"][H] < B and len(set(ref["lengths"].tolist())) > 2     # rows end at different steps
    assert np.array_equal(ref["counts"][:H], [len(i) for i in ids])
    assert np.array_equal(ref["lengths"], length)
    assert np.array_equal(ref["returns"], ret) and np.array_equal(ref["discounted_returns"], ret_disc)


def test_model_return_runs_in_float64_with_float64_parameters():
    p, pol, obs = _hopper()
    p64 = {k: (v.double() if v.is_floating_point() else v) for k, v in p.items()}
    pol64 = {k: v.double() for k, v in pol.items()}
    a = model_return(p, pol, 1.0, obs, 8, 0.99, 4, 0, 0, 2, 5.0, record=True)
    b = model_return(p64, pol64, 1.0, obs.astype(np.float64), 8, 0.99, 4, 0, 0, 2, 5.0, record=True)
    assert a["trace"][0][1].dtype == np.float32 and b["trace"][0][1].dtype == np.float64
    same = a["lengths"] == b["lengths"]
    assert same.mean() > 0.9
    assert np.max(np.abs(a["returns"] - b["returns"])[same]) < 1e-4 * np.mean(np.abs(b["returns"]))
    assert not np.array_equal(a["returns"], b["returns"])
