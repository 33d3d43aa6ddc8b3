#!/usr/bin/env python
"""One SHA-256 per case of mobody_step, called through the C ABI, over a case matrix that reaches every tensor-core step
kernel: step_tc_kernel<2> (bf16x2), step_duo_kernel<false> (bf16), step_tc_kernel<1> (bf16 where two tiles do not fit),
step_duo_kernel<true> (fp16) and both step_wide_kernel instantiations (bf16x2_wide, bf16x2_t64, fp16_t64).

A case hashes next_obs, reward, raw_reward, penalty, terminal, mean and act_out (outputs start zeroed, so rows a case does
not write hash too).  Parameters, inputs and Philox keys are seeded: two builds of the library compute the same bits iff
their outputs are identical.  Compare two builds by running the script once per build and diffing the outputs:

  MOBODY_B200_LIB=/path/to/other/libmobody_b200.so python scripts/step_digest.py > other.txt
  python scripts/step_digest.py > this.txt && diff other.txt this.txt

Flags covered: B of 1, one tile - 1, one tile, one tile + 1 (and two tiles +- 1 on the two-tile kernel), 1 000 and 100 000
rows; fused policy and given actions; Philox and injected eps; Philox elite pick and injected idx; use_trg and use_penalty
on and off; every termination kind the shape allows; a live row count below B on the device; explicit row ids; row strides
above S / A.
"""
import ctypes as C
import hashlib
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import torch  # noqa: E402

E = 7
# (mode name, precision code, S, A, row tile of the kernel it reaches)
CASES = [
    ("bf16x2", 1, 17, 6, 128),
    ("bf16", 2, 17, 6, 256),          # two tiles per CTA
    ("bf16", 2, 60, 16, 128),         # 2S+A > 112: two tiles do not fit, the one-tile kernel with a single plane
    ("fp16", 3, 17, 6, 256),
    ("bf16x2_wide", 4, 111, 8, 64),
    ("bf16x2_wide", 4, 128, 32, 64),
    ("bf16x2_t64", 5, 45, 24, 64),
    ("bf16x2_t64", 5, 2, 17, 64),
    ("fp16_t64", 6, 111, 8, 64),
    ("fp16_t64", 6, 128, 32, 64),
    ("fp16_t64", 6, 45, 24, 64),
    ("fp16_t64", 6, 2, 17, 64),
]
TERM_KINDS = range(7)   # never, halfcheetah, hopper, walker2d, ant, humanoid, pen (S >= 27)


def dyn_dims(S, A):
    """(in, out) of the 13 dynamics layers, MbLayer order (weight [E, in, out], bias [E, 1, out])."""
    return list(zip([S, 256, 256, 16 + A, 32, 16 + A, 32, 16, 256, 256, 2 * S + A, 256, 256],
                    [256, 256, 32, 32, 32, 32, 32, 256, 256, S, 256, 256, 2]))


class Model:
    def __init__(self, ffi, prec, S, A, dev, gen):
        L = ffi.lib()
        st = ffi.stream_ptr()
        self.dyn = [(torch.randn(E, i, o, generator=gen, device=dev) / i ** 0.5,
                     0.1 * torch.randn(E, 1, o, generator=gen, device=dev)) for i, o in dyn_dims(S, A)]
        self.dyn[9][1][:, :, 0] += 0.6        # transition3: x0 near the healthy ranges, so part of the rows terminate
        self.pol = [(torch.randn(o, i, generator=gen, device=dev) / i ** 0.5, 0.1 * torch.randn(o, generator=gen, device=dev))
                    for i, o in ((S, 256), (256, 256), (256, A))]
        self.dp = ffi.DynParams()
        for k, (w, b) in enumerate(self.dyn):
            self.dp.w[k], self.dp.b[k] = w.data_ptr(), b.data_ptr()
        self.mp = ffi.MlpParams()
        for k, (w, b) in enumerate(self.pol):
            self.mp.w[k], self.mp.b[k] = w.data_ptr(), b.data_ptr()
        self.dyn_blob = torch.empty(int(L.mobody_dyn_pack_bytes(S, A, prec)), dtype=torch.uint8, device=dev)
        self.pol_blob = torch.empty(int(L.mobody_mlp_pack_bytes(S, A, prec)), dtype=torch.uint8, device=dev)
        ffi.check(L.mobody_dyn_pack(C.byref(self.dp), S, A, prec, self.dyn_blob.data_ptr(), None, st))
        ffi.check(L.mobody_mlp_pack(C.byref(self.mp), S, A, prec, self.pol_blob.data_ptr(), None, st))


def run(ffi, m, prec, S, A, B, dev, gen, policy=True, eps=False, idx=False, use_trg=1, use_penalty=1, term=0,
        n_live=None, row_ids=False, ld=0):
    obs_ld, act_ld = S + ld, A + ld
    obs = 0.2 * torch.randn(B, obs_ld, generator=gen, device=dev)
    obs[:, 0] += 0.6
    act = torch.rand(B, act_ld, generator=gen, device=dev) * 2 - 1
    out = {"next_obs": torch.zeros(B, S, device=dev), "reward": torch.zeros(B, device=dev),
           "raw_reward": torch.zeros(B, device=dev), "penalty": torch.zeros(B, device=dev),
           "terminal": torch.zeros(B, dtype=torch.uint8, device=dev), "mean": torch.zeros(E, B, S, device=dev),
           "act_out": torch.zeros(B, A, device=dev)}
    keep = [obs, act]
    d = ffi.StepDesc()
    d.precision, d.B, d.S, d.A, d.obs_ld, d.act_ld = prec, B, S, A, obs_ld, act_ld
    d.obs = obs.data_ptr()
    if policy:
        d.policy, d.policy_pack, d.max_action = C.pointer(m.mp), m.pol_blob.data_ptr(), 1.0
    else:
        d.act = act.data_ptr()
    d.dyn, d.dyn_pack = C.pointer(m.dp), m.dyn_blob.data_ptr()
    d.use_trg, d.use_penalty, d.penalty_coef, d.term_kind = use_trg, use_penalty, 1.0, term
    if eps:
        keep.append(torch.randn(E, B, S, generator=gen, device=dev))
        d.eps = keep[-1].data_ptr()
    if idx:
        keep.append(torch.randint(0, E, (B,), generator=gen, device=dev, dtype=torch.int64))
        d.idx = keep[-1].data_ptr()
    keep.append(torch.tensor([0, 2, 3, 5, 6], dtype=torch.int64, device=dev))
    d.elites, d.n_elites = keep[-1].data_ptr(), 5
    if n_live is not None:
        keep.append(torch.tensor([n_live], dtype=torch.int32, device=dev))
        d.n_rows_dev = keep[-1].data_ptr()
    if row_ids:
        keep.append(torch.randperm(10 * B, generator=gen, device=dev)[:B].to(torch.int64))
        d.row_ids = keep[-1].data_ptr()
    d.seed, d.step, d.row0 = 1234567, 42, 1000
    for k in out:
        setattr(d, k, out[k].data_ptr())
    ffi.check(ffi.lib().mobody_step(C.byref(d), ffi.stream_ptr()))
    h = hashlib.sha256()
    for k in ("next_obs", "reward", "raw_reward", "penalty", "terminal", "mean", "act_out"):
        h.update(out[k].cpu().numpy().tobytes())
    return h.hexdigest()


def main():
    if not torch.cuda.is_available():
        raise SystemExit("step_digest: needs a CUDA device")
    from mobody_b200 import _ffi as ffi
    dev = torch.device("cuda:0")
    print(f"# library {os.path.abspath(ffi.LIB_PATH)}", file=sys.stderr)
    for name, prec, S, A, tile in CASES:
        gen = torch.Generator(device=dev).manual_seed(prec * 1000 + S * 40 + A)
        m = Model(ffi, prec, S, A, dev, gen)
        terms = [t for t in TERM_KINDS if t != 6 or S >= 27]
        rows = sorted({1, tile - 1, tile, tile + 1, 1000, 100_000} | ({127, 128, 129} if tile == 256 else set()))
        variants = [(f"B{B}", dict(B=B, term=terms[i % len(terms)])) for i, B in enumerate(rows)]
        variants += [(k, dict({"B": 1000}, **kw)) for k, kw in (
            ("B1000 given_act", dict(policy=False)), ("B1000 eps", dict(eps=True)), ("B1000 idx", dict(idx=True)),
            ("B1000 src", dict(use_trg=0)), ("B1000 no_penalty", dict(use_penalty=0)), ("B1000 n_live", dict(n_live=777)),
            ("B1000 row_ids", dict(row_ids=True)), ("B1000 ld", dict(ld=3)),
            ("B1000 given_act eps idx row_ids n_live", dict(policy=False, eps=True, idx=True, row_ids=True, n_live=501)),
            ("B100000 given_act src n_live", dict(B=100_000, policy=False, use_trg=0, n_live=99_937)))]
        variants += [(f"B1000 term{t}", dict(B=1000, term=t)) for t in terms]
        for label, kw in variants:
            print(f"{name} S{S}/A{A} {label}: {run(ffi, m, prec, S, A, dev=dev, gen=gen, **kw)}", flush=True)


if __name__ == "__main__":
    main()
