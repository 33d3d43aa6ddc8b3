"""Updates/s of the train step for every update-branch flag set, fused (train_on_rows) and through the torch autograd
reference (_train_torch_path), at batch 128 (S17/A6, 320 rows: 128 src + 128 tar + 64 fake) and batch 4096 (S27/A8,
10 240 rows).  Before timing, one update of each path from the same state must agree (test_gpu_train.adam_close).
Timing: CUDA events around `--steps` updates after `--warmup`; the card's name and power limit are read in the same run.
One JSON line per (batch, flags, path); `--out` also writes them to a file.

    python scripts/train_branch_bench.py --steps 200 --warmup 20
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

FLAGS = {"default": {}, "advantage": dict(advantage=1), "scale_Q=0": dict(scale_Q=0), "q_weighted=0": dict(q_weighted=0),
         "advantage,q_weighted=0": dict(advantage=1, q_weighted=0), "all three": dict(advantage=1, scale_Q=0, q_weighted=0)}
BATCHES = {128: (17, 6, 320, 256), 4096: (27, 8, 10240, 8192)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def agent(S, A, flags):
    from collections import OrderedDict
    from helpers import cuda_agent
    from oracle import mobody_oracle as M
    ag, _ = cuda_agent(S, A, 3, **flags)
    ag.v_func.load_state_dict(OrderedDict(("network." + k, v) for k, v in M.make_mlp_params(S, 1, 10).items()))
    return ag


def rows_for(S, A, N):
    from mobody_b200 import _ffi
    rng = np.random.default_rng(N)
    RW = _ffi.lib().mobody_row_width(S, A)
    rows = np.zeros((N, RW), np.float32)
    rows[:, :2 * S + A + 1] = rng.standard_normal((N, 2 * S + A + 1))
    rows[:, S:S + A] = rng.uniform(-1, 1, (N, A))
    rows[:, 2 * S + A + 1] = rng.random(N) > 0.1
    return torch.from_numpy(rows).cuda()


def check_agree(S, A, N, n_true, flags, rows):
    """One update of each path from the same state: every parameter tensor under the test suite's post-Adam criterion."""
    from test_gpu_train import adam_close
    a1, a2 = agent(S, A, flags), agent(S, A, flags)
    a1.train_on_rows(rows, n_true)
    a2._train_torch_path(rows, n_true, None, None)
    torch.cuda.synchronize()
    for m1, m2 in ((a1.policy, a2.policy), (a1.q_funcs, a2.q_funcs), (a1.target_q_funcs, a2.target_q_funcs), (a1.v_func, a2.v_func)):
        for (k, x1), x2 in zip(m1.state_dict().items(), m2.state_dict().values()):
            adam_close(x1.cpu().numpy(), x2.cpu().numpy(), 3e-4, 1, (flags, N, k))


def rate(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    t1.synchronize()
    return steps / (t0.elapsed_time(t1) / 1e3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--torch-steps", type=int, default=50, help="timed updates of the (slow) torch path")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_branch_bench needs a CUDA device")
    import mobody_b200  # noqa: F401
    dev = card()
    lines = []
    for batch, (S, A, N, n_true) in BATCHES.items():
        rows = rows_for(S, A, N)
        for name, flags in FLAGS.items():
            check_agree(S, A, N, n_true, flags, rows)
            ag, ref = agent(S, A, flags), agent(S, A, flags)
            for path, fn, steps in (("fused", lambda: ag.train_on_rows(rows, n_true), a.steps),
                                    ("torch", lambda: ref._train_torch_path(rows, n_true, None, None), a.torch_steps)):
                r = rate(fn, steps, a.warmup)
                ln = dict(batch=batch, S=S, A=A, rows=N, flags=name, path=path, updates_per_s=round(r, 1), timed_steps=steps, card=dev)
                print(json.dumps(ln), flush=True)
                lines.append(ln)
    if a.out:
        with open(a.out, "w") as f:
            f.write("".join(json.dumps(ln) + "\n" for ln in lines))


if __name__ == "__main__":
    main()
