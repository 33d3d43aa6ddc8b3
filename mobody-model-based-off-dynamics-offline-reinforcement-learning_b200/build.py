"""Build libmobody_b200.so in-tree with nvcc for sm_100a (no torch / pybind dependency in the .so)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmobody_b200.so")
SOURCES = ["api.cu", "step_simt.cu", "buffer.cu", "peer.cu", "tc_selftest.cu", "step_tc.cu", "step_duo.cu", "step_wide.cu", "train.cu", "train_tc.cu", "dynfit.cu"]
NVCC_FLAGS = (["-DUG_TRACE"] if os.environ.get("UG_TRACE") else []) + ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose=False, force=False):
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(os.path.dirname(HERE), "include", "mobody_b200.h"))
    objs, jobs = [], []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src in SOURCES:
        sp = os.path.join(CSRC, src)
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        if force or _stale(obj, [sp] + hdrs):
            jobs.append((src, [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", sp, "-o", obj]))
        objs.append(obj)
    if jobs:   # translation units are independent: compile them side by side
        from concurrent.futures import ThreadPoolExecutor
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            results = list(ex.map(lambda j: (j[0], subprocess.run(j[1], capture_output=True, text=True)), jobs))
        for src, r in results:
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
        bad = [src for src, r in results if r.returncode]
        if bad:
            raise RuntimeError(f"nvcc failed on {', '.join(bad)}")
    if force or _stale(LIB, objs):
        cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs + ["-lcudart"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv))
