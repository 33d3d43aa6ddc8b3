"""CPU-side checks of the C-ABI boundary: the library builds, loads and exports every declared symbol."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mobody_b200.h")


@pytest.fixture(scope="module")
def libpath():
    import __graft_entry__ as g
    g.build()
    from mobody_b200 import _ffi
    assert os.path.exists(_ffi.LIB_PATH)
    return _ffi.LIB_PATH


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?(?:int|long long|char\s*\*|const char\s*\*)\s+(mobody_\w+)\s*\(", src, flags=re.M)
    assert len(names) >= 12
    return names


def test_every_declared_symbol_is_exported(libpath):
    lib = ctypes.CDLL(libpath)
    for name in declared_functions():
        assert hasattr(lib, name), f"{name} declared in include/mobody_b200.h but not exported"


def test_abi_version_and_pure_host_calls(libpath):
    from mobody_b200 import _ffi
    L = _ffi.lib()
    assert L.mobody_abi_version() == 2 == _ffi.ABI_VERSION
    assert int(re.search(r"#define MOBODY_TC_TRAIN_MIN_ROWS (\d+)", open(HEADER).read()).group(1)) == _ffi.TC_TRAIN_MIN_ROWS
    assert L.mobody_row_width(17, 6) == 44 and L.mobody_row_width(11, 3) == 28 and L.mobody_row_width(27, 8) == 64
    assert L.mobody_compact_scratch_ints(1) == 2 and L.mobody_compact_scratch_ints(1025) == 3


def test_argument_errors_are_reported_not_raised_across_abi(libpath):
    from mobody_b200 import _ffi
    L = _ffi.lib()
    assert L.mobody_step(None, None) == -1 and b"null descriptor" in L.mobody_last_error()
    assert L.mobody_gather_rows(None, None, 4, 7, None, None) == -1     # row width not a multiple of 4
    assert L.mobody_ring_insert(None, 10, None, 44, 0, 5, None, None) == -1   # batch larger than capacity
    assert L.mobody_termination(None, 1, 17, 99, None, None) == -1
    # whole-rollout / classifier / sampling entry points: descriptor validation happens before any launch
    assert L.mobody_rollout(None, None) == -1 and b"null descriptor" in L.mobody_last_error()
    rd = _ffi.RolloutDesc()
    rd.T, rd.step.B, rd.step.S, rd.step.A = 0, 4, 17, 6
    assert L.mobody_rollout(ctypes.byref(rd), None) == -1 and b"bad T" in L.mobody_last_error()
    rd.T = 2
    assert L.mobody_rollout(ctypes.byref(rd), None) == -1 and b"policy" in L.mobody_last_error()
    assert L.mobody_classifier_step(None, None) == -1
    assert L.mobody_dynfit_step(None, None) == -1 and b"null descriptor" in L.mobody_last_error()
    assert L.mobody_dynfit_workspace_bytes(256, 17, 6, 4) > L.mobody_dynfit_workspace_bytes(128, 17, 6, 4) > 0
    assert L.mobody_dara_relabel(None, 5, 17, 6, 44, None, None, 1.0, None, None) == -1
    assert L.mobody_sample_rows(None, 3, 44, None) == -1
    sj = (_ffi.SampleJob * 1)()
    sj[0].n, sj[0].size = 4, 0
    assert L.mobody_sample_rows(sj, 1, 44, None) == -1 and b"empty buffer" in L.mobody_last_error()
    assert 2 * L.mobody_dyn_pack_bytes(17, 6, 3) > L.mobody_dyn_pack_bytes(17, 6, 1) > L.mobody_dyn_pack_bytes(17, 6, 3) > 0   # one fp16 plane vs bf16 hi+lo
    assert L.mobody_par_penalty(None, 4, 17, 6, 40, None, 1.0, None, None) == -1 and b"bad arguments" in L.mobody_last_error()   # wrong row width
    assert L.mobody_rollout_stats_doubles() >= 4
    assert L.mobody_dyn_pack_bytes(17, 6, 0) == 0                                           # fp32 mode has no packed image
    with pytest.raises(RuntimeError, match="mobody_b200"):
        _ffi.check(-1)


def test_struct_mirrors_match_header_sizes(libpath):
    from mobody_b200 import _ffi
    assert ctypes.sizeof(_ffi.DynParams) == 2 * 13 * 8 and ctypes.sizeof(_ffi.MlpParams) == 6 * 8


def test_struct_layouts_match_header_via_gcc(libpath, tmp_path):
    """Compile include/mobody_b200.h with gcc and compare sizeof/offsetof with the ctypes mirrors field by field."""
    import subprocess
    from mobody_b200 import _ffi
    structs = {"mobody_step_desc": _ffi.StepDesc, "mobody_train_desc": _ffi.TrainDesc,
               "mobody_dyn_params": _ffi.DynParams, "mobody_mlp_params": _ffi.MlpParams, "mobody_mlp_state": _ffi.MlpState,
               "mobody_rollout_desc": _ffi.RolloutDesc, "mobody_classifier_desc": _ffi.ClassifierDesc,
               "mobody_sample_job": _ffi.SampleJob, "mobody_peer_desc": _ffi.PeerDesc,
               "mobody_dyn_state": _ffi.DynState, "mobody_dynfit_desc": _ffi.DynFitDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){']
    for cname, ct in structs.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in ct._fields_:
            lines.append(f'printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['return 0;}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, ct in structs.items():
        assert int(got[cname]) == ctypes.sizeof(ct), cname
        for fname, _ in ct._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(ct, fname).offset, f"{cname}.{fname}"


def test_no_cpu_path():
    """Product classes refuse CPU devices instead of silently falling back."""
    import torch
    import mobody_b200 as mb
    with pytest.raises(RuntimeError):
        mb.ReplayBuffer(3, 2, "cpu", max_size=8)
    with pytest.raises(RuntimeError):
        mb._ffi.ptr(torch.zeros(2))


def test_termination_dispatch_order():
    import mobody_b200 as mb
    kinds = {n: mb.get_termination_fn(n).kind for n in
             ["halfcheetahvel-x", "halfcheetah-medium-v2", "hopper-medium-v2", "antangle", "antmaze-umaze-v0",
              "walker2d-medium-v2", "pendulum", "humanoid", "pen-human-v0", "door-human"]}
    assert kinds == {"halfcheetahvel-x": 0, "halfcheetah-medium-v2": 1, "hopper-medium-v2": 2, "antangle": 4,
                     "antmaze-umaze-v0": 4, "walker2d-medium-v2": 3, "pendulum": 0, "humanoid": 5, "pen-human-v0": 6,
                     "door-human": 0}
    with pytest.raises(TypeError):
        mb.get_termination_fn("unknown")


def test_checkpoint_formats_match_the_reference(golden_dir, tmp_path):
    """SURVEY.md section 8f rank 2: dynamics.pth / _actor / _critic written by the reference load unchanged — the mirror
    modules expose exactly the reference's state_dict keys and shapes (golden list generated from the reference)."""
    import json
    import torch
    import mobody_b200 as mb
    want = json.load(open(os.path.join(golden_dir, "checkpoint_keys.json")))
    for tag, (S, A) in (("S17A6", (17, 6)), ("S11A3", (11, 3))):
        m = mb.MOBODYModule(S, A, 256, 7, 5, device="cpu", config={"mopo": 0, "latent_reward": 0})
        assert {k: list(v.shape) for k, v in m.state_dict().items()} == want[tag]["dynamics.pth"]
        assert {k: list(v.shape) for k, v in mb.Policy(S, A, 1.0).state_dict().items()} == want[tag]["_actor"]
        assert {k: list(v.shape) for k, v in mb.DoubleQFunc(S, A).state_dict().items()} == want[tag]["_critic"]
        assert {k: list(v.shape) for k, v in mb.Classifier(S, A).state_dict().items()} == want[tag]["classifier"]
    # the identity scaler writes / reads the reference's mu.npy / std.npy side files (mobody_dynamics.py:133-154)
    sc = mb.StandardScaler()
    sc.save_scaler(str(tmp_path)); sc.load_scaler(str(tmp_path))
    assert sc.mu == 0 and sc.std == 1 and sorted(os.listdir(tmp_path)) == ["mu.npy", "std.npy"]
