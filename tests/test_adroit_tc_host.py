"""CPU checks of the 64-row tensor-core step mode for the S <= 64 shapes bf16x2 refuses (precision "bf16x2_t64",
MOBODY_PREC_BF16X2_T64; Adroit's pen, door, relocate and hammer): header constants against the Python mirror, the
partition of the fp32 mode's shapes between the three bf16x2-arithmetic modes, the argument rejections of mobody_step
(they happen before any launch), the packed-image sizes, and that the automatic precision choice is unchanged."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mobody_b200.h")
CONSTS = ("MOBODY_PREC_BF16X2", "MOBODY_PREC_BF16X2_WIDE", "MOBODY_PREC_BF16X2_T64", "MOBODY_TC_MAX_S", "MOBODY_TC_MAX_A",
          "MOBODY_TC_BF16X2_MAX_SAS", "MOBODY_TC_T64_MAX_S", "MOBODY_TC_T64_MAX_A", "MOBODY_ABI_VERSION")
ADROIT = {"pen": (45, 24), "door": (39, 28), "relocate": (39, 30), "hammer": (46, 26)}
T64_ERR = b"mobody_step: bf16x2_t64 takes S <= 64, A <= 32 with A > 16 or 2S+A > 96"


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from mobody_b200 import _ffi
    return _ffi.lib()


def test_header_constants_match_the_python_mirror(tmp_path):
    from mobody_b200 import _ffi
    src = tmp_path / "consts.c"
    src.write_text("\n".join(['#include <stdio.h>', f'#include "{HEADER}"', 'int main(void){'] +
                             [f'printf("{c} %d\\n", (int){c});' for c in CONSTS] + ['return 0;}']))
    exe = tmp_path / "consts"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    got = {k: int(v) for k, v in (l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True,
                                                                     text=True).stdout.splitlines())}
    assert got["MOBODY_PREC_BF16X2_T64"] == _ffi.PREC["bf16x2_t64"] == 5
    assert got["MOBODY_PREC_BF16X2_WIDE"] == _ffi.PREC["bf16x2_wide"] and got["MOBODY_PREC_BF16X2"] == _ffi.PREC["bf16x2"]
    assert (got["MOBODY_TC_T64_MAX_S"], got["MOBODY_TC_T64_MAX_A"]) == (_ffi.TC_T64_MAX_S, _ffi.TC_T64_MAX_A) == (64, 32)
    assert got["MOBODY_TC_T64_MAX_S"] == got["MOBODY_TC_MAX_S"]                # the range ends where bf16x2_wide's begins
    assert got["MOBODY_TC_BF16X2_MAX_SAS"] == _ffi.TC_MAX_SAS["bf16x2"] and got["MOBODY_TC_MAX_A"] == _ffi.TC_MAX_A
    assert got["MOBODY_ABI_VERSION"] == _ffi.ABI_VERSION == 2


def test_the_three_bf16x2_modes_partition_the_fp32_shapes():
    """Every (S, A) the fp32 mode takes (2 <= S <= 128, 1 <= A <= 32) is taken by exactly one of bf16x2, bf16x2_t64 and
    bf16x2_wide; bf16x2_t64 takes exactly 2 <= S <= 64, 1 <= A <= 32 with A > 16 or 2S+A > 96."""
    from mobody_b200.dynamics import tc_step_supports
    modes = ("bf16x2", "bf16x2_t64", "bf16x2_wide")
    for S in range(2, 129):
        for A in range(1, 33):
            takes = [m for m in modes if tc_step_supports(S, A, m)]
            assert len(takes) == 1, (S, A, takes)
            assert (takes[0] == "bf16x2_t64") == (S <= 64 and (A > 16 or 2 * S + A > 96)), (S, A)
    for S, A in ((1, 20), (64, 33), (65, 20), (45, 0), (200, 24)):
        assert not tc_step_supports(S, A, "bf16x2_t64"), (S, A)
    assert all(tc_step_supports(S, A, "bf16x2_t64") for S, A in ADROIT.values())
    assert tc_step_supports(45, 17, "bf16x2_t64")                               # the truncated Humanoid observation


def test_auto_still_resolves_to_fp32_at_the_adroit_shapes():
    import mobody_b200 as mb
    for task, (S, A) in (("pen-human-v0", ADROIT["pen"]), ("door-human-v0", ADROIT["door"]), ("humanoid-v2", (45, 17))):
        m = mb.MOBODYModule(S, A, 256, 7, 5, device="cpu", config={"mopo": 0, "latent_reward": 0})
        d = mb.MOBODYEnsembleDynamics({}, m, None, None, mb.get_termination_fn(task), precision=None)
        assert d.precision == "fp32", (task, d.precision)
        d = mb.MOBODYEnsembleDynamics({"b200_precision": "bf16x2_t64"}, m, None, None, mb.get_termination_fn(task))
        assert d.precision == "bf16x2_t64"


def _desc(S, A, precision=5, pack=True, policy=False, term_kind=0):
    from mobody_b200 import _ffi
    dp, mp = _ffi.DynParams(), _ffi.MlpParams()
    for i in range(13):
        dp.w[i] = dp.b[i] = 0x1000
    for i in range(3):
        mp.w[i] = mp.b[i] = 0x1000
    d = _ffi.StepDesc()
    d.precision, d.B, d.S, d.A, d.term_kind = precision, 100, S, A, term_kind
    d.obs, d.act, d.next_obs, d.reward, d.penalty, d.terminal, d.mean = (0x1000,) * 7
    d.dyn, d.elites, d.n_elites = ctypes.pointer(dp), 0x1000, 5
    d.dyn_pack = 0x1000 if pack else None
    if policy:
        d.policy, d.act_out = ctypes.pointer(mp), 0x1000
    return d, (dp, mp)


@pytest.mark.parametrize("S,A", [(17, 6), (40, 16), (2, 16), (47, 2), (65, 8), (111, 24), (64, 33), (45, 33)])
def test_step_rejects_shapes_outside_the_t64_range(lib, S, A):
    """Shapes bf16x2 takes (up to 2S+A = 96 with A <= 16), bf16x2_wide's (S > 64) and A > 32."""
    d, keep = _desc(S, A)
    assert lib.mobody_step(ctypes.byref(d), None) == -1
    assert lib.mobody_last_error() == T64_ERR


def test_step_rejects_a_missing_pack(lib):
    d, keep = _desc(45, 24, pack=False)
    assert lib.mobody_step(ctypes.byref(d), None) == -1 and b"needs dyn_pack" in lib.mobody_last_error()
    d, keep = _desc(45, 24, policy=True)
    assert lib.mobody_step(ctypes.byref(d), None) == -1 and b"fused policy needs policy_pack" in lib.mobody_last_error()


def test_pen_termination_still_needs_27_columns(lib):
    d, keep = _desc(20, 24, term_kind=6)
    assert lib.mobody_step(ctypes.byref(d), None) == -1
    assert lib.mobody_last_error() == b"mobody_step: pen termination needs S >= 27"


def test_existing_rejection_texts_are_unchanged(lib):
    d, keep = _desc(45, 24, precision=1)
    assert lib.mobody_step(ctypes.byref(d), None) == -1
    assert lib.mobody_last_error() == b"mobody_step: tensor-core modes take S <= 64, A <= 16 and 2S+A <= 96 (bf16x2) / 112 (fp16)"
    d, keep = _desc(45, 24, precision=4)
    assert lib.mobody_step(ctypes.byref(d), None) == -1
    assert lib.mobody_last_error() == b"mobody_step: bf16x2_wide takes 65 <= S <= 128 and A <= 32"


def test_packed_images_are_the_bf16x2_images(lib):
    for S, A in list(ADROIT.values()) + [(45, 17), (2, 17), (64, 32)]:
        assert lib.mobody_dyn_pack_bytes(S, A, 5) == lib.mobody_dyn_pack_bytes(S, A, 1) > 0
        assert lib.mobody_mlp_pack_bytes(S, A, 5) == lib.mobody_mlp_pack_bytes(S, A, 1) > 0
