"""CPU checks of the wide tensor-core step mode (precision "bf16x2_wide", MOBODY_PREC_BF16X2_WIDE): header constants
against the Python mirror, the shape range it takes, the argument rejections of mobody_step (they happen before any
launch), the packed-image sizes, and that the automatic precision choice is unchanged."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mobody_b200.h")
CONSTS = ("MOBODY_PREC_BF16X2", "MOBODY_PREC_BF16X2_WIDE", "MOBODY_TC_MAX_S", "MOBODY_TC_MAX_A", "MOBODY_TC_WIDE_MIN_S",
          "MOBODY_TC_WIDE_MAX_S", "MOBODY_TC_WIDE_MAX_A", "MOBODY_ABI_VERSION")


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
    assert got["MOBODY_PREC_BF16X2_WIDE"] == _ffi.PREC["bf16x2_wide"] == 4
    assert got["MOBODY_PREC_BF16X2"] == _ffi.PREC["bf16x2"]
    assert (got["MOBODY_TC_WIDE_MIN_S"], got["MOBODY_TC_WIDE_MAX_S"], got["MOBODY_TC_WIDE_MAX_A"]) == \
        (_ffi.TC_WIDE_MIN_S, _ffi.TC_WIDE_MAX_S, _ffi.TC_WIDE_MAX_A) == (65, 128, 32)
    assert got["MOBODY_TC_WIDE_MIN_S"] == got["MOBODY_TC_MAX_S"] + 1          # the two tensor-core ranges meet
    assert (got["MOBODY_TC_MAX_S"], got["MOBODY_TC_MAX_A"]) == (_ffi.TC_MAX_S, _ffi.TC_MAX_A)
    assert got["MOBODY_ABI_VERSION"] == _ffi.ABI_VERSION == 2


def test_tc_step_supports_at_the_edges():
    from mobody_b200.dynamics import tc_step_supports
    takes = [(65, 1), (65, 32), (111, 8), (128, 1), (128, 32)]
    refuses = [(64, 8), (64, 16), (2, 1), (129, 8), (111, 33), (111, 0), (200, 8)]
    assert all(tc_step_supports(S, A, "bf16x2_wide") for S, A in takes)
    assert not any(tc_step_supports(S, A, "bf16x2_wide") for S, A in refuses)
    assert not tc_step_supports(111, 8, "bf16x2") and tc_step_supports(17, 6, "bf16x2")   # the existing modes are unchanged


def test_auto_still_resolves_to_fp32_for_wide_observations():
    import mobody_b200 as mb
    for S, A, want in ((111, 8, "fp32"), (65, 1, "fp32"), (17, 6, "bf16x2")):
        m = mb.MOBODYModule(S, A, 256, 7, 5, device="cpu", config={"mopo": 0, "latent_reward": 0})
        d = mb.MOBODYEnsembleDynamics({}, m, None, None, mb.get_termination_fn("ant-medium-v2"), precision=None)
        assert d.precision == want, (S, A, d.precision)
        d = mb.MOBODYEnsembleDynamics({"b200_precision": "bf16x2_wide"}, m, None, None, mb.get_termination_fn("ant-medium-v2"))
        assert d.precision == "bf16x2_wide"


def _desc(S, A, precision=4, pack=True, policy=False):
    from mobody_b200 import _ffi
    dp, mp = _ffi.DynParams(), _ffi.MlpParams()
    for i in range(13):
        dp.w[i] = dp.b[i] = 0x1000
    for i in range(3):
        mp.w[i] = mp.b[i] = 0x1000
    d = _ffi.StepDesc()
    d.precision, d.B, d.S, d.A = precision, 100, S, A
    d.obs, d.act, d.next_obs, d.reward, d.penalty, d.terminal, d.mean = (0x1000,) * 7
    d.dyn, d.elites, d.n_elites = ctypes.pointer(dp), 0x1000, 5
    d.dyn_pack = 0x1000 if pack else None
    if policy:
        d.policy, d.act_out = ctypes.pointer(mp), 0x1000
    return d, (dp, mp)


@pytest.mark.parametrize("S,A", [(64, 8), (129, 8), (111, 33), (2, 1)])
def test_step_rejects_shapes_outside_the_wide_range(lib, S, A):
    d, keep = _desc(S, A)
    assert lib.mobody_step(ctypes.byref(d), None) == -1
    assert b"bf16x2_wide takes 65 <= S <= 128 and A <= 32" in lib.mobody_last_error()


def test_step_rejects_a_missing_pack(lib):
    d, keep = _desc(111, 8, pack=False)
    assert lib.mobody_step(ctypes.byref(d), None) == -1 and b"needs dyn_pack" in lib.mobody_last_error()
    d, keep = _desc(111, 8, policy=True)
    assert lib.mobody_step(ctypes.byref(d), None) == -1 and b"fused policy needs policy_pack" in lib.mobody_last_error()


def test_existing_rejection_text_is_unchanged(lib):
    d, keep = _desc(111, 8, precision=1)
    assert lib.mobody_step(ctypes.byref(d), None) == -1
    assert lib.mobody_last_error() == b"mobody_step: tensor-core modes take S <= 64, A <= 16 and 2S+A <= 96 (bf16x2) / 112 (fp16)"


def test_packed_images_are_the_bf16x2_images(lib):
    for S, A in ((65, 1), (111, 8), (128, 32)):
        assert lib.mobody_dyn_pack_bytes(S, A, 4) == lib.mobody_dyn_pack_bytes(S, A, 1) > 0
        assert lib.mobody_mlp_pack_bytes(S, A, 4) == lib.mobody_mlp_pack_bytes(S, A, 1) > 0
