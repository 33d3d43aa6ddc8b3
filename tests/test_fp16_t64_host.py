"""CPU checks of the fp16 step mode on 64-row tiles (precision "fp16_t64", MOBODY_PREC_FP16_T64; Ant's 111 dimensions,
Adroit's pen, door, relocate and hammer): the header constant against the Python mirror, the partition of the fp32 mode's
shapes between fp16 and fp16_t64, the argument rejections of mobody_step (they happen before any launch) and their
texts, the packed-image sizes, and that the automatic precision choice is unchanged."""
import ctypes
import subprocess

import pytest

from test_adroit_tc_host import HEADER, _desc

CONSTS = ("MOBODY_PREC_FP16", "MOBODY_PREC_FP16_T64", "MOBODY_TC_MAX_S", "MOBODY_TC_MAX_A", "MOBODY_TC_FP16_MAX_SAS",
          "MOBODY_TC_WIDE_MAX_S", "MOBODY_TC_WIDE_MAX_A", "MOBODY_ABI_VERSION")
SHAPES = {"ant": (111, 8), "pen": (45, 24), "door": (39, 28), "relocate": (39, 30), "hammer": (46, 26)}
F16_T64_ERR = b"mobody_step: fp16_t64 takes S <= 128, A <= 32 outside fp16's S <= 64, A <= 16, 2S+A <= 112"


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from mobody_b200 import _ffi
    return _ffi.lib()


def test_header_constant_matches_the_python_mirror(tmp_path):
    from mobody_b200 import _ffi
    src = tmp_path / "consts.c"
    src.write_text("\n".join(['#include <stdio.h>', f'#include "{HEADER}"', 'int main(void){'] +
                             [f'printf("{c} %d\\n", (int){c});' for c in CONSTS] + ['return 0;}']))
    exe = tmp_path / "consts"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    got = {k: int(v) for k, v in (l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True,
                                                                     text=True).stdout.splitlines())}
    assert got["MOBODY_PREC_FP16_T64"] == _ffi.PREC["fp16_t64"] == 6
    assert got["MOBODY_PREC_FP16"] == _ffi.PREC["fp16"] == 3
    assert (got["MOBODY_TC_MAX_S"], got["MOBODY_TC_MAX_A"], got["MOBODY_TC_FP16_MAX_SAS"]) == (_ffi.TC_MAX_S, _ffi.TC_MAX_A,
                                                                                             _ffi.TC_MAX_SAS["fp16"])
    assert (got["MOBODY_TC_WIDE_MAX_S"], got["MOBODY_TC_WIDE_MAX_A"]) == (_ffi.TC_WIDE_MAX_S, _ffi.TC_WIDE_MAX_A) == (128, 32)
    assert got["MOBODY_ABI_VERSION"] == _ffi.ABI_VERSION == 2
    assert "fp16_t64" not in _ffi.ENABLED_PRECISIONS


def test_fp16_and_fp16_t64_partition_the_fp32_shapes():
    """Every (S, A) the fp32 mode takes (2 <= S <= 128, 1 <= A <= 32) is taken by exactly one of fp16 and fp16_t64;
    fp16_t64 takes exactly those outside S <= 64, A <= 16, 2S+A <= 112."""
    from mobody_b200.dynamics import tc_step_supports
    for S in range(2, 129):
        for A in range(1, 33):
            takes = [m for m in ("fp16", "fp16_t64") if tc_step_supports(S, A, m)]
            assert len(takes) == 1, (S, A, takes)
            assert (takes[0] == "fp16_t64") == (S > 64 or A > 16 or 2 * S + A > 112), (S, A)
    for S, A in ((1, 20), (129, 8), (111, 33), (64, 33), (45, 0)):
        assert not tc_step_supports(S, A, "fp16_t64"), (S, A)
    assert all(tc_step_supports(S, A, "fp16_t64") for S, A in SHAPES.values())
    assert tc_step_supports(56, 1, "fp16_t64") and not tc_step_supports(55, 2, "fp16_t64")    # 2S+A = 113 / 112


def test_the_three_bf16x2_modes_still_partition_the_fp32_shapes():
    from mobody_b200.dynamics import tc_step_supports
    for S in range(2, 129):
        for A in range(1, 33):
            takes = [m for m in ("bf16x2", "bf16x2_t64", "bf16x2_wide") if tc_step_supports(S, A, m)]
            assert len(takes) == 1, (S, A, takes)
            assert (takes[0] == "bf16x2") == (S <= 64 and A <= 16 and 2 * S + A <= 96), (S, A)
            assert (takes[0] == "bf16x2_wide") == (S > 64), (S, A)


def test_auto_is_unchanged():
    import mobody_b200 as mb
    for task, (S, A), want in (("ant-medium-v2", SHAPES["ant"], "fp32"), ("pen-human-v0", SHAPES["pen"], "fp32"),
                               ("door-human-v0", SHAPES["door"], "fp32"), ("halfcheetah-medium-v2", (17, 6), "bf16x2"),
                               ("hopper-medium-v2", (56, 1), "fp32")):
        m = mb.MOBODYModule(S, A, 256, 7, 5, device="cpu", config={"mopo": 0, "latent_reward": 0})
        d = mb.MOBODYEnsembleDynamics({}, m, None, None, mb.get_termination_fn(task), precision=None)
        assert d.precision == want, (task, d.precision)
        d = mb.MOBODYEnsembleDynamics({"b200_precision": "fp16_t64"}, m, None, None, mb.get_termination_fn(task))
        assert d.precision == "fp16_t64"


@pytest.mark.parametrize("S,A", [(17, 6), (55, 2), (27, 8), (40, 16), (48, 16), (2, 1), (129, 8), (111, 33), (64, 33)])
def test_step_rejects_shapes_outside_the_fp16_t64_range(lib, S, A):
    """fp16's shapes (2S+A = 112 at S55/A2 included) and those beyond the fp32 mode's S <= 128, A <= 32."""
    d, keep = _desc(S, A, precision=6)
    assert lib.mobody_step(ctypes.byref(d), None) == -1
    assert lib.mobody_last_error() == F16_T64_ERR


def test_step_rejects_a_missing_pack(lib):
    for S, A in (SHAPES["ant"], SHAPES["pen"]):
        d, keep = _desc(S, A, precision=6, pack=False)
        assert lib.mobody_step(ctypes.byref(d), None) == -1
        assert lib.mobody_last_error() == b"mobody_step: tensor-core precision needs dyn_pack (mobody_dyn_pack)"
        d, keep = _desc(S, A, precision=6, policy=True)
        assert lib.mobody_step(ctypes.byref(d), None) == -1
        assert lib.mobody_last_error() == b"mobody_step: fused policy needs policy_pack (mobody_mlp_pack)"


def test_existing_rejection_texts_are_unchanged(lib):
    for prec, S, A, text in ((3, 111, 8, b"mobody_step: tensor-core modes take S <= 64, A <= 16 and 2S+A <= 96 (bf16x2) / 112 (fp16)"),
                             (3, 45, 24, b"mobody_step: tensor-core modes take S <= 64, A <= 16 and 2S+A <= 96 (bf16x2) / 112 (fp16)"),
                             (1, 56, 1, b"mobody_step: tensor-core modes take S <= 64, A <= 16 and 2S+A <= 96 (bf16x2) / 112 (fp16)"),
                             (4, 45, 24, b"mobody_step: bf16x2_wide takes 65 <= S <= 128 and A <= 32"),
                             (5, 111, 8, b"mobody_step: bf16x2_t64 takes S <= 64, A <= 32 with A > 16 or 2S+A > 96")):
        d, keep = _desc(S, A, precision=prec)
        assert lib.mobody_step(ctypes.byref(d), None) == -1
        assert lib.mobody_last_error() == text


def test_packed_images_are_the_fp16_images(lib):
    for S, A in list(SHAPES.values()) + [(2, 17), (56, 1), (64, 16), (128, 32), (65, 1)]:
        assert lib.mobody_dyn_pack_bytes(S, A, 6) == lib.mobody_dyn_pack_bytes(S, A, 3) > 0
        assert lib.mobody_mlp_pack_bytes(S, A, 6) == lib.mobody_mlp_pack_bytes(S, A, 3) > 0
        assert lib.mobody_dyn_pack_bytes(S, A, 6) < lib.mobody_dyn_pack_bytes(S, A, 1)     # one plane, not bf16x2's two
