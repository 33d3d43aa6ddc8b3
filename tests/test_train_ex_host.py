"""CPU checks of mobody_train_step_ex's C-ABI boundary: the struct mirror, argument rejections, workspace sizes."""
import ctypes
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "mobody_b200.h")


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from mobody_b200 import _ffi
    return _ffi.lib()


def test_ex_desc_layout_matches_header_via_gcc(lib, tmp_path):
    from mobody_b200 import _ffi
    ct, cname = _ffi.TrainExDesc, "mobody_train_ex_desc"
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             f'printf("{cname} %zu\\n", sizeof({cname}));']
    lines += [f'printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));' for f, _ in ct._fields_]
    lines += ['return 0;}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    assert int(got[cname]) == ctypes.sizeof(ct)
    for f, _ in ct._fields_:
        assert int(got[f"{cname}.{f}"]) == getattr(ct, f).offset, f


def _valid_desc():
    """A descriptor that passes every host-side check (dummy non-null pointers: the rejections below come before any launch)."""
    from mobody_b200 import _ffi
    x = _ffi.TrainExDesc()
    d = x.base
    d.rows, d.N, d.n_true, d.S, d.A = 16, 64, 32, 17, 6
    d.row_width = _ffi.lib().mobody_row_width(17, 6)
    for name in ("policy", "q1", "q2", "q1_target", "q2_target", "policy_m", "policy_v", "q1_m", "q1_v", "q2_m", "q2_v"):
        st = getattr(d, name)
        for i in range(3):
            st.w[i], st.b[i] = 16, 16
    d.t_q = d.t_pi = 1
    x.advantage, x.scale_q, x.q_weighted = 1, 1, 1
    for name in ("value", "value_m", "value_v"):
        st = getattr(x, name)
        for i in range(3):
            st.w[i], st.b[i] = 16, 16
    x.t_v = 1
    return x


@pytest.mark.parametrize("field,value,msg", [
    ("advantage", 2, b"advantage / scale_q / q_weighted must be 0 or 1"),
    ("scale_q", -1, b"advantage / scale_q / q_weighted must be 0 or 1"),
    ("q_weighted", 3, b"advantage / scale_q / q_weighted must be 0 or 1"),
    ("value", None, b"advantage=1 needs the value function and its Adam moments"),
    ("value_m", None, b"advantage=1 needs the value function and its Adam moments"),
    ("value_v", None, b"advantage=1 needs the value function and its Adam moments"),
    ("t_v", 0, b"the value optimiser step count is 1-based"),
])
def test_ex_argument_errors(lib, field, value, msg):
    x = _valid_desc()
    if value is None:
        getattr(x, field).b[2] = None                               # one null pointer of the MLP state
    else:
        setattr(x, field, value)
    assert lib.mobody_train_step_ex(ctypes.byref(x), None) == -1
    assert lib.mobody_last_error() == b"mobody_train_step_ex: " + msg


def test_ex_value_state_is_optional_without_advantage_and_base_checks_apply(lib):
    x = _valid_desc()
    x.advantage, x.t_v = 0, 0
    x.value.w[0] = None
    x.base.row_width += 4                                          # the base checks still run, under the ex name
    assert lib.mobody_train_step_ex(ctypes.byref(x), None) == -1
    assert lib.mobody_last_error() == b"mobody_train_step_ex: row_width does not match (S, A)"
    assert lib.mobody_train_step_ex(None, None) == -1 and b"null descriptor" in lib.mobody_last_error()


def test_ex_workspace_bytes(lib):
    for S, A in ((17, 6), (111, 8), (128, 32)):
        sizes = [lib.mobody_train_ex_workspace_bytes(N, S, A, 4) for N in (1, 77, 320, 1279, 1280, 1500, 10240)]
        assert all(b > a for a, b in zip(sizes, sizes[1:])), (S, A, sizes)
        assert lib.mobody_train_ex_workspace_bytes(320, S, A, 4) > lib.mobody_train_workspace_bytes(320, S, A, 4) > 0
    assert lib.mobody_train_ex_workspace_bytes(0, 17, 6, 1) == 0
