"""mobody_step refuses, before any launch, a shape whose statistics scratch cannot hold one member's squared deviations.

The single-pass bf16 diagnostic mode (code 2) falls back to the one-tile kernel when two row tiles do not fit; at S = 64
that kernel's single operand plane holds the tile's next states and member picks but no member batch, so the statistics
loop would never advance.  The descriptor carries fake device pointers: the refusal happens on the host, before any
launch, but if the refusal ever regressed the call would launch a kernel on them.  So the test runs only where no CUDA
device is present (there a launch cannot happen and the call fails with a CUDA error instead).
"""
import ctypes as C

import pytest
import torch

PREC_BF16, ERR_UNSUPPORTED = 2, -2


@pytest.mark.skipif(torch.cuda.is_available(), reason="fake device pointers: run only where nothing can be launched")
def test_bf16_one_tile_fallback_refuses_S64():
    import __graft_entry__ as g
    g.build()
    from mobody_b200 import _ffi
    L = _ffi.lib()
    dp, fake = _ffi.DynParams(), 0x1000
    for i in range(_ffi.N_DYN_LAYERS):
        dp.w[i], dp.b[i] = fake, fake
    d = _ffi.StepDesc()
    d.precision, d.B, d.S, d.A = PREC_BF16, 1000, 64, 16
    d.obs = d.act = d.idx = d.dyn_pack = d.next_obs = d.reward = d.penalty = d.terminal = d.mean = fake
    d.dyn = C.pointer(dp)
    assert L.mobody_step(C.byref(d), None) == ERR_UNSUPPORTED
    assert b"statistics scratch" in L.mobody_last_error()
