"""Host side of the restricted decoder: the plan wrappers keep their destructors, and the new C-ABI entry points refuse
bad arguments before touching the device."""
import ctypes as C

import pytest


def test_plan_wrappers_release_their_native_handles():
    from dram_b200 import ops

    for cls in (ops.Conv3dPlan, ops.Upsample2xPlan):
        assert "__del__" in cls.__dict__, cls.__name__
    assert callable(ops.decoder_support)


@pytest.mark.parametrize("call", [
    lambda lib, n: lib.dram_decoder_support(None, 1, 8, 8, 8, 4, 4, 4, None, None, None),
    lambda lib, n: lib.dram_decoder_support(C.c_void_p(16), 1, 8, 8, 8, 9, 4, 4, C.c_void_p(16), C.c_void_p(16), None),
    lambda lib, n: lib.dram_conv3d_worklist_size(None, C.byref(n)),
    lambda lib, n: lib.dram_conv3d_worklist(None, None, 0, None, None, None, None),
    lambda lib, n: lib.dram_conv3d_run_listed(None, None, None, 0, None),
    lambda lib, n: lib.dram_upsample2x_worklist_size(None, C.byref(n)),
    lambda lib, n: lib.dram_upsample2x_worklist(None, None, 0, None, None, None, None),
    lambda lib, n: lib.dram_upsample2x_plan_run_listed(None, None, None, 0, None),
])
def test_worklist_entry_points_refuse_bad_arguments(lib, call):
    from dram_b200 import _capi

    assert call(lib, C.c_int32()) != _capi.DRAM_OK
    assert _capi.last_error()
