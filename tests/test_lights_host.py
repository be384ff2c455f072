"""The device-built light list without a GPU: rtx_collect_emissive_triangles and rtx_read_emissive_triangles reject a null context
before any device work."""
import ctypes as C

import numpy as np


def test_light_list_calls_with_a_null_context_fail_before_touching_a_device(rtdx):
    lib = rtdx.load_library()
    n = C.c_uint32(7)
    out = np.zeros(2, dtype=rtdx.light_dt)
    for call in (lambda: lib.rtx_collect_emissive_triangles(None, C.byref(n)),
                 lambda: lib.rtx_collect_emissive_triangles(None, None),
                 lambda: lib.rtx_read_emissive_triangles(None, out.ctypes.data_as(C.c_void_p), out.size, C.byref(n)),
                 lambda: lib.rtx_read_emissive_triangles(None, None, 0, None)):
        assert call() == 1
        assert b"null context" in lib.rtx_last_error()
    assert n.value == 7
