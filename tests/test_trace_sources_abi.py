"""CPU test of geoac_trace_sources' C entry point: a NULL context is refused before any device call."""
import ctypes as C

import numpy as np

from geoac_b200 import abi, api


def test_trace_sources_refuses_a_null_context(built_lib):
    x, s = np.zeros(64), np.zeros(64, np.int32)
    d, i = x.ctypes.data_as(C.POINTER(C.c_double)), s.ctypes.data_as(C.POINTER(C.c_int32))
    L, bad = api.lib(), abi.GEOAC_ERR_BAD_ARG
    assert L.geoac_trace_sources(None, 1, d, 1, i, d, d, d, i, i) == bad
    assert L.geoac_trace_sources(None, 0, None, 0, None, None, None, None, None, None) == bad
