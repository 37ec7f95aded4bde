"""CPU test of the ensemble entry points: geoac_set_ensemble_1d and geoac_trace_ensemble refuse a NULL context before any
device call."""
import ctypes as C

import numpy as np

from geoac_b200 import abi, api


def test_ensemble_entry_points_refuse_a_null_context(built_lib):
    x, s = np.linspace(0.0, 1.0, 64), np.zeros(64, np.int32)
    offs = np.array([0, 3], np.int64)
    d, i = x.ctypes.data_as(C.POINTER(C.c_double)), s.ctypes.data_as(C.POINTER(C.c_int32))
    o = offs.ctypes.data_as(C.POINTER(C.c_int64))
    L, bad = api.lib(), abi.GEOAC_ERR_BAD_ARG
    assert L.geoac_set_ensemble_1d(None, 1, o, d, d, d, d, d) == bad
    assert L.geoac_set_ensemble_1d(None, 0, None, None, None, None, None, None) == bad
    assert L.geoac_trace_ensemble(None, 1, i, d, d, d, i, i) == bad
    assert L.geoac_trace_ensemble(None, 0, None, None, None, None, None, None) == bad
