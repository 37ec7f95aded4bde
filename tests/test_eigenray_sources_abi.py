"""CPU test of the many-source eigenray entry points: geoac_eigenray_search_sources, geoac_trace_sources_paths_compact and
geoac_last_eigenray_ms are exported and refuse a NULL context before any device call."""
import ctypes as C

import numpy as np

from geoac_b200 import abi, api


def test_many_source_eigenray_entry_points_refuse_a_null_context(built_lib):
    for name in ("geoac_eigenray_search_sources", "geoac_trace_sources_paths_compact", "geoac_last_eigenray_ms"):
        assert name in api.EXPORTED_SYMBOLS and hasattr(C.CDLL(built_lib), name)
    x, s, o64 = np.zeros(64), np.zeros(64, np.int32), np.zeros(64, np.int64)
    d, i = x.ctypes.data_as(C.POINTER(C.c_double)), s.ctypes.data_as(C.POINTER(C.c_int32))
    lp = o64.ctypes.data_as(C.POINTER(C.c_int64))
    L, bad = api.lib(), abi.GEOAC_ERR_BAD_ARG
    opts = abi.GeoacEigOpts()
    assert L.geoac_default_eig_opts(C.byref(opts)) == abi.GEOAC_OK
    n_rows = C.c_int64(-5)
    assert L.geoac_eigenray_search_sources(None, C.byref(opts), 1, d, 1, i, d, 4, d, C.byref(n_rows), lp) == bad
    assert L.geoac_eigenray_search_sources(None, None, 0, None, 0, None, None, 0, None, None, None) == bad
    assert n_rows.value == -5
    assert L.geoac_trace_sources_paths_compact(None, 1, d, 1, i, d, d, d, i, i, 25, 4, 4, d, lp, 0, 0, None, None) == bad
    assert L.geoac_trace_sources_paths_compact(None, 0, None, 0, None, None, None, None, None, None, 0, 0, 0, None, None, 0, 0, None, None) == bad
    assert L.geoac_last_eigenray_ms(None, d) == bad
