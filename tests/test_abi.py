"""CPU tests of the drop-in boundary: the C-ABI library builds for sm_100a, loads, exports every symbol declared in
include/geoac_b200.h, and REFUSES to run without a B200 (no CPU fallback).  No compute calls here."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from geoac_b200 import abi, api
from tests import util

HDR = os.path.join(util.ROOT, "include", "geoac_b200.h")


def declared_symbols():
    txt = open(HDR).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(geoac_[a-z0-9_]+)\s*\(", txt)))


def test_header_and_binding_agree():
    assert declared_symbols() == sorted(api.EXPORTED_SYMBOLS)


def test_library_exports_every_declared_symbol(built_lib):
    lib = C.CDLL(built_lib)
    for s in declared_symbols():
        assert hasattr(lib, s), f"{s} declared in include/geoac_b200.h but not exported"


def test_params_struct_layout_matches_header():
    # 15 doubles + 4 int32 = 136 bytes, no padding
    assert C.sizeof(abi.GeoacParams) == 15 * 8 + 4 * 4
    p = api.default_params(abi.GEOAC_GLOBAL) if os.path.exists(api.library_path()) else None
    if p is not None:
        assert p.ray_limit == 10000.0 and p.ds_min == 0.001 and p.bounces == 2 and p.calc_amp == 1
        assert abs(p.src[1] - 30.0 * util.PI / 180.0) < 1e-15


def test_defaults_match_reference_parameters(built_lib):
    p2, p3 = api.default_params(abi.GEOAC_2D), api.default_params(abi.GEOAC_3D)
    assert (p3.ds_min, p3.ds_max, p3.ray_limit) == (0.001, 0.5, 5000.0)       # GeoAc.Parameters.cpp:20-24
    assert p2.accum_per_segment == 1 and p3.accum_per_segment == 0            # SURVEY App. A-2
    assert (p3.freq, p3.tweak_abs, p3.z_grnd) == (0.1, 0.3, 0.0)
    for v, (a, n) in {abi.GEOAC_2D: (6, 3), abi.GEOAC_3D: (12, 4), abi.GEOAC_GLOBAL: (18, 6)}.items():
        assert api.lib().geoac_eq_count(v, 1) == a and api.lib().geoac_eq_count(v, 0) == n


def test_host_loader_matches_oracle_loader(built_lib, oracle):
    for glob in (False, True):
        a = api.load_met_1d(util.TOY, global_taper=glob)
        b = oracle.load_met_1d(util.TOY, global_taper=glob)
        for x, y in zip(a, b):
            assert np.array_equal(x, y)
    assert len(a[0]) == 1400


def test_grid_loader_matches_oracle_loader_and_fixture(built_lib, oracle, tmp_path):
    """geoac_load_met_grid (product host code) == oracle loader == the committed grid fixture, bit for bit, for both variants."""
    from tests.golden import make_grid
    files = make_grid.write_cartesian(str(tmp_path / "c"), np.arange(-500.0, 501.0, 200.0), np.arange(-450.0, 451.0, 150.0))
    a, b = api.load_met_grid(*files), oracle.load_met_grid(*files)
    fix = np.load(os.path.join(util.GOLD, "grid_cart.npz"))
    for x, y, k in zip(a, b, ("ax0", "ax1", "axz", "T", "u", "v", "rho")):
        assert np.array_equal(x, y) and np.array_equal(x, fix[k])
    files = make_grid.write_global(str(tmp_path / "g"), np.arange(20.0, 51.0, 6.0), np.arange(-15.0, 16.0, 5.0))
    a, b = api.load_met_grid(*files, is_global=True), oracle.load_met_grid(*files, is_global=True)
    fix = np.load(os.path.join(util.GOLD, "grid_glob.npz"))
    for x, y, k in zip(a, b, ("ax0", "ax1", "axz", "T", "u", "v", "rho")):
        assert np.array_equal(x, y) and np.array_equal(x, fix[k])


def test_prop_angles_reproduce_the_mains_loops():
    th_deg, ph_deg, th, ph = api.prop_angles(0.5, 45.0, 0.5, -90.0, -90.0, 1.0)       # GeoAc2D defaults: 90 rays
    assert len(th) == 90 and th_deg[0] == 0.5 and ph_deg[0] == -90.0
    d, _ = util.load_case("2d_config1")
    assert np.array_equal(th_deg, d["theta_deg"])
    # config 2 grid: 60 x 3600 (SURVEY 8d)
    th_deg, ph_deg, _, _ = api.prop_angles(1, 60.5, 1, 0, 359.95, 0.1)
    assert len(th_deg) == 60 * 3600


def test_no_cpu_fallback(built_lib):
    """Without a CUDA device the library must fail loudly, not compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(api.GeoAcError) as e:
        api.Tracer(abi.GEOAC_3D, 0)
    assert "no CUDA device" in str(e.value) or "failed (1)" in str(e.value)


def test_synthetic_grids_match_their_node_files(built_lib, tmp_path):
    """bench.py builds the config 4 / 5 atmospheres in memory (geoac_b200/synth.py); the golden vectors trace the same
    formulas through .met node files and the reference's loader.  The two must agree to the files' text precision, so the
    parity shown on the file-based cases carries over to the in-memory grids the full-size runs use."""
    from geoac_b200 import synth
    xs, ys = np.arange(-500.0, 501.0, 250.0), np.arange(-500.0, 501.0, 200.0)
    files = synth.write_config4_files(str(tmp_path / "c4"), xs, ys, nz=40)
    got = api.load_met_grid(*files, is_global=False)
    want = synth.config4_grid(nz=40, x=xs, y=ys)
    lats, lons = np.arange(25.0, 46.0, 5.0), np.arange(-12.0, 13.0, 4.0)
    files5 = synth.write_config5_files(str(tmp_path / "c5"), lats, lons, nz=40)
    got5 = api.load_met_grid(*files5, is_global=True)
    want5 = synth.config5_grid(nr=40, lat_deg=lats, lon_deg=lons)
    for g_, w_ in ((got, want), (got5, want5)):
        names = ("ax0", "ax1", "axz", "T", "u", "v", "rho")
        atol = dict(ax0=1e-6, ax1=1e-6, axz=1e-9, T=1e-6, u=2e-9, v=2e-9)        # %.6f text: 5e-7 in file units (winds m/s -> km/s)
        for nm, a, b in zip(names, g_, w_):
            a, b = np.asarray(a), np.asarray(b)
            assert a.shape == b.shape, nm
            if nm == "rho":
                assert np.allclose(a, b, rtol=2e-6, atol=0.0), nm                   # %.6e text
            else:
                assert np.allclose(a, b, rtol=0.0, atol=atol[nm]), (nm, float(np.abs(a - b).max()))


def test_trace_entry_points_refuse_a_null_context(built_lib):
    """geoac_trace, geoac_trace_paths(_compact), geoac_reserve and geoac_trace_multi return GEOAC_ERR_BAD_ARG for a NULL
    context (or a NULL entry of the context list) before any device call."""
    L, bad = api.lib(), abi.GEOAC_ERR_BAD_ARG
    x, s, o = np.zeros(64), np.zeros(64, np.int32), np.zeros(2, np.int64)
    d, i, l = (a.ctypes.data_as(C.POINTER(t)) for a, t in ((x, C.c_double), (s, C.c_int32), (o, C.c_int64)))
    assert L.geoac_trace(None, 1, d, d, d, i, i) == bad
    assert L.geoac_trace_paths(None, 1, d, d, d, i, i, 25, 4, d, i, 2, d, i) == bad
    assert L.geoac_trace_paths_compact(None, 1, d, d, d, i, i, 25, 4, 4, d, l, 2, 2, d, l) == bad
    assert L.geoac_reserve(None, 1) == bad
    assert L.geoac_trace_multi(None, 1, 1, d, d, d, i, i) == bad
    assert L.geoac_trace_multi((C.c_void_p * 2)(), 2, 1, d, d, d, i, i) == bad


def test_pinned_host_allocation_binding(built_lib):
    """geoac_host_alloc / geoac_host_free: NULL (and a GeoAcError from the wrapper) without a device, a usable buffer with one."""
    p = api.lib().geoac_host_alloc(4096)
    if p:                                   # a GPU box
        api.lib().geoac_host_free(p)
        a = api.PinnedArray((4, 8), np.int32)
        a.array[:] = 7
        assert a.array.sum() == 7 * 32 and a.array.flags["WRITEABLE"] and a.array.flags["C_CONTIGUOUS"]
        a.close()
    else:
        with pytest.raises(api.GeoAcError):
            api.PinnedArray((4, 8), np.int32)
    api.lib().geoac_host_free(None)         # no-op
    assert not api.lib().geoac_host_alloc(0)
