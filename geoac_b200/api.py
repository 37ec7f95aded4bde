"""Host-side mirror of the reference's `-prop` interface on top of the C ABI (include/geoac_b200.h).

The product path is: Python (or the C++ front ends) -> libgeoac_b200.so (extern "C") -> sm_100a CUDA kernels.
There is no CPU implementation behind this module: if the library is missing or no B200 is present, it raises.
Reference call sites this replaces: Code/GeoAc3D_main.cpp:226-304 and the four sibling mains.
"""
import ctypes as C
import os

import numpy as np

from . import abi
from .abi import GeoacParams

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_LIB = None


class GeoAcError(RuntimeError):
    pass


def library_path():
    """The product library; GEOAC_B200_LIB names an experimental build in the same directory (A/B measurements only)."""
    name = os.environ.get("GEOAC_B200_LIB", "libgeoac_b200.so")
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), "_lib", os.path.basename(name))


def lib():
    """Load libgeoac_b200.so (built by geoac_b200.build.build()); fail loudly if it is absent."""
    global _LIB
    if _LIB is None:
        path = library_path()
        if not os.path.exists(path):
            raise GeoAcError(f"{path} not found: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
                             "There is no CPU fallback.")
        L = C.CDLL(path)
        L.geoac_create.restype = C.c_void_p
        L.geoac_create.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_int)]
        L.geoac_destroy.argtypes = [C.c_void_p]
        L.geoac_last_error.restype = C.c_char_p
        L.geoac_last_error.argtypes = [C.c_void_p]
        L.geoac_default_params.argtypes = [C.c_int, C.POINTER(GeoacParams)]
        L.geoac_set_atmosphere_1d.argtypes = [C.c_void_p, C.c_int, _dp, _dp, _dp, _dp, _dp]
        L.geoac_set_atmosphere_3d.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp]
        L.geoac_get_params.argtypes = [C.c_void_p, C.POINTER(GeoacParams)]
        L.geoac_set_params.argtypes = [C.c_void_p, C.POINTER(GeoacParams)]
        L.geoac_trace.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, _dp, _ip, _ip]
        L.geoac_trace_paths.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, _dp, _ip, _ip, C.c_int, C.c_int64, _dp, _ip, C.c_int64, _dp, _ip]
        _lp = C.POINTER(C.c_int64)
        L.geoac_trace_paths_compact.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, _dp, _ip, _ip, C.c_int, C.c_int64, C.c_int64, _dp, _lp,
                                                C.c_int64, C.c_int64, _dp, _lp]
        L.geoac_trace_sources.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int64, _ip, _dp, _dp, _dp, _ip, _ip]
        L.geoac_trace_sources_paths_compact.argtypes = [C.c_void_p, C.c_int, _dp, C.c_int64, _ip, _dp, _dp, _dp, _ip, _ip,
                                                        C.c_int, C.c_int64, C.c_int64, _dp, _lp, C.c_int64, C.c_int64, _dp, _lp]
        L.geoac_set_ensemble_1d.argtypes = [C.c_void_p, C.c_int, _lp, _dp, _dp, _dp, _dp, _dp]
        L.geoac_trace_ensemble.argtypes = [C.c_void_p, C.c_int64, _ip, _dp, _dp, _dp, _ip, _ip]
        L.geoac_trace_device.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.geoac_reserve.argtypes = [C.c_void_p, C.c_int64]
        L.geoac_host_alloc.restype = C.c_void_p
        L.geoac_host_alloc.argtypes = [C.c_size_t]
        L.geoac_host_free.restype = None
        L.geoac_host_free.argtypes = [C.c_void_p]
        L.geoac_last_trace_stats.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_double)]
        L.geoac_load_met_1d.argtypes = [C.c_char_p, C.c_char_p, C.c_double, C.c_int, C.c_int, C.POINTER(C.c_int), _dp, _dp, _dp, _dp, _dp]
        L.geoac_load_met_grid.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), _dp, _dp, _dp, _dp, _dp, _dp, _dp]
        L.geoac_eq_count.argtypes = [C.c_int, C.c_int]
        L.geoac_last_trace_counters.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.geoac_selftest_math.argtypes = [C.c_void_p, C.c_int, _dp]
        L.geoac_get_grid_tables.argtypes = [C.c_void_p, C.c_int64, _dp, C.c_int64, _dp]
        L.geoac_default_eig_opts.argtypes = [C.POINTER(abi.GeoacEigOpts)]
        L.geoac_eigenray_search.argtypes = [C.c_void_p, C.POINTER(abi.GeoacEigOpts), C.c_int, _dp, C.c_int64, _dp,
                                            C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.geoac_eigenray_direct.argtypes = [C.c_void_p, C.POINTER(abi.GeoacEigOpts), C.c_int, _dp, _dp, _dp, C.POINTER(C.c_int64)]
        L.geoac_eigenray_search_sources.argtypes = [C.c_void_p, C.POINTER(abi.GeoacEigOpts), C.c_int, _dp, C.c_int, _ip, _dp, C.c_int64, _dp,
                                                    C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.geoac_last_eigenray_ms.argtypes = [C.c_void_p, _dp]
        L.geoac_get_variant.argtypes = [C.c_void_p]
        L.geoac_source_state.argtypes = [C.c_void_p, _dp]
        L.geoac_sample_atmosphere.argtypes = [C.c_void_p, C.c_int64, _dp, _dp, _dp, _dp]
        L.geoac_set_knob.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
        L.geoac_last_schedule.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.geoac_last_launch_ms.argtypes = [C.c_void_p, _dp]
        L.geoac_get_costs.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_uint32)]
        _cp = C.POINTER(C.c_void_p)
        L.geoac_create_multi.argtypes = [C.c_int, C.POINTER(C.c_int), C.c_int, _cp, C.POINTER(C.c_int)]
        L.geoac_multi_set_atmosphere_1d.argtypes = [_cp, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp]
        L.geoac_multi_set_atmosphere_3d.argtypes = [_cp, C.c_int, C.c_int, C.c_int, C.c_int, _dp, _dp, _dp, _dp, _dp, _dp, _dp]
        L.geoac_multi_set_params.argtypes = [_cp, C.c_int, C.POINTER(GeoacParams)]
        L.geoac_trace_multi.argtypes = [_cp, C.c_int, C.c_int64, _dp, _dp, _dp, _ip, _ip]
        L.geoac_measure_fp64_peak.restype = C.c_double
        L.geoac_measure_fp64_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
        _LIB = L
    return _LIB


EXPORTED_SYMBOLS = [
    "geoac_create", "geoac_destroy", "geoac_last_error", "geoac_default_params", "geoac_set_atmosphere_1d",
    "geoac_set_atmosphere_3d", "geoac_get_params", "geoac_set_params", "geoac_trace", "geoac_trace_paths", "geoac_trace_device",
    "geoac_trace_sources", "geoac_set_ensemble_1d", "geoac_trace_ensemble", "geoac_trace_sources_paths_compact",
    "geoac_eigenray_search_sources", "geoac_last_eigenray_ms",
    "geoac_reserve", "geoac_last_trace_stats", "geoac_last_trace_counters", "geoac_selftest_math", "geoac_load_met_1d", "geoac_load_met_grid", "geoac_eq_count", "geoac_measure_fp64_peak",
    "geoac_get_grid_tables", "geoac_default_eig_opts", "geoac_eigenray_search", "geoac_eigenray_direct", "geoac_get_variant", "geoac_source_state",
    "geoac_sample_atmosphere",
    "geoac_set_knob", "geoac_last_schedule", "geoac_last_launch_ms", "geoac_trace_paths_compact", "geoac_get_costs",
    "geoac_host_alloc", "geoac_host_free",
    "geoac_create_multi", "geoac_multi_set_atmosphere_1d", "geoac_multi_set_atmosphere_3d", "geoac_multi_set_params", "geoac_trace_multi",
]


def _p(a):
    return a.ctypes.data_as(_dp)


def load_met_1d(path, fmt="zTuvdp", z_grnd_taper=0.0, global_taper=False, cap=200000):
    """Load_G2S mirror (reference Code/Atmo/G2S_Spline1D.cpp:109-142): returns z, T, u, v, rho (winds tapered, km/s)."""
    arrs = [np.zeros(cap) for _ in range(5)]
    n = C.c_int(0)
    rc = lib().geoac_load_met_1d(os.fsencode(path), fmt.encode(), z_grnd_taper, int(global_taper), cap, C.byref(n), *[_p(a) for a in arrs])
    if rc != abi.GEOAC_OK:
        raise GeoAcError(f"geoac_load_met_1d({path}) failed with status {rc}")
    return [a[: n.value].copy() for a in arrs]


def load_met_grid(prefix, loc0, loc1, fmt="zTuvdp", is_global=False):
    """Load_G2S_Multi mirror (reference Code/Atmo/G2S_MultiDimSpline3D.cpp:139-189): returns ax0, ax1, axz, T, u, v, rho with
    fields shaped [n0][n1][nz] (winds tapered, km/s; Global node coordinates in radians)."""
    n0g = len(open(loc0).read().split())
    n1g = len(open(loc1).read().split())
    nzg = sum(1 for _ in open(f"{prefix}0.met"))
    ax0, ax1, axz = np.zeros(n0g), np.zeros(n1g), np.zeros(nzg)
    fields = [np.zeros(n0g * n1g * nzg) for _ in range(4)]
    n0, n1, nz = C.c_int(0), C.c_int(0), C.c_int(0)
    rc = lib().geoac_load_met_grid(os.fsencode(prefix), os.fsencode(loc0), os.fsencode(loc1), fmt.encode(), int(is_global), n0g, n1g, nzg,
                                   C.byref(n0), C.byref(n1), C.byref(nz), _p(ax0), _p(ax1), _p(axz), *[_p(f) for f in fields])
    if rc != abi.GEOAC_OK or (n0.value, n1.value, nz.value) != (n0g, n1g, nzg):
        raise GeoAcError(f"geoac_load_met_grid({prefix}) failed with status {rc}")
    return [ax0, ax1, axz] + [f.reshape(n0g, n1g, nzg) for f in fields]


class PinnedArray:
    """A numpy array on page-locked host memory from geoac_host_alloc (the buffers a C++ front end would hand to geoac_trace):
    `.array` is the view; the memory is released by close() / when the object is collected -- keep it alive while the view is used."""

    def __init__(self, shape, dtype=np.float64):
        dt = np.dtype(dtype)
        n = int(np.prod(shape, dtype=np.int64))
        self._nbytes = max(1, n * dt.itemsize)
        self._p = lib().geoac_host_alloc(self._nbytes)
        if not self._p:
            raise GeoAcError(f"geoac_host_alloc({self._nbytes}) failed (no CUDA device or out of page-locked memory)")
        buf = (C.c_char * self._nbytes).from_address(self._p)
        self.array = np.frombuffer(buf, dtype=dt, count=n).reshape(shape)

    def close(self):
        if getattr(self, "_p", None):
            self.array = None
            lib().geoac_host_free(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def default_params(variant):
    p = GeoacParams()
    lib().geoac_default_params(variant, C.byref(p))
    return p


def prop_angles(theta_min, theta_max, theta_step, phi_min, phi_max, phi_step):
    """Enumerate launch angles exactly like the mains' loops `for(double a=min; a<=max; a+=step)` (phi outer, theta
    inner; reference Code/GeoAc3D_main.cpp:226-229) and convert to the radians stored in GeoAc_theta/GeoAc_phi."""
    Pi = 3.141592653589793238462643
    thetas, phis = [], []
    t = float(theta_min)
    while t <= theta_max:
        thetas.append(t)
        t += theta_step
    p = float(phi_min)
    while p <= phi_max:
        phis.append(p)
        p += phi_step
    th = np.tile(np.array(thetas), len(phis))
    ph = np.repeat(np.array(phis), len(thetas))
    return th, ph, th * Pi / 180.0, Pi / 2.0 - ph * Pi / 180.0


class Tracer:
    """One context = one variant on one GPU (geoac_create ... geoac_destroy)."""

    def __init__(self, variant, device=0):
        st = C.c_int(0)
        self._h = lib().geoac_create(variant, device, C.byref(st))
        if not self._h:
            raise GeoAcError(f"geoac_create failed ({st.value}): {lib().geoac_last_error(None).decode()}")
        self.variant = variant
        self.device = device

    def close(self):
        if getattr(self, "_h", None):
            lib().geoac_destroy(self._h)
            self._h = None

    __del__ = close

    def _check(self, rc, what):
        if rc != abi.GEOAC_OK:
            raise GeoAcError(f"{what} failed ({rc}): {lib().geoac_last_error(self._h).decode()}")

    def set_knob(self, name, value):
        """Tuning / experiment knob of this context (include/geoac_b200.h: geoac_set_knob)."""
        self._check(lib().geoac_set_knob(self._h, name.encode(), int(value)), f"geoac_set_knob({name})")

    def set_atmosphere_1d(self, z, T, u, v, rho):
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (z, T, u, v, rho)]
        if any(a.ndim != 1 or a.shape != arrs[0].shape for a in arrs):
            raise GeoAcError("set_atmosphere_1d: z, T, u, v, rho must be 1-D arrays of one length")
        self._check(lib().geoac_set_atmosphere_1d(self._h, len(arrs[0]), *[_p(a) for a in arrs]), "geoac_set_atmosphere_1d")

    def set_ensemble_1d(self, members):
        """An ensemble of stratified profiles, next to the context's own atmosphere: members is a list of (z, T, u, v, rho), each
        in the form set_atmosphere_1d takes (include/geoac_b200.h: geoac_set_ensemble_1d)."""
        members = [[np.ascontiguousarray(a, dtype=np.float64) for a in m] for m in members]
        if not members or any(len(m) != 5 or any(a.ndim != 1 or a.shape != m[0].shape for a in m) for m in members):
            raise GeoAcError("set_ensemble_1d: members must be a non-empty list of (z, T, u, v, rho), 1-D arrays of one length each")
        offs = np.zeros(len(members) + 1, dtype=np.int64)
        offs[1:] = np.cumsum([len(m[0]) for m in members])
        cols = [np.ascontiguousarray(np.concatenate([m[k] for m in members])) for k in range(5)]
        self._check(lib().geoac_set_ensemble_1d(self._h, len(members), offs.ctypes.data_as(C.POINTER(C.c_int64)), *[_p(a) for a in cols]),
                    "geoac_set_ensemble_1d")

    def set_atmosphere_3d(self, ax0, ax1, axz, T, u, v, rho):
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (ax0, ax1, axz, T, u, v, rho)]
        nodes = len(arrs[0]) * len(arrs[1]) * len(arrs[2])
        if any(a.ndim != 1 for a in arrs[:3]) or any(a.size != nodes for a in arrs[3:]):
            raise GeoAcError(f"set_atmosphere_3d: fields must hold n0*n1*nz = {nodes} values ([n0][n1][nz], z fastest)")
        self._check(lib().geoac_set_atmosphere_3d(self._h, len(arrs[0]), len(arrs[1]), len(arrs[2]), *[_p(a) for a in arrs]),
                    "geoac_set_atmosphere_3d")

    @staticmethod
    def _eig_opts(opts):
        o = abi.GeoacEigOpts()
        lib().geoac_default_eig_opts(C.byref(o))
        for k, v in opts.items():
            if not hasattr(o, k):
                raise TypeError(f"unknown eigenray option {k}")
            setattr(o, k, v)
        return o

    def eigenray_search(self, receivers, cap_rows=4096, **opts):
        """GeoAc3D[.RngDep] -eig_search for one source (params.src) and many receivers [(x, y) km]: rows [n][EIG_NF] (one per
        GeoAc_EstimateEigenray call of the reference, include/geoac_b200.h) and stats {rounds, rays, found}.
        opts: theta_min, theta_max, bnc_min, bnc_max, iterations, azimuth_err_lim, d_theta_big, d_theta_small, tolerance."""
        o = self._eig_opts(opts)
        rc = np.ascontiguousarray(receivers, dtype=np.float64).reshape(-1, 2)
        rows = np.zeros((cap_rows, abi.EIG_NF))
        n = C.c_int64(0)
        stats = (C.c_int64 * 3)()
        self._check(lib().geoac_eigenray_search(self._h, C.byref(o), len(rc), _p(rc), cap_rows, _p(rows), C.byref(n), stats),
                    "geoac_eigenray_search")
        return rows[:n.value].copy(), {"rounds": stats[0], "rays": stats[1], "found": stats[2]}

    def eigenray_direct(self, receivers, estimates, **opts):
        """-eig_direct: LM search from caller-supplied estimates [(theta_est, phi_est (deg from the x axis), bounces)], one per
        receiver entry; rows as eigenray_search."""
        o = self._eig_opts(opts)
        rc = np.ascontiguousarray(receivers, dtype=np.float64).reshape(-1, 2)
        est = np.ascontiguousarray(estimates, dtype=np.float64).reshape(-1, 3)
        assert len(rc) == len(est)
        rows = np.zeros((len(rc), abi.EIG_NF))
        stats = (C.c_int64 * 3)()
        self._check(lib().geoac_eigenray_direct(self._h, C.byref(o), len(rc), _p(rc), _p(est), _p(rows), stats), "geoac_eigenray_direct")
        return rows, {"rounds": stats[0], "rays": stats[1], "found": stats[2]}

    def eigenray_search_sources(self, src, src_id, receivers, cap_rows=None, **opts):
        """eigenray_search() from many sources in one call: search i runs from src[src_id[i]] to receivers[i].  src: [n_src, 3],
        Cartesian (x, y, z) [km], Global (altitude [km], lat [deg], lon [deg]); src_id: int32 [n]; receivers: [n, 2] as for
        eigenray_search.  Rows as eigenray_search's with column 0 the search index; search i's rows equal those of
        eigenray_search([receivers[i]]) from its source (include/geoac_b200.h: geoac_eigenray_search_sources).
        cap_rows: row capacity (default: an estimate; grown and retried once if the library reports it too small)."""
        o = self._eig_opts(opts)
        src = np.ascontiguousarray(src, dtype=np.float64)
        if src.ndim != 2 or src.shape[1] != 3:
            raise GeoAcError("eigenray_search_sources: src must be an array of shape [n_src, 3]")
        rc = np.ascontiguousarray(receivers, dtype=np.float64).reshape(-1, 2)
        src_id = np.asarray(src_id)
        if src_id.dtype != np.int32 or src_id.shape != (len(rc),):
            raise GeoAcError("eigenray_search_sources: src_id must be an int32 array with one entry per receiver")
        src_id = np.ascontiguousarray(src_id)
        if cap_rows is None:
            cap_rows = max(1, len(rc) * (o.bnc_max - o.bnc_min + 1) * 8)
        n = C.c_int64(0)
        stats = (C.c_int64 * 3)()
        for attempt in range(2):
            rows = np.zeros((max(cap_rows, 1), abi.EIG_NF))
            st = lib().geoac_eigenray_search_sources(self._h, C.byref(o), len(src), _p(src), len(rc), src_id.ctypes.data_as(_ip), _p(rc),
                                                     cap_rows, _p(rows), C.byref(n), stats)
            if st == abi.GEOAC_ERR_TOO_LARGE and attempt == 0 and n.value > cap_rows:
                cap_rows = int(n.value)
                continue
            self._check(st, "geoac_eigenray_search_sources")
            break
        return rows[:n.value].copy(), {"rounds": stats[0], "rays": stats[1], "found": stats[2]}

    def last_eigenray_ms(self):
        """Where the time of the last eigenray search went [ms]: host replay of the searches, kernel time of its traces, the call."""
        ms = np.zeros(3)
        self._check(lib().geoac_last_eigenray_ms(self._h, _p(ms)), "geoac_last_eigenray_ms")
        return {"replay_ms": float(ms[0]), "kernel_ms": float(ms[1]), "call_ms": float(ms[2])}

    def source_state(self):
        """c, u, v, rho at the source point as the kernels sample them."""
        out = np.zeros(4)
        self._check(lib().geoac_source_state(self._h, _p(out)), "geoac_source_state")
        return out

    def sample_atmosphere(self, p0, p1, p2):
        """The atmosphere as the kernels evaluate it at n points in the variant's coordinates ((x, y, z) [km], or Global
        (r [km from the Earth's centre], lat [rad], lon [rad])): array [ATM_NF, n] (rows: abi.ATM_*)."""
        pts = [np.ascontiguousarray(a, dtype=np.float64) for a in (p0, p1, p2)]
        if any(a.ndim != 1 or a.shape != pts[0].shape for a in pts):
            raise GeoAcError("sample_atmosphere: p0, p1, p2 must be 1-D arrays of one length")
        n = len(pts[0])
        out = np.empty((abi.ATM_NF, n))
        self._check(lib().geoac_sample_atmosphere(self._h, n, *[_p(a) for a in pts], _p(out)), "geoac_sample_atmosphere")
        return out

    def grid_tables(self, n0, n1, nz):
        """Test hook: the device-built node tables (tuv [n0][n1][nz][18], rho [n0][n1][nz][2])."""
        tuv = np.empty((n0, n1, nz, 18)); rho = np.empty((n0, n1, nz, 2))
        self._check(lib().geoac_get_grid_tables(self._h, tuv.size, _p(tuv), rho.size, _p(rho)), "geoac_get_grid_tables")
        return tuv, rho

    @property
    def params(self):
        p = GeoacParams()
        self._check(lib().geoac_get_params(self._h, C.byref(p)), "geoac_get_params")
        return p

    @params.setter
    def params(self, p):
        self._check(lib().geoac_set_params(self._h, C.byref(p)), "geoac_set_params")

    def _rays_and_records(self, what, theta, phi, out):
        """The angles as contiguous float64 arrays and the record buffers of a trace of them (`out`, checked, or new ones)."""
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        n = len(theta)
        n_rec = self.params.bounces + 1
        if phi.shape != theta.shape or theta.ndim != 1:
            raise GeoAcError(f"{what}: theta and phi must be 1-D arrays of one length")
        if out is None:
            out = {"rec": np.empty((abi.NFIELDS, n, n_rec)), "status": np.empty((n, n_rec), dtype=np.int32),
                   "n_steps": np.empty((n, n_rec), dtype=np.int32)}
        else:
            for k, dt, size in (("rec", np.float64, abi.NFIELDS * n * n_rec), ("status", np.int32, n * n_rec), ("n_steps", np.int32, n * n_rec)):
                a = out[k]
                if not (isinstance(a, np.ndarray) and a.dtype == dt and a.flags["C_CONTIGUOUS"] and a.flags["WRITEABLE"] and a.size == size):
                    raise GeoAcError(f"{what}: out['{k}'] must be a writeable C-contiguous {np.dtype(dt).name} array of {size} elements")
        return theta, phi, out

    def trace(self, theta, phi, out=None):
        """Host buffers in, host buffers out (H2D + kernels + D2H inside). Returns dict(rec, status, n_steps)."""
        theta, phi, out = self._rays_and_records("trace", theta, phi, out)
        self._check(lib().geoac_trace(self._h, len(theta), _p(theta), _p(phi), _p(out["rec"]), out["status"].ctypes.data_as(_ip),
                                      out["n_steps"].ctypes.data_as(_ip)), "geoac_trace")
        return out

    def trace_sources(self, src, src_id, theta, phi, out=None):
        """trace() for rays from many sources in one call: ray r starts from src[src_id[r]].  src: [n_src, 3] in the
        convention of params.src; src_id: int32 [n].  Ray r's records equal those of trace() with params.src = src[src_id[r]]
        (include/geoac_b200.h: geoac_trace_sources).  Lay the batch out source by source."""
        theta, phi, out = self._rays_and_records("trace_sources", theta, phi, out)
        src = np.ascontiguousarray(src, dtype=np.float64)
        if src.ndim != 2 or src.shape[1] != 3:
            raise GeoAcError("trace_sources: src must be an array of shape [n_src, 3]")
        src_id = np.asarray(src_id)
        if src_id.dtype != np.int32 or src_id.shape != theta.shape:
            raise GeoAcError("trace_sources: src_id must be an int32 array with one entry per ray")
        src_id = np.ascontiguousarray(src_id)
        self._check(lib().geoac_trace_sources(self._h, len(src), _p(src), len(theta), src_id.ctypes.data_as(_ip), _p(theta), _p(phi),
                                              _p(out["rec"]), out["status"].ctypes.data_as(_ip), out["n_steps"].ctypes.data_as(_ip)),
                    "geoac_trace_sources")
        return out

    def trace_ensemble(self, atm_id, theta, phi, out=None):
        """trace() for rays through many atmospheres in one call: ray r runs through member atm_id[r] (int32 [n]) of the
        ensemble of set_ensemble_1d.  Ray r's records equal those of trace() on a context with that member's profile and
        these parameters (include/geoac_b200.h: geoac_trace_ensemble).  Lay the batch out member by member."""
        theta, phi, out = self._rays_and_records("trace_ensemble", theta, phi, out)
        atm_id = np.asarray(atm_id)
        if atm_id.dtype != np.int32 or atm_id.shape != theta.shape:
            raise GeoAcError("trace_ensemble: atm_id must be an int32 array with one entry per ray")
        atm_id = np.ascontiguousarray(atm_id)
        self._check(lib().geoac_trace_ensemble(self._h, len(theta), atm_id.ctypes.data_as(_ip), _p(theta), _p(phi), _p(out["rec"]),
                                               out["status"].ctypes.data_as(_ip), out["n_steps"].ctypes.data_as(_ip)),
                    "geoac_trace_ensemble")
        return out

    def trace_paths(self, theta, phi, stride=25, cap=2400, caustic_cap=0):
        """trace() plus the raypath rows of WriteRays=True (path [n][cap][PATH_NF], path_rows [n]) and, with caustic_cap > 0,
        the WriteCaustics=True events (caustic [n][caustic_cap][CAUSTIC_NF], caustic_rows [n])."""
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        n = len(theta)
        n_rec = self.params.bounces + 1
        out = {"rec": np.empty((abi.NFIELDS, n, n_rec)), "status": np.empty((n, n_rec), dtype=np.int32),
               "n_steps": np.empty((n, n_rec), dtype=np.int32), "path": np.zeros((n, max(cap, 1), abi.PATH_NF)),
               "path_rows": np.zeros(n, dtype=np.int32), "caustic": np.zeros((n, max(caustic_cap, 1), abi.CAUSTIC_NF)),
               "caustic_rows": np.zeros(n, dtype=np.int32)}
        self._check(lib().geoac_trace_paths(self._h, n, _p(theta), _p(phi), _p(out["rec"]), out["status"].ctypes.data_as(_ip),
                                            out["n_steps"].ctypes.data_as(_ip), stride, cap, _p(out["path"]),
                                            out["path_rows"].ctypes.data_as(_ip), caustic_cap, _p(out["caustic"]),
                                            out["caustic_rows"].ctypes.data_as(_ip)), "geoac_trace_paths")
        return out

    def trace_paths_compact(self, theta, phi, stride=25, cap=2400, caustic_cap=0, total_rows=None, total_events=None):
        """trace_paths() with compacted rows: path [total][PATH_NF] + path_offset [n + 1] (ray i owns rows offset[i]:offset[i+1]),
        likewise caustic / caustic_offset.  total_rows / total_events: output capacities in rows (default: generous estimates;
        grown and retried once if the library reports they were too small)."""
        theta = np.ascontiguousarray(theta, dtype=np.float64)
        phi = np.ascontiguousarray(phi, dtype=np.float64)
        n = len(theta)
        n_rec = self.params.bounces + 1
        out = {"rec": np.empty((abi.NFIELDS, n, n_rec)), "status": np.empty((n, n_rec), dtype=np.int32), "n_steps": np.empty((n, n_rec), dtype=np.int32)}
        return self._paths_compact(lambda *cap_args: lib().geoac_trace_paths_compact(
            self._h, n, _p(theta), _p(phi), _p(out["rec"]), out["status"].ctypes.data_as(_ip), out["n_steps"].ctypes.data_as(_ip), *cap_args),
            "geoac_trace_paths_compact", n, out, stride, cap, caustic_cap, total_rows, total_events)

    def _paths_compact(self, call, what, n, out, stride, cap, caustic_cap, total_rows, total_events):
        """The capture buffers of a compacted-rows call (call(*capture arguments) -> status), grown and retried once when the
        library reports them too small; adds them to `out`."""
        total_rows = total_rows if total_rows is not None else max(1, n * min(cap, 1024)) if stride > 0 else 1
        total_events = total_events if total_events is not None else max(1, n * min(max(caustic_cap, 1), 8))
        for attempt in range(2):
            path = np.zeros((max(total_rows, 1), abi.PATH_NF)); poff = np.zeros(n + 1, dtype=np.int64)
            caus = np.zeros((max(total_events, 1), abi.CAUSTIC_NF)); coff = np.zeros(n + 1, dtype=np.int64)
            rc = call(stride, cap, total_rows, _p(path), poff.ctypes.data_as(C.POINTER(C.c_int64)),
                      caustic_cap, total_events, _p(caus), coff.ctypes.data_as(C.POINTER(C.c_int64)))
            if rc == abi.GEOAC_ERR_TOO_LARGE and attempt == 0:
                total_rows, total_events = max(total_rows, int(poff[-1])), max(total_events, int(coff[-1]))
                continue
            self._check(rc, what)
            break
        out.update(path=path[: poff[-1]], path_offset=poff, caustic=caus[: coff[-1]], caustic_offset=coff)
        return out

    def trace_sources_paths_compact(self, src, src_id, theta, phi, stride=25, cap=2400, caustic_cap=0, total_rows=None, total_events=None):
        """trace_paths_compact() for rays from many sources in one call: ray r starts from src[src_id[r]] (src, src_id as for
        trace_sources).  Ray r's records and rows equal those of trace_paths_compact() with params.src = src[src_id[r]]
        (include/geoac_b200.h: geoac_trace_sources_paths_compact)."""
        theta, phi, out = self._rays_and_records("trace_sources_paths_compact", theta, phi, None)
        src = np.ascontiguousarray(src, dtype=np.float64)
        if src.ndim != 2 or src.shape[1] != 3:
            raise GeoAcError("trace_sources_paths_compact: src must be an array of shape [n_src, 3]")
        src_id = np.asarray(src_id)
        if src_id.dtype != np.int32 or src_id.shape != theta.shape:
            raise GeoAcError("trace_sources_paths_compact: src_id must be an int32 array with one entry per ray")
        src_id = np.ascontiguousarray(src_id)
        return self._paths_compact(lambda *cap_args: lib().geoac_trace_sources_paths_compact(
            self._h, len(src), _p(src), len(theta), src_id.ctypes.data_as(_ip), _p(theta), _p(phi), _p(out["rec"]),
            out["status"].ctypes.data_as(_ip), out["n_steps"].ctypes.data_as(_ip), *cap_args),
            "geoac_trace_sources_paths_compact", len(theta), out, stride, cap, caustic_cap, total_rows, total_events)

    def reserve(self, n_rays):
        """Pre-allocate the device staging of trace() for batches of up to n_rays rays."""
        self._check(lib().geoac_reserve(self._h, n_rays), "geoac_reserve")

    def trace_device(self, n, d_theta, d_phi, d_rec, d_status, d_n_steps, stream=0):
        """Device pointers (ints) in/out, enqueued on `stream` (cudaStream_t as int); no synchronisation."""
        self._check(lib().geoac_trace_device(self._h, n, d_theta, d_phi, d_rec, d_status, d_n_steps, stream), "geoac_trace_device")

    def last_stats(self):
        s = C.c_int64(0)
        ms = C.c_double(0)
        self._check(lib().geoac_last_trace_stats(self._h, C.byref(s), C.byref(ms)), "geoac_last_trace_stats")
        return s.value, ms.value

    def last_lane_occupancy(self):
        """Average fraction of a warp's 32 lanes that carried a ray during the last trace."""
        steps, _ = self.last_stats()
        t = C.c_int64(0)
        self._check(lib().geoac_last_trace_counters(self._h, C.byref(t), None), "geoac_last_trace_counters")
        return steps / (32.0 * t.value) if t.value else 0.0

    def last_kernel_launches(self):
        """Kernels the last trace enqueued (1; 6 or 7 for the range-dependent sets and 10 for the stratified ones with the
        longest-ray-first scheduling pass)."""
        k = C.c_int64(0)
        self._check(lib().geoac_last_trace_counters(self._h, None, C.byref(k)), "geoac_last_trace_counters")
        return k.value

    def last_schedule(self):
        """Scheduling facts of the last trace: long-region packets, quarter packets, exclusive long-region CTAs, kernels."""
        o = (C.c_int64 * 8)()
        self._check(lib().geoac_last_schedule(self._h, o), "geoac_last_schedule")
        ms = np.zeros(2)
        lib().geoac_last_launch_ms(self._h, _p(ms))
        return {"long_packets": o[1], "quarter_packets": o[4], "long_ctas": o[2], "launches": o[3], "main_ms": float(ms[0]), "long_ms": float(ms[1])}

    def predicted_costs(self, n):
        """RK4 step counts the cost scout predicted for the n rays of the last trace (diagnosis hook)."""
        c = np.zeros(n, dtype=np.uint32)
        self._check(lib().geoac_get_costs(self._h, n, c.ctypes.data_as(C.POINTER(C.c_uint32))), "geoac_get_costs")
        return c

    def selftest_math(self, n_per_thread=2000):
        """Max relative error of the kernel's rcp / rsqrt / sqrt / exp / exp10 against the CUDA math library."""
        out = np.zeros(7)
        self._check(lib().geoac_selftest_math(self._h, n_per_thread, _p(out)), "geoac_selftest_math")
        return dict(zip(("rcp", "rsqrt", "sqrt", "exp", "exp10", "sin", "cos"), out.tolist()))

    def measure_fp64_peak(self):
        ms = C.c_double(0)
        return lib().geoac_measure_fp64_peak(self._h, C.byref(ms)), ms.value


def trace_multi(tracers, theta, phi, out=None):
    """geoac_trace_multi over existing contexts (one per device; same variant / atmosphere / parameters on each): the batch is
    dealt to them in interleaved GEOAC_SHARD_BLOCK-ray blocks by host threads INSIDE the library and merged by ray index.
    Bitwise identical to tracing the batch on one context."""
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    phi = np.ascontiguousarray(phi, dtype=np.float64)
    if phi.shape != theta.shape or theta.ndim != 1:
        raise GeoAcError("trace_multi: theta and phi must be 1-D arrays of one length")
    n = len(theta)
    n_rec = tracers[0].params.bounces + 1
    if out is None:
        out = {"rec": np.empty((abi.NFIELDS, n, n_rec)), "status": np.empty((n, n_rec), dtype=np.int32),
               "n_steps": np.empty((n, n_rec), dtype=np.int32)}
    handles = (C.c_void_p * len(tracers))(*[t._h for t in tracers])
    rc = lib().geoac_trace_multi(handles, len(tracers), n, _p(theta), _p(phi), _p(out["rec"]), out["status"].ctypes.data_as(_ip),
                                 out["n_steps"].ctypes.data_as(_ip))
    if rc != abi.GEOAC_OK:
        raise GeoAcError(f"geoac_trace_multi failed ({rc}): {lib().geoac_last_error(tracers[0]._h).decode()}")
    return out


class MultiTracer:
    """One context per device behind one object (geoac_create_multi + the geoac_multi_* helpers + geoac_trace_multi)."""

    def __init__(self, variant, devices):
        devices = list(devices)
        ids = (C.c_int * len(devices))(*devices)
        hs = (C.c_void_p * len(devices))()
        st = C.c_int(0)
        rc = lib().geoac_create_multi(variant, ids, len(devices), hs, C.byref(st))
        if rc != abi.GEOAC_OK:
            raise GeoAcError(f"geoac_create_multi failed ({st.value}): {lib().geoac_last_error(None).decode()}")
        self.tracers = []
        for h, d in zip(hs, devices):
            t = Tracer.__new__(Tracer)
            t._h, t.variant, t.device = h, variant, d
            self.tracers.append(t)
        self._hs = hs
        self.variant = variant

    def _check(self, rc, what):
        if rc != abi.GEOAC_OK:
            raise GeoAcError(f"{what} failed ({rc}): {lib().geoac_last_error(self.tracers[0]._h).decode()}")

    def set_atmosphere_1d(self, z, T, u, v, rho):
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (z, T, u, v, rho)]
        self._check(lib().geoac_multi_set_atmosphere_1d(self._hs, len(self.tracers), len(arrs[0]), *[_p(a) for a in arrs]), "geoac_multi_set_atmosphere_1d")

    def set_atmosphere_3d(self, ax0, ax1, axz, T, u, v, rho):
        arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in (ax0, ax1, axz, T, u, v, rho)]
        self._check(lib().geoac_multi_set_atmosphere_3d(self._hs, len(self.tracers), len(arrs[0]), len(arrs[1]), len(arrs[2]), *[_p(a) for a in arrs]),
                    "geoac_multi_set_atmosphere_3d")

    @property
    def params(self):
        return self.tracers[0].params

    @params.setter
    def params(self, p):
        self._check(lib().geoac_multi_set_params(self._hs, len(self.tracers), C.byref(p)), "geoac_multi_set_params")

    def trace(self, theta, phi, out=None):
        return trace_multi(self.tracers, theta, phi, out)

    def close(self):
        for t in self.tracers:
            t.close()
        self.tracers = []
