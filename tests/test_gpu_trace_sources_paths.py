"""geoac_trace_sources_paths_compact -- raypath rows and caustic events of rays from many sources in one call -- against
geoac_trace_paths_compact with params.src set to each ray's source, bit for bit (records, status, step counts, offsets,
raypath rows and caustic rows), for all ten capture kernels (five variants x calc_amp) in the natural and the forced claim
order, and the global-table kernels of a profile too large for shared memory.  Also: too-small output capacities, the
argument checks, and the raypaths of the eigenrays a many-source search finds."""
import ctypes as C

import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, api
from tests import util
from tests.test_gpu_device_path import CASES, make_tracer, seeded_angles
from tests.test_gpu_trace_sources import SOURCES, BOUNCES_RD, with_source

pytestmark = pytest.mark.gpu

RAGGED = (1, 5, 17, 33, 40)            # rays per source
STRIDE, CAP, CAUS_CAP = 25, 400, 8


def tracer(case, calc_amp=1, knobs=None):
    variant = int(util.load_case(case)[0]["variant"])
    return make_tracer(case, calc_amp, knobs=knobs, accum_per_segment=1, **({"bounces": BOUNCES_RD} if util.is_rngdep(variant) else {}))


def split(out, r):
    """Ray r's raypath and caustic rows of a compacted result."""
    po, co = out["path_offset"], out["caustic_offset"]
    return out["path"][po[r]:po[r + 1]], out["caustic"][co[r]:co[r + 1]]


def per_source(tr, src, src_id, th, ph, caustic_cap):
    """One geoac_trace_paths_compact per source on `tr` (params.src set to it): records in batch order and each ray's rows."""
    n, n_rec = len(th), tr.params.bounces + 1
    want = {"rec": np.empty((abi.NFIELDS, n, n_rec)), "status": np.empty((n, n_rec), np.int32), "n_steps": np.empty((n, n_rec), np.int32)}
    rows = [None] * n
    for s in range(len(src)):
        idx = np.flatnonzero(src_id == s)
        if not len(idx):
            continue
        with_source(tr, src[s])
        o = tr.trace_paths_compact(th[idx], ph[idx], STRIDE, CAP, caustic_cap=caustic_cap)
        want["rec"][:, idx] = o["rec"]
        want["status"][idx] = o["status"]
        want["n_steps"][idx] = o["n_steps"]
        for j, r in enumerate(idx):
            rows[r] = split(o, j)
    return want, rows


def assert_equal(got, want, rows, label):
    for k in ("rec", "status", "n_steps"):
        assert np.array_equal(got[k].view(np.uint8), want[k].view(np.uint8)), (label, k)
    for r, (wp, wc) in enumerate(rows):
        gp, gc = split(got, r)
        assert np.array_equal(gp.view(np.uint64), wp.view(np.uint64)), (label, "path", r)
        assert np.array_equal(gc.view(np.uint64), wc.view(np.uint64)), (label, "caustic", r)
    assert got["path_offset"][-1] == sum(len(p) for p, _ in rows) and got["caustic_offset"][-1] == sum(len(c) for _, c in rows), label


@pytest.mark.parametrize("calc_amp", [1, 0])
@pytest.mark.parametrize("variant", sorted(CASES), ids=[abi.VARIANT_NAMES[v] for v in sorted(CASES)])
def test_equals_one_capture_per_source(variant, calc_amp):
    case = CASES[variant]
    src = np.array(SOURCES[variant])
    rng = np.random.default_rng(20261023 + variant)
    src_id = rng.permutation(np.repeat(np.arange(len(src), dtype=np.int32), RAGGED))
    th, ph = seeded_angles(len(src_id), 300 + variant)
    caus = CAUS_CAP if calc_amp else 0
    want, rows = per_source(tracer(case, calc_amp, {"lpt": 0}), src, src_id, th, ph, caus)
    assert sum(len(p) for p, _ in rows) > 0 and (want["status"] == abi.ST_ARRIVAL).any()
    if calc_amp and variant != abi.GEOAC_2D:
        assert sum(len(c) for _, c in rows) > 0, "some caustics to compare"
    for lpt in (0, 2):
        tr = tracer(case, calc_amp, {"lpt": lpt})
        p0 = bytes(tr.params)
        got = tr.trace_sources_paths_compact(src, src_id, th, ph, STRIDE, CAP, caustic_cap=caus)
        assert_equal(got, want, rows, f"{case} calc_amp={calc_amp} lpt={lpt}")
        assert bytes(tr.params) == p0
        assert (tr.last_kernel_launches() > 1) == (lpt == 2)


def test_global_table_kernels():
    """A profile with more levels than fit in shared memory (levels appended above the propagation ceiling, as
    test_gpu_scale does): the capture kernels that read the table through L1 / L2."""
    z, T, u, v, rho = g.load_met_1d(util.TOY)
    zx = np.concatenate([z, z[-1] + 0.1 * np.arange(1, 2001)])
    ext = lambda f: np.concatenate([f, np.full(2000, f[-1])])
    src = np.array(SOURCES[abi.GEOAC_3D])
    src_id = np.repeat(np.arange(len(src), dtype=np.int32), 12)
    th, ph = seeded_angles(len(src_id), 77)
    for calc_amp in (1, 0):
        def big():
            tr = g.Tracer(abi.GEOAC_3D, 0)
            tr.set_atmosphere_1d(z, T, u, v, rho)
            vert = tr.params.vert_limit
            tr.set_atmosphere_1d(zx, ext(T), ext(u), ext(v), ext(rho))
            p = tr.params
            p.vert_limit, p.accum_per_segment, p.calc_amp = vert, 1, calc_amp
            tr.params = p
            return tr
        caus = CAUS_CAP if calc_amp else 0
        want, rows = per_source(big(), src, src_id, th, ph, caus)
        got = big().trace_sources_paths_compact(src, src_id, th, ph, STRIDE, CAP, caustic_cap=caus)
        assert_equal(got, want, rows, f"global table calc_amp={calc_amp}")


def _raw(tr, src, sid, th, ph, out, stride=STRIDE, cap=CAP, total=10 ** 6, ccap=CAUS_CAP, ctotal=10 ** 5):
    dp = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))
    lp = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_int64))
    return [len(src) if src is not None else 0, dp(src), len(th) if th is not None else 0, ip(sid), dp(th), dp(ph), dp(out["rec"]),
            ip(out["status"]), ip(out["n_steps"]), stride, cap, total, dp(out["path"]), lp(out["poff"]), ccap, ctotal, dp(out["caus"]),
            lp(out["coff"])]


def test_capacities_and_argument_checks():
    L = api.lib()
    tr = tracer("3d_sub")
    src = np.array(SOURCES[abi.GEOAC_3D][:3])
    n = 12
    sid = (np.arange(n) % 3).astype(np.int32)
    th, ph = seeded_angles(n, 11)

    def bufs(total=4000, ctotal=200):
        return {"rec": np.full((abi.NFIELDS, n, 3), -7.0), "status": np.full((n, 3), -7, np.int32), "n_steps": np.full((n, 3), -7, np.int32),
                "path": np.full((total, abi.PATH_NF), -7.0), "poff": np.full(n + 1, -7, np.int64),
                "caus": np.full((ctotal, abi.CAUSTIC_NF), -7.0), "coff": np.full(n + 1, -7, np.int64)}
    call = lambda a: L.geoac_trace_sources_paths_compact(tr._h, *a)
    msg = lambda: L.geoac_last_error(tr._h).decode()
    bad = abi.GEOAC_ERR_BAD_ARG
    want = tr.trace_sources_paths_compact(src, sid, th, ph, STRIDE, CAP, caustic_cap=CAUS_CAP)
    total, ctotal = int(want["path_offset"][-1]), int(want["caustic_offset"][-1])
    assert total > 1 and ctotal > 1
    # too small: GEOAC_ERR_TOO_LARGE with the offsets filled in; then exactly large enough
    for t, ct in ((total - 1, ctotal), (total, ctotal - 1)):
        b = bufs(max(t, 1), max(ct, 1))
        assert call(_raw(tr, src, sid, th, ph, b, total=t, ctotal=ct)) == abi.GEOAC_ERR_TOO_LARGE and "rows produced" in msg()
        assert np.array_equal(b["poff"], want["path_offset"]) and np.array_equal(b["coff"][: 1], [0])
        if t == total:
            assert np.array_equal(b["coff"], want["caustic_offset"])
    b = bufs(total, ctotal)
    assert call(_raw(tr, src, sid, th, ph, b, total=total, ctotal=ctotal)) == abi.GEOAC_OK
    assert np.array_equal(b["path"].view(np.uint64), want["path"].view(np.uint64))
    assert np.array_equal(b["caus"].view(np.uint64), want["caustic"].view(np.uint64))
    # the source arguments, refused as geoac_trace_sources refuses them; nothing written
    p0 = bytes(tr.params)
    assert L.geoac_trace_sources_paths_compact(None, *_raw(tr, src, sid, th, ph, bufs())) == bad
    for k, v in ((0, 0), (0, -2), (1, None), (3, None), (4, None), (5, None), (6, None), (7, None), (8, None)):
        b = bufs(); a = _raw(tr, src, sid, th, ph, b); a[k] = v
        assert call(a) == bad and ("n_src" in msg() or "non-null" in msg()), k
        assert (b["rec"] == -7.0).all() and (b["poff"] == -7).all()
    b = bufs(); a = _raw(tr, src, sid, th, ph, b); a[2] = -1
    assert call(a) == bad and "n_rays < 0" in msg()
    s2 = src.copy(); s2[2, 0] = np.nan
    b = bufs()
    assert call(_raw(tr, s2, sid, th, ph, b)) == bad and "source 2 " in msg()
    s3 = sid.copy(); s3[4] = 3
    assert call(_raw(tr, src, s3, th, ph, b)) == bad and "ray 4 " in msg()
    # the capture arguments, refused as geoac_trace_paths_compact refuses them
    for kw, words in (({"stride": 0, "ccap": 0}, "ask for"), ({"stride": -1}, "ask for"), ({"cap": 0}, "positive per-ray capacity"),
                      ({"ccap": -1}, "ask for")):
        b = bufs()
        assert call(_raw(tr, src, sid, th, ph, b, **kw)) == bad and words in msg(), kw
    b = bufs(); a = _raw(tr, src, sid, th, ph, b); a[12] = None
    assert call(a) == bad and "raypath capture" in msg()
    b = bufs(); a = _raw(tr, src, sid, th, ph, b); a[17] = None
    assert call(a) == bad and "caustic capture needs its buffers" in msg()
    assert (b["rec"] == -7.0).all()
    noamp = tracer("3d_sub", calc_amp=0)
    assert L.geoac_trace_sources_paths_compact(noamp._h, *_raw(noamp, src, sid, th, ph, bufs())) == bad
    flat = tracer("3d_sub")
    p = flat.params; p.accum_per_segment = 0; flat.params = p
    assert L.geoac_trace_sources_paths_compact(flat._h, *_raw(flat, src, sid, th, ph, bufs())) == bad
    bare = g.Tracer(abi.GEOAC_3D, 0)
    pb = bare.params; pb.accum_per_segment = 1; bare.params = pb
    assert L.geoac_trace_sources_paths_compact(bare._h, *_raw(bare, src, sid, th, ph, bufs())) == abi.GEOAC_ERR_NO_ATMO
    # n_rays == 0: the first offsets set, nothing else
    b = bufs()
    a = _raw(tr, None, None, None, None, b); a[12], a[13], a[16], a[17] = b["path"].ctypes.data_as(C.POINTER(C.c_double)), \
        b["poff"].ctypes.data_as(C.POINTER(C.c_int64)), b["caus"].ctypes.data_as(C.POINTER(C.c_double)), b["coff"].ctypes.data_as(C.POINTER(C.c_int64))
    assert call(a) == abi.GEOAC_OK and b["poff"][0] == 0 and b["coff"][0] == 0 and (b["poff"][1:] == -7).all() and (b["path"] == -7.0).all()
    assert bytes(tr.params) == p0
