"""geoac_trace_sources -- rays from many sources in one call -- against geoac_trace with params.src set to each ray's source,
bit for bit (status, n_steps and every record field), for all ten record kernels (five variants x calc_amp) in the natural
and the sorted claim order.  Also: one source equal to params.src against geoac_trace of the same batch, the range-dependent
long region and quarter claims, a batch above the lane count, the context left as it was, and the argument checks."""
import ctypes as C

import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, api
from tests import util
from tests.test_gpu_device_path import CASES, assert_bitwise, make_tracer, seeded_angles
from tests.test_gpu_rngdep_schedule import mixed_angles

pytestmark = pytest.mark.gpu

D2R = util.PI / 180.0
RAGGED = (1, 7, 33, 64, 100)           # rays per source
# five sources per variant, each as geoac_params.src takes it: one below the ground (clamped to it); Global ones at several
# latitudes / longitudes; range-dependent ones near a corner of the grid and outside it (every ray breaks at once)
SOURCES = {
    abi.GEOAC_2D: [(0.0, 0.0, 0.0), (0.0, 0.0, 0.5), (0.0, 0.0, -1.0), (0.0, 0.0, 2.0), (0.0, 0.0, 12.0)],
    abi.GEOAC_3D: [(0.0, 0.0, 0.0), (120.0, -40.0, 0.0), (-200.0, 150.0, 1.5), (30.0, 60.0, -2.0), (0.0, 0.0, 12.0)],
    abi.GEOAC_GLOBAL: [(0.0, 30 * D2R, 0.0), (0.0, -20 * D2R, 45 * D2R), (1.5, 60 * D2R, -100 * D2R), (-1.0, 10 * D2R, 170 * D2R),
                       (8.0, 0.0, 0.0)],
    abi.GEOAC_3D_RNGDEP: [(0.0, 0.0, 0.0), (-480.0, 470.0, 0.0), (650.0, 0.0, 0.0), (100.0, -200.0, -1.0), (200.0, 300.0, 2.0)],
    abi.GEOAC_GLOBAL_RNGDEP: [(0.0, 35 * D2R, 0.0), (0.0, 44.5 * D2R, -11.5 * D2R), (0.0, 50 * D2R, 0.0), (-1.0, 30 * D2R, 5 * D2R),
                              (3.0, 40 * D2R, -5 * D2R)],
}
BOUNCES_RD = 1         # range-dependent sets: one reflection per ray keeps their GPU time small (as test_gpu_rngdep_schedule)


def with_source(tr, s):
    p = tr.params
    p.src[0], p.src[1], p.src[2] = s
    tr.params = p


def per_source(tr, src, src_id, th, ph):
    """The records of the batch from one geoac_trace per source on `tr` (params.src set to it), put back in batch order."""
    n, n_rec = len(th), tr.params.bounces + 1
    want = {"rec": np.empty((abi.NFIELDS, n, n_rec)), "status": np.empty((n, n_rec), np.int32), "n_steps": np.empty((n, n_rec), np.int32)}
    for s in range(len(src)):
        m = src_id == s
        if not m.any():
            continue
        with_source(tr, src[s])
        o = tr.trace(th[m], ph[m])
        want["rec"][:, m] = o["rec"]
        want["status"][m] = o["status"]
        want["n_steps"][m] = o["n_steps"]
    return want


def tracer(case, calc_amp=1, knobs=None):
    variant = int(util.load_case(case)[0]["variant"])
    return make_tracer(case, calc_amp, knobs=knobs, **({"bounces": BOUNCES_RD} if util.is_rngdep(variant) else {}))


@pytest.mark.parametrize("calc_amp", [1, 0])
@pytest.mark.parametrize("variant", sorted(CASES), ids=[abi.VARIANT_NAMES[v] for v in sorted(CASES)])
def test_equals_one_trace_per_source(variant, calc_amp):
    case = CASES[variant]
    src = np.array(SOURCES[variant])
    rng = np.random.default_rng(20261022 + variant)
    src_id = rng.permutation(np.repeat(np.arange(len(src), dtype=np.int32), RAGGED))      # ragged counts, interleaved
    th, ph = seeded_angles(len(src_id), 100 + variant)
    want = per_source(tracer(case, calc_amp, {"lpt": 0}), src, src_id, th, ph)
    assert (want["status"][:, 0] != abi.ST_NONE).all() and (want["status"] == abi.ST_ARRIVAL).any()
    if util.is_rngdep(variant):
        assert (want["status"][src_id == 2, 0] == abi.ST_BREAK).all()                  # the source outside the grid
    for lpt in (0, 2):
        tr = tracer(case, calc_amp, {"lpt": lpt})
        p0 = tr.params.src[:]
        got = tr.trace_sources(src, src_id, th, ph)
        assert_bitwise(got, want, f"{case} calc_amp={calc_amp} lpt={lpt}")
        assert tr.params.src[:] == p0
        assert (tr.last_kernel_launches() > 1) == (lpt == 2)


@pytest.mark.parametrize("case", ["3d_sub", "3drngdep_c4"])
def test_one_source_equals_geoac_trace(case):
    """One source equal to params.src: geoac_trace of the same batch, for 1, 33 and 1000 rays; a permuted batch gives the
    permuted records."""
    tr = tracer(case)
    src = np.array([tr.params.src[:]])
    th, ph = seeded_angles(1000, 5)
    for n in (1, 33, 1000):
        want = tr.trace(th[:n], ph[:n])
        got = tr.trace_sources(src, np.zeros(n, np.int32), th[:n], ph[:n])
        assert_bitwise(got, want, f"{case} n={n}")
    perm = np.random.default_rng(9).permutation(1000)
    got = tr.trace_sources(src, np.zeros(1000, np.int32), th[perm], ph[perm])
    assert_bitwise(got, {"rec": want["rec"][:, perm], "status": want["status"][perm], "n_steps": want["n_steps"][perm]}, f"{case} permuted")


@pytest.mark.parametrize("case", ["3drngdep_c4", "globalrngdep_c5"])
def test_rngdep_long_region_and_quarter_claims(case):
    """Two sources, 500 rays each, laid out source by source; the claim order forced on and every long packet long enough
    for quarter claims.  The long region, its exclusive launch and the quarter claims run, and the records equal the
    per-source traces in the natural order."""
    variant = int(util.load_case(case)[0]["variant"])
    src = np.array([SOURCES[variant][0], SOURCES[variant][4]])
    th0, ph0 = mixed_angles(500, 160, seed=7)
    th1, ph1 = mixed_angles(500, 160, seed=17)
    th, ph = np.concatenate([th0, th1]), np.concatenate([ph0, ph1])
    src_id = np.repeat(np.arange(2, dtype=np.int32), 500)
    want = per_source(tracer(case, knobs={"lpt": 0}), src, src_id, th, ph)
    tr = tracer(case, knobs={"lpt": 2, "quarter_alpha": 100})
    got = tr.trace_sources(src, src_id, th, ph)
    assert_bitwise(got, want, case)
    s = tr.last_schedule()
    assert s["long_packets"] > 0 and s["long_ctas"] > 0 and s["quarter_packets"] > 0, s
    assert s["long_packets"] < len(th) // 32, s                                   # a main region beside the long one


def test_above_the_lane_count():
    """64 sources on an 8 x 8 grid, 1000 rays each (3D, 64 000 rays: more than the 148 x 384 lanes of the launch): the
    automatic claim order engages, and the records equal one geoac_trace per source."""
    tr = tracer("3d_sub")
    xy = np.linspace(-200.0, 200.0, 8)
    src = np.array([(x, y, 0.0) for x in xy for y in xy])
    _, _, th1, ph1 = g.prop_angles(1.0, 50.0, 1.0, 0.0, 342.0, 18.0)              # 50 x 20 angles, the mains' loop order
    th, ph = np.tile(th1, len(src)), np.tile(ph1, len(src))
    src_id = np.repeat(np.arange(len(src), dtype=np.int32), len(th1))
    got = tr.trace_sources(src, src_id, th, ph)
    assert tr.last_kernel_launches() > 1
    want = per_source(tracer("3d_sub"), src, src_id, th, ph)
    assert_bitwise(got, want, "64 sources")


def test_context_is_left_as_it_was():
    """Parameters, the source state and a geoac_trace are the same before and after a sources call, and the call reports
    its own statistics: total_steps is the sum of its step counts."""
    tr = tracer("3d_sub")
    th, ph = seeded_angles(200, 3)
    before = (bytes(tr.params), tr.source_state().tobytes(), tr.trace(th, ph))
    src = np.array(SOURCES[abi.GEOAC_3D])
    src_id = (np.arange(200) % len(src)).astype(np.int32)
    out = tr.trace_sources(src, src_id, th[::-1].copy(), ph)
    steps, ms = tr.last_stats()
    assert steps == int(out["n_steps"].sum()) and ms > 0.0
    assert bytes(tr.params) == before[0] and tr.source_state().tobytes() == before[1]
    assert_bitwise(tr.trace(th, ph), before[2], "after a sources call")


def test_argument_checks():
    L = api.lib()
    tr = tracer("3d_sub")
    n = 8
    th, ph = seeded_angles(n, 1)
    src = np.array([[0.0, 0.0, 0.0], [10.0, 0.0, 1.0]])
    sid = np.array([0, 1] * 4, np.int32)
    rec, st, ns = np.full((abi.NFIELDS, n, 3), -7.0), np.full((n, 3), -7, np.int32), np.full((n, 3), -7, np.int32)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    args = lambda: [2, dp(src), n, ip(sid), dp(th), dp(ph), dp(rec), ip(st), ip(ns)]
    call = lambda t, a: L.geoac_trace_sources(t._h, *a)
    msg = lambda t: L.geoac_last_error(t._h).decode()
    bad = abi.GEOAC_ERR_BAD_ARG
    assert L.geoac_trace_sources(None, *args()) == bad
    a = args(); a[2] = -1
    assert call(tr, a) == bad and "n_rays < 0" in msg(tr)
    for nsrc in (0, -3):
        a = args(); a[0] = nsrc
        assert call(tr, a) == bad and "n_src" in msg(tr)
    for i in (1, 3, 4, 5, 6, 7, 8):
        a = args(); a[i] = None
        assert call(tr, a) == bad and "non-null" in msg(tr), i
    for v in (np.nan, np.inf, -np.inf):
        s2 = src.copy(); s2[1, 2] = v
        a = args(); a[1] = dp(s2)
        assert call(tr, a) == bad and "source 1 " in msg(tr), v
    for v in (-1, 2, 1 << 30):
        s3 = sid.copy(); s3[5] = v; s3[6] = -1
        a = args(); a[3] = ip(s3)
        assert call(tr, a) == bad and "ray 5 " in msg(tr), v
    bare = g.Tracer(abi.GEOAC_3D, 0)
    assert call(bare, args()) == abi.GEOAC_ERR_NO_ATMO and "atmosphere" in msg(bare)
    a = args(); a[2] = 0
    assert call(tr, a) == abi.GEOAC_OK and call(bare, a) == abi.GEOAC_OK
    assert call(tr, [0, None, 0, None, None, None, None, None, None]) == abi.GEOAC_OK
    assert (rec == -7.0).all() and (st == -7).all() and (ns == -7).all()          # no refused or empty call wrote anything
    with pytest.raises(api.GeoAcError):
        tr.trace_sources(src, sid.astype(np.int64), th, ph)
    with pytest.raises(api.GeoAcError):
        tr.trace_sources(src[:, :2], sid, th, ph)
    assert call(tr, args()) == abi.GEOAC_OK and (st[:, 0] != abi.ST_NONE).all()
