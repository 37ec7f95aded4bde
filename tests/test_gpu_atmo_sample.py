"""geoac_sample_atmosphere on the device: the rows match the oracle's row helper on every variant (seeded points uniform, on
knots / grid nodes, on cell edges, on the first and last knots and outside the domain; the same bar as the host-emulation
test), columns 0-3 at the source point are geoac_source_state() bit for bit, a point's row does not depend on the batch it
comes in, sampling leaves the trace and its reported statistics untouched, and every invalid argument is refused."""
import ctypes as C

import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, api
from tests import atmo_sample_cases as S

pytestmark = pytest.mark.gpu

DP = C.POINTER(C.c_double)
CASES = [(c[0], c[1], c[2], c[3], {}) for c in S.GPU_CASES] + [
    ("toy_3d_medium", abi.GEOAC_3D, "profile", "toy", S.MEDIUM),
    ("grid_glob_medium", abi.GEOAC_GLOBAL_RNGDEP, "grid", "grid_glob", S.MEDIUM),
]


def _tracer(po, variant, kind, source, medium=None):
    arrays = S.load(kind, source, po)
    tr = g.Tracer(variant, 0)
    if kind == "profile":
        tr.set_atmosphere_1d(*arrays)
    else:
        tr.set_atmosphere_3d(*arrays)
    if medium:
        p = tr.params
        for k, v in medium.items():
            setattr(p, k, v)
        tr.params = p
    return tr, arrays


@pytest.mark.parametrize("label,variant,kind,source,medium", CASES, ids=[c[0] for c in CASES])
def test_device_matches_oracle(oracle, label, variant, kind, source, medium):
    tr, arrays = _tracer(oracle, variant, kind, source, medium)
    p = S.params(oracle, variant, medium)
    pts = S.points(S.axes(variant, kind, arrays), seed=S.SEED)
    want = S.oracle_rows(oracle, S.oracle_atmo(oracle, variant, kind, arrays, p), pts, p.freq)
    got = tr.sample_atmosphere(*pts)
    problems, _ = S.check(got, want, p, label)
    assert not problems, "\n".join(problems)


@pytest.mark.parametrize("label,variant,kind,source", S.GPU_CASES, ids=[c[0] for c in S.GPU_CASES])
def test_source_point_is_the_source_state(oracle, label, variant, kind, source):
    tr, _ = _tracer(oracle, variant, kind, source)
    p = tr.params
    if variant in (abi.GEOAC_GLOBAL, abi.GEOAC_GLOBAL_RNGDEP):
        pt = (max(p.z_grnd, p.src[0]) + S.R_EARTH, p.src[1], p.src[2])
    else:
        pt = (p.src[0], p.src[1], max(p.z_grnd, p.src[2]))
    row = tr.sample_atmosphere(*[np.array([x]) for x in pt])
    assert np.array_equal(row[:4, 0], tr.source_state())


@pytest.mark.parametrize("label,variant,kind,source", [S.GPU_CASES[1], S.GPU_CASES[4]], ids=["toy_3d", "grid_glob"])
def test_rows_do_not_depend_on_the_batch(oracle, label, variant, kind, source):
    """GEOAC_SAMPLE_BLOCK + 37 points in one call (two device passes) == the same points in calls of 1, 33 and 4096 points,
    and the reversed points give the reversed rows, bit for bit."""
    tr, arrays = _tracer(oracle, variant, kind, source)
    n = abi.SAMPLE_BLOCK + 37
    ax = S.axes(variant, kind, arrays)
    rng = np.random.default_rng(S.SEED + 1)
    base = S.points(ax, seed=S.SEED + 1)
    pick = rng.integers(0, len(base[0]), n)
    pts = [np.ascontiguousarray(a[pick] + np.where(rng.random(n) < 0.5, 0.0, rng.uniform(-1e-3, 1e-3, n) * (a.max() - a.min())))
           for a in base]
    whole = tr.sample_atmosphere(*pts)
    parts, at = [], 0
    for size in [1] * 40 + [33] * 40:
        parts.append(tr.sample_atmosphere(*[a[at:at + size] for a in pts])); at += size
    while at < n:
        parts.append(tr.sample_atmosphere(*[a[at:at + 4096] for a in pts])); at += 4096
    assert np.array_equal(whole, np.concatenate(parts, axis=1))
    rev = tr.sample_atmosphere(*[np.ascontiguousarray(a[::-1]) for a in pts])
    assert np.array_equal(rev, whole[:, ::-1])


@pytest.mark.parametrize("label,variant,kind,source", [S.GPU_CASES[1], S.GPU_CASES[4]], ids=["toy_3d", "grid_glob"])
def test_sampling_leaves_the_trace_alone(oracle, label, variant, kind, source):
    tr, arrays = _tracer(oracle, variant, kind, source)
    th, ph = np.radians(np.linspace(3.0, 40.0, 64)), np.radians(np.linspace(-60.0, 250.0, 64))
    first = tr.trace(th, ph)
    stats = tr.last_stats()
    trips = C.c_int64(0); launches = C.c_int64(0)
    api.lib().geoac_last_trace_counters(tr._h, C.byref(trips), C.byref(launches))
    counters = (trips.value, launches.value)
    schedule = tr.last_schedule()
    pts = S.points(S.axes(variant, kind, arrays), seed=S.SEED)
    tr.sample_atmosphere(*pts)
    assert tr.last_stats() == stats
    api.lib().geoac_last_trace_counters(tr._h, C.byref(trips), C.byref(launches))
    assert (trips.value, launches.value) == counters
    assert tr.last_schedule() == schedule
    second = tr.trace(th, ph)
    for k in ("rec", "status", "n_steps"):
        assert np.array_equal(first[k], second[k]), k


def test_invalid_arguments_are_refused(oracle):
    L = api.lib()
    tr = g.Tracer(abi.GEOAC_3D, 0)
    x, out = np.zeros(4), np.full(abi.ATM_NF * 4, 7.0)
    d, o = x.ctypes.data_as(DP), out.ctypes.data_as(DP)
    err = lambda: L.geoac_last_error(tr._h).decode()
    assert L.geoac_sample_atmosphere(None, 4, d, d, d, o) == abi.GEOAC_ERR_BAD_ARG
    assert L.geoac_sample_atmosphere(tr._h, -1, d, d, d, o) == abi.GEOAC_ERR_BAD_ARG
    for k in range(4):
        args = [d, d, d, o]
        args[k] = None
        assert L.geoac_sample_atmosphere(tr._h, 4, *args) == abi.GEOAC_ERR_BAD_ARG
    for bad in (np.nan, np.inf, -np.inf):
        for j in range(3):
            cs = [np.zeros(4) for _ in range(3)]
            cs[j][2] = bad
            assert L.geoac_sample_atmosphere(tr._h, 4, *[c.ctypes.data_as(DP) for c in cs], o) == abi.GEOAC_ERR_BAD_ARG
            assert "point 2 " in err(), err()
    assert L.geoac_sample_atmosphere(tr._h, 4, d, d, d, o) == abi.GEOAC_ERR_NO_ATMO
    tr.set_atmosphere_1d(*S.profile(oracle, "toy"))
    assert L.geoac_sample_atmosphere(tr._h, 0, None, None, None, None) == abi.GEOAC_OK
    assert L.geoac_sample_atmosphere(tr._h, 0, d, d, d, o) == abi.GEOAC_OK
    assert np.all(out == 7.0)
    assert L.geoac_sample_atmosphere(tr._h, 4, d, d, d, o) == abi.GEOAC_OK and not np.all(out == 7.0)
    with pytest.raises(api.GeoAcError):
        tr.sample_atmosphere(np.zeros(3), np.zeros(3), np.zeros(2))
