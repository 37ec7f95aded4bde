"""geoac_trace_ensemble -- rays through many stratified atmospheres in one call -- against geoac_trace on a second context
holding each ray's member (geoac_set_atmosphere_1d with the member, then geoac_set_params with the ensemble context's
parameters), bit for bit (status, n_steps and every record field), for the six stratified record kernels (2D, 3D, Global x
calc_amp) in the natural and the sorted claim order.  Also: one member equal to the context's own atmosphere against
geoac_trace of the same batch, a batch above the lane count, parameter changes between calls, the context and the ensemble
left as they were, and the argument checks."""
import ctypes as C

import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, api
from tests import util
from tests.test_gpu_device_path import CASES, assert_bitwise, make_tracer, seeded_angles

pytestmark = pytest.mark.gpu

STRATIFIED = (abi.GEOAC_2D, abi.GEOAC_3D, abi.GEOAC_GLOBAL)
R_EARTH = 6370.0                       # km, the Global tables' radial offset (core.cuh: kREarth)
RAGGED = (1, 7, 33, 64, 100)           # rays per member


def case_profile(case):
    d, _ = util.load_case(case)
    return g.load_met_1d(util.profile_path(d), global_taper=util.is_global(int(d["variant"])))


def perturbed(prof, wind, dT):
    """The profile with its winds scaled by `wind` and dT(z) [K] added to its temperatures."""
    z, T, u, v, rho = prof
    return z, T + dT(z), u * wind, v * wind, rho


def members_of(prof):
    """Five members from one profile: itself, two wind / temperature perturbations, every other level (the first and last
    kept), and the levels below 80 % of its top."""
    z = prof[0]
    coarse = np.unique(np.concatenate([np.arange(0, len(z), 2), [len(z) - 1]]))
    low = z <= z[0] + 0.8 * (z[-1] - z[0])
    return [prof,
            perturbed(prof, 1.15, lambda z: 4.0 * np.sin(z / 12.0)),
            perturbed(prof, 0.8, lambda z: -3.0 + 0.02 * z),
            tuple(a[coarse] for a in prof),
            tuple(a[low] for a in prof)]


def reference(variant, members, p, atm_id, th, ph, knobs=None):
    """The records of the batch from one geoac_trace per member on a second context (the member's profile, then the
    parameters p), put back in batch order."""
    ref = g.Tracer(variant, 0)
    for k, v in (knobs or {}).items():
        ref.set_knob(k, v)
    n, n_rec = len(th), p.bounces + 1
    want = {"rec": np.empty((abi.NFIELDS, n, n_rec)), "status": np.empty((n, n_rec), np.int32), "n_steps": np.empty((n, n_rec), np.int32)}
    for m, prof in enumerate(members):
        sel = atm_id == m
        if not sel.any():
            continue
        ref.set_atmosphere_1d(*prof)
        ref.params = p
        o = ref.trace(th[sel], ph[sel])
        want["rec"][:, sel] = o["rec"]
        want["status"][sel] = o["status"]
        want["n_steps"][sel] = o["n_steps"]
    ref.close()
    return want


def ensemble_tracer(case, members, calc_amp=1, knobs=None):
    """The golden case's context with `members` as its ensemble; the case's range limit kept, vert_limit as the ensemble
    sets it."""
    tr = make_tracer(case, calc_amp, knobs=knobs)
    rng_lim = tr.params.range_limit
    tr.set_ensemble_1d(members)
    p = tr.params
    p.range_limit = rng_lim
    tr.params = p
    return tr


@pytest.mark.parametrize("calc_amp", [1, 0])
@pytest.mark.parametrize("variant", STRATIFIED, ids=[abi.VARIANT_NAMES[v] for v in STRATIFIED])
def test_equals_one_trace_per_member(variant, calc_amp):
    case = CASES[variant]
    members = members_of(case_profile(case))
    rng = np.random.default_rng(20261022 + variant)
    atm_id = rng.permutation(np.repeat(np.arange(len(members), dtype=np.int32), RAGGED))     # ragged counts, interleaved
    th, ph = seeded_angles(len(atm_id), 200 + variant)
    want = None
    for lpt in (0, 2):
        tr = ensemble_tracer(case, members, calc_amp, {"lpt": lpt})
        p = tr.params
        top = members[4][0][-1] + (R_EARTH if util.is_global(variant) else 0.0)
        assert p.vert_limit == top                                                  # the lowest top among the members
        if want is None:
            want = reference(variant, members, p, atm_id, th, ph)
            assert (want["status"][:, 0] != abi.ST_NONE).all()
            assert (want["status"] == abi.ST_ARRIVAL).any() and (want["status"] == abi.ST_BREAK).any()
        got = tr.trace_ensemble(atm_id, th, ph)
        assert_bitwise(got, want, f"{case} calc_amp={calc_amp} lpt={lpt}")
        assert bytes(tr.params) == bytes(p)
        assert (tr.last_kernel_launches() > 1) == (lpt == 2)
        tr.close()


@pytest.mark.parametrize("variant", STRATIFIED, ids=[abi.VARIANT_NAMES[v] for v in STRATIFIED])
def test_own_atmosphere_as_the_only_member(variant):
    """One member equal to the context's own atmosphere: geoac_trace of the same batch, for 1, 33 and 1000 rays; a permuted
    batch gives the permuted records."""
    case = CASES[variant]
    tr = make_tracer(case)
    tr.set_ensemble_1d([case_profile(case)])
    th, ph = seeded_angles(1000, 5)
    for n in (1, 33, 1000):
        want = tr.trace(th[:n], ph[:n])
        got = tr.trace_ensemble(np.zeros(n, np.int32), th[:n], ph[:n])
        assert_bitwise(got, want, f"{case} n={n}")
    perm = np.random.default_rng(9).permutation(1000)
    got = tr.trace_ensemble(np.zeros(1000, np.int32), th[perm], ph[perm])
    assert_bitwise(got, {"rec": want["rec"][:, perm], "status": want["status"][perm], "n_steps": want["n_steps"][perm]}, f"{case} permuted")


def toy_members(n):
    """n members from ToyAtmo, winds scaled and temperatures offset member by member (deterministic)."""
    prof = case_profile("3d_sub")
    return [perturbed(prof, 0.7 + 0.6 * k / max(1, n - 1), lambda z, k=k: (k % 9 - 4) * 0.75 + 0.0 * z) for k in range(n)]


def test_above_the_lane_count():
    """64 members x 1000 rays (3D, 64 000 rays: more than the 148 x 384 lanes of the launch), member by member in the mains'
    loop order: the automatic claim order engages, and the records equal one geoac_trace per member."""
    members = toy_members(64)
    tr = ensemble_tracer("3d_sub", members)
    _, _, th1, ph1 = g.prop_angles(1.0, 50.0, 1.0, 0.0, 342.0, 18.0)              # 50 x 20 angles
    th, ph = np.tile(th1, len(members)), np.tile(ph1, len(members))
    atm_id = np.repeat(np.arange(len(members), dtype=np.int32), len(th1))
    got = tr.trace_ensemble(atm_id, th, ph)
    assert tr.last_kernel_launches() > 1
    want = reference(abi.GEOAC_3D, members, tr.params, atm_id, th, ph)
    assert_bitwise(got, want, "64 members")


@pytest.mark.parametrize("variant", STRATIFIED, ids=[abi.VARIANT_NAMES[v] for v in STRATIFIED])
def test_parameter_changes_between_calls(variant):
    """freq, tweak_abs, z_grnd, the source and bounces change between two ensemble calls: the second call equals the
    reference traced with the new parameters (the members' invariants are rebuilt).  Knob sbpoly = 0 also matches."""
    case = CASES[variant]
    members = members_of(case_profile(case))
    atm_id = np.repeat(np.arange(len(members), dtype=np.int32), 40)
    th, ph = seeded_angles(len(atm_id), 300 + variant)
    tr = ensemble_tracer(case, members)
    first = tr.trace_ensemble(atm_id, th, ph)
    assert_bitwise(first, reference(variant, members, tr.params, atm_id, th, ph), f"{case} before")
    p = tr.params
    p.freq, p.tweak_abs, p.z_grnd, p.bounces = 0.5, 0.7, 0.25, p.bounces + 1
    k = 0 if util.is_global(variant) else 2
    p.src[k] = 1.5
    tr.params = p
    assert_bitwise(tr.trace_ensemble(atm_id, th, ph), reference(variant, members, p, atm_id, th, ph), f"{case} after")
    tr.set_knob("sbpoly", 0)
    assert_bitwise(tr.trace_ensemble(atm_id, th, ph), reference(variant, members, p, atm_id, th, ph, {"sbpoly": 0}), f"{case} sbpoly=0")


def test_context_and_ensemble_state():
    case = "3d_sub"
    members = members_of(case_profile(case))
    tr = ensemble_tracer(case, members)
    th, ph = seeded_angles(200, 3)
    atm_id = (np.arange(200) % len(members)).astype(np.int32)
    # an ensemble call leaves the parameters, the source state and geoac_trace as they were, and reports its own statistics
    before = (bytes(tr.params), tr.source_state().tobytes(), tr.trace(th, ph))
    first = tr.trace_ensemble(atm_id, th, ph)
    steps, ms = tr.last_stats()
    assert steps == int(first["n_steps"].sum()) and ms > 0.0
    assert bytes(tr.params) == before[0] and tr.source_state().tobytes() == before[1]
    assert_bitwise(tr.trace(th, ph), before[2], "geoac_trace after an ensemble call")
    # a refused set_ensemble_1d (altitudes not increasing in member 2) leaves the ensemble tracing as before
    broken = [tuple(a.copy() for a in m) for m in members]
    broken[2][0][5] = broken[2][0][4]
    with pytest.raises(api.GeoAcError, match="member 2: altitudes must be strictly increasing"):
        tr.set_ensemble_1d(broken)
    assert_bitwise(tr.trace_ensemble(atm_id, th, ph), first, "after a refused set_ensemble_1d")
    # set_atmosphere_1d does not disturb the ensemble (the parameters it resets are put back)
    p = tr.params
    tr.set_atmosphere_1d(*members[4])
    tr.params = p
    assert_bitwise(tr.trace_ensemble(atm_id, th, ph), first, "after set_atmosphere_1d")
    # a second set_ensemble_1d with another member count replaces the first
    two = [members[3], members[1]]
    tr.set_ensemble_1d(two)
    tr.params = p
    ids2 = (np.arange(200) % 2).astype(np.int32)
    assert_bitwise(tr.trace_ensemble(ids2, th, ph), reference(abi.GEOAC_3D, two, p, ids2, th, ph), "replaced ensemble")


def test_argument_checks():
    L = api.lib()
    tr = make_tracer("3d_sub")
    members = members_of(case_profile("3d_sub"))[:2]
    n = 8
    th, ph = seeded_angles(n, 1)
    aid = np.array([0, 1] * 4, np.int32)
    rec, st, ns = np.full((abi.NFIELDS, n, 3), -7.0), np.full((n, 3), -7, np.int32), np.full((n, 3), -7, np.int32)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
    lp = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))
    msg = lambda t: L.geoac_last_error(t._h).decode()
    bad = abi.GEOAC_ERR_BAD_ARG
    # geoac_trace_ensemble before any ensemble: no atmosphere to trace through (the context's own does not count)
    targs = lambda: [n, ip(aid), dp(th), dp(ph), dp(rec), ip(st), ip(ns)]
    tcall = lambda t, a: L.geoac_trace_ensemble(t._h, *a)
    assert tcall(tr, targs()) == abi.GEOAC_ERR_NO_ATMO and "ensemble" in msg(tr)
    # geoac_set_ensemble_1d
    offs = np.array([0, len(members[0][0]), len(members[0][0]) + len(members[1][0])], np.int64)
    cols = [np.concatenate([m[k] for m in members]) for k in range(5)]
    sargs = lambda: [2, lp(offs)] + [dp(c) for c in cols]
    scall = lambda t, a: L.geoac_set_ensemble_1d(t._h, *a)
    assert L.geoac_set_ensemble_1d(None, *sargs()) == bad
    for na in (0, -1):
        a = sargs(); a[0] = na
        assert scall(tr, a) == bad and "n_atm" in msg(tr)
    for i in range(1, 7):
        a = sargs(); a[i] = None
        assert scall(tr, a) == bad and "non-null" in msg(tr), i
    for o, what in (([1, 40, 80], "level_offset[0]"), ([0, 40, 39], "member 1: level_offset"), ([0, 2, offs[2]], "member 0: need >= 3")):
        o = np.array(o, np.int64)
        a = sargs(); a[1] = lp(o)
        assert scall(tr, a) == bad and what in msg(tr), what
    rd = g.Tracer(abi.GEOAC_3D_RNGDEP, 0)
    assert scall(rd, sargs()) == bad and "stratified variants" in msg(rd)
    rd.close()
    assert scall(tr, sargs()) == abi.GEOAC_OK
    # geoac_trace_ensemble
    assert L.geoac_trace_ensemble(None, *targs()) == bad
    a = targs(); a[0] = -1
    assert tcall(tr, a) == bad and "n_rays < 0" in msg(tr)
    for i in range(1, 7):
        a = targs(); a[i] = None
        assert tcall(tr, a) == bad and "non-null" in msg(tr), i
    for v in (-1, 2, 1 << 30):
        a3 = aid.copy(); a3[5] = v; a3[6] = -1
        a = targs(); a[1] = ip(a3)
        assert tcall(tr, a) == bad and "ray 5 " in msg(tr), v
    a = targs(); a[0] = 0
    assert tcall(tr, a) == abi.GEOAC_OK
    assert tcall(tr, [0, None, None, None, None, None, None]) == abi.GEOAC_OK
    assert (rec == -7.0).all() and (st == -7).all() and (ns == -7).all()          # no refused or empty call wrote anything
    with pytest.raises(api.GeoAcError):
        tr.trace_ensemble(aid.astype(np.int64), th, ph)
    with pytest.raises(api.GeoAcError):
        tr.set_ensemble_1d([members[0][:4]])
    assert tcall(tr, targs()) == abi.GEOAC_OK and (st[:, 0] != abi.ST_NONE).all()
