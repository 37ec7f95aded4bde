"""geoac_eigenray_search_sources -- eigenray searches from many sources in one call -- against one geoac_eigenray_search per
(source, receiver), bit for bit (column 0, the search index, aside), for 3D, 3D.RngDep, Global and Global.RngDep; against
the unmodified reference's golden cases placed among other sources; the rounds shared between searches; the contract on
the context's parameters and the argument checks; and the raypaths of the eigenrays found, traced from their sources by
geoac_trace_sources_paths_compact, against geoac_trace_paths_compact per source."""
import ctypes as C

import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, api
from tests import util
from tests.test_eigenray import check_attributes, check_rows, is_glob, load, opts_from, receiver

pytestmark = pytest.mark.gpu

OPTS = dict(bnc_min=0, bnc_max=2, azimuth_err_lim=0.5, iterations=12)
# per variant: the grid of a golden case for the range-dependent sets (ToyAtmo otherwise), the sources -- as
# geoac_eigenray_search_sources takes them -- and the receivers of each source relative to it (km, or degrees)
SETUPS = {
    abi.GEOAC_3D: (None, [(0.0, 0.0, 0.0), (120.0, -40.0, 0.0), (-60.0, 80.0, 1.5), (30.0, 60.0, -2.0)],
                   [(-250.0, 0.0), (180.0, 170.0), (40.0, -290.0), (-200.0, -150.0)]),
    abi.GEOAC_GLOBAL: (None, [(0.0, 30.0, 0.0), (0.8, 41.5, 12.25), (0.0, -20.0, 45.0), (-1.0, 60.0, -100.0)],
                       [(0.0, -2.5), (1.1, -3.35), (-2.0, 1.5), (2.2, 0.8)]),
    abi.GEOAC_3D_RNGDEP: ("eig3drngdep", [(13.7, -21.3, 0.0), (-150.0, 120.0, 0.0), (160.0, -90.0, 0.5), (90.0, 200.0, -1.0)],
                          [(-243.7, 116.3), (-230.0, -40.0), (220.0, 60.0)]),
    abi.GEOAC_GLOBAL_RNGDEP: ("eigglobalrngdep", [(0.0, 33.3, 1.7), (0.0, 37.0, -6.0), (0.5, 41.0, 3.0), (-1.0, 35.5, -2.5)],
                              [(0.8, -2.9), (-1.0, 2.0), (1.5, 1.0)]),
}


def tracer(variant, grid_case=None):
    tr = g.Tracer(variant, 0)
    if grid_case:
        tr.set_atmosphere_3d(*util.load_grid(load(grid_case)[0]))
    else:
        tr.set_atmosphere_1d(*g.load_met_1d(util.TOY, global_taper=is_glob(variant)))
    return tr


def searches(variant, seed):
    """Sources, a shuffled src_id and the receivers of every (source, receiver) pair of SETUPS."""
    _, src, rel = SETUPS[variant]
    pairs = [(s, (src[s][1] + dx, src[s][2] + dy) if is_glob(variant) else (src[s][0] + dx, src[s][1] + dy))
             for s in range(len(src)) for dx, dy in rel]
    perm = np.random.default_rng(seed).permutation(len(pairs))
    return np.array(src), np.array([pairs[k][0] for k in perm], np.int32), np.array([pairs[k][1] for k in perm])


def one_search(tr, variant, s, rcv, **opts):
    """geoac_eigenray_search for one receiver on `tr` from source s (a row of geoac_eigenray_search_sources' src)."""
    p = tr.params
    before = bytes(p)
    if is_glob(variant):
        p.src[0] = s[0]
        opts = dict(opts, src_lat_deg=s[1], src_lon_deg=s[2])
    else:
        p.src[0], p.src[1], p.src[2] = s
    tr.params = p
    rows, st = tr.eigenray_search([rcv], **opts)
    p = abi.GeoacParams.from_buffer_copy(before)
    tr.params = p
    return rows, st


def masked(rows):
    r = rows.copy()
    r[:, 0] = 0
    return r.view(np.uint64)


@pytest.mark.parametrize("variant", sorted(SETUPS), ids=[abi.VARIANT_NAMES[v] for v in sorted(SETUPS)])
def test_equals_one_search_per_source(variant):
    tr = tracer(variant, SETUPS[variant][0])
    src, sid, rcv = searches(variant, 20261022 + variant)
    before = bytes(tr.params)
    rows, stats = tr.eigenray_search_sources(src, sid, rcv, **OPTS)
    assert bytes(tr.params) == before
    assert np.array_equal(rows[:, 0], np.sort(rows[:, 0], kind="stable")), "rows in search order"
    rounds = 0
    for i in range(len(sid)):
        want, st = one_search(tr, variant, src[sid[i]], rcv[i], **OPTS)
        rounds += st["rounds"]
        assert np.array_equal(masked(rows[rows[:, 0] == i]), masked(want)), (i, sid[i], rcv[i])
    assert stats["found"] == int(rows[:, 6].sum()) > 0
    assert (rows[:, 16] > 1).any(), "LM iterations ran"
    assert stats["rounds"] < rounds, (stats, rounds)                # the searches share their rounds
    print(f"\n[{abi.VARIANT_NAMES[variant]}] {len(sid)} searches: {stats['rounds']} rounds in one call, {rounds} one by one; "
          f"{stats['found']} eigenrays; {tr.last_eigenray_ms()}")
    # the raypaths of the eigenrays found (the <title>_Eigenray-N.dat files), traced from their sources in one call
    found = rows[rows[:, 6] == 1]
    sid_f = sid[found[:, 0].astype(int)]
    th, ph = found[:, 7] * util.PI / 180.0, found[:, 8] * util.PI / 180.0          # as the search launches them
    tsrc = np.array([(s[0], s[1] * util.PI / 180.0, s[2] * util.PI / 180.0) if is_glob(variant) else s for s in src])   # params.src convention
    p = tr.params
    p.bounces, p.calc_amp, p.accum_per_segment = int(found[:, 1].max()), 1, 1
    tr.params = p
    got = tr.trace_sources_paths_compact(tsrc, sid_f, th, ph, 25, 4000)
    for s in np.unique(sid_f):
        idx = np.flatnonzero(sid_f == s)
        q = tr.params
        q.src[0], q.src[1], q.src[2] = tsrc[s]
        tr.params = q
        want = tr.trace_paths_compact(th[idx], ph[idx], 25, 4000)
        for j, r in enumerate(idx):
            a = got["path"][got["path_offset"][r]:got["path_offset"][r + 1]]
            b = want["path"][want["path_offset"][j]:want["path_offset"][j + 1]]
            assert len(a) > 0 and np.array_equal(a.view(np.uint64), b.view(np.uint64)), (s, r)
        assert np.array_equal(got["rec"][:, idx].view(np.uint64), want["rec"].view(np.uint64))


GOLDEN = ["eig3d_axis", "eig3d_east", "eigglobal_nw", "eig3drngdep", "eigglobalrngdep"]


@pytest.mark.parametrize("name", GOLDEN)
def test_golden_case_among_other_sources(name):
    """The reference's (source, receiver, opts) as one search of a call with other sources and receivers: its rows are the
    reference's."""
    d, kv = load(name)
    variant = int(d["variant"])
    tr = tracer(variant, name if util.is_rngdep(variant) else None)
    if is_glob(variant):
        gsrc = (float(kv.get("z_src", 0.0)), float(kv.get("lat_src", 30.0)), float(kv.get("lon_src", 0.0)))
    else:
        gsrc = (float(kv.get("x_src", 0.0)), float(kv.get("y_src", 0.0)), float(kv.get("z_src", 0.0)))
    others = [s for s in SETUPS[variant][1] if tuple(s) != gsrc][-2:]
    src = np.array([others[0], gsrc, others[1]])
    grc = receiver(kv, variant)
    rcv = np.array([(others[0][1] + 0.9, others[0][2] - 1.2) if is_glob(variant) else (others[0][0] - 240.0, others[0][1] + 30.0),
                    grc, grc, (others[1][1] - 1.0, others[1][2] + 1.0) if is_glob(variant) else (others[1][0] + 150.0, others[1][1] - 200.0)])
    sid = np.array([0, 1, 2, 2], np.int32)
    opts = {k: v for k, v in opts_from(kv).items() if not k.startswith("src_")}
    rows, stats = tr.eigenray_search_sources(src, sid, rcv, **opts)
    mine = rows[rows[:, 0] == 1]
    check_rows(mine, d["rows"], name)
    check_attributes(mine, str(d["text"]), name)


def test_contract_and_argument_checks():
    L = api.lib()
    tr = tracer(abi.GEOAC_3D)
    p = tr.params
    p.src[0], p.src[1], p.src[2] = 5.0, -7.0, 0.25
    tr.params = p
    before = bytes(tr.params)
    src = np.array([(0.0, 0.0, 0.0), (40.0, 10.0, 0.0)])
    sid = np.array([1, 0, 1], np.int32)
    rcv = np.array([(-210.0, 10.0), (-250.0, 0.0), (-180.0, -90.0)])
    o = abi.GeoacEigOpts()
    L.geoac_default_eig_opts(C.byref(o))
    o.bnc_max = 1
    dp = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))
    ip = lambda a: None if a is None else a.ctypes.data_as(C.POINTER(C.c_int32))
    rows = np.full((64, abi.EIG_NF), -7.0)
    n_rows, stats = C.c_int64(-1), (C.c_int64 * 3)()
    args = lambda: [C.byref(o), len(src), dp(src), len(sid), ip(sid), dp(rcv), 64, dp(rows), C.byref(n_rows), stats]
    call = lambda t, a: L.geoac_eigenray_search_sources(t._h, *a)
    msg = lambda t: L.geoac_last_error(t._h).decode()
    bad = abi.GEOAC_ERR_BAD_ARG
    # success, and the parameters as they were
    assert call(tr, args()) == abi.GEOAC_OK and bytes(tr.params) == before
    n_ok = n_rows.value
    assert 0 < n_ok < 64 and (rows[n_ok:] == -7.0).all()
    want = rows[:n_ok].copy()
    # too few rows: GEOAC_ERR_TOO_LARGE, n_rows set, the rows that fit written
    rows[:] = -7.0
    a = args(); a[6] = n_ok - 1
    assert call(tr, a) == abi.GEOAC_ERR_TOO_LARGE and n_rows.value == n_ok and bytes(tr.params) == before
    assert np.array_equal(rows[: n_ok - 1].view(np.uint64), want[: n_ok - 1].view(np.uint64)) and (rows[n_ok - 1:] == -7.0).all()
    # refused arguments: their code and a message, nothing written, the parameters as they were
    rows[:] = -7.0
    n_rows.value = -1
    assert L.geoac_eigenray_search_sources(None, *args()) == bad
    refusals = [((0, None), "non-null"), ((8, None), "non-null"), ((2, None), "non-null"), ((4, None), "non-null"), ((5, None), "non-null"),
                ((7, None), "non-null"), ((3, -1), "n_rcvr < 0"), ((1, 0), "n_src >= 1")]
    for (k, v), words in refusals:
        a = args(); a[k] = v
        assert call(tr, a) == bad and words in msg(tr), (k, v, msg(tr))
    for v in (np.nan, np.inf):
        s2 = src.copy(); s2[1, 1] = v
        a = args(); a[2] = dp(s2)
        assert call(tr, a) == bad and "source 1 " in msg(tr)
    for v in (-1, 2):
        s3 = sid.copy(); s3[2] = v
        a = args(); a[4] = ip(s3)
        assert call(tr, a) == bad and "search 2 " in msg(tr)
    for field, v in (("bnc_min", 2), ("iterations", -1), ("d_theta_big", 0.0)):
        o2 = abi.GeoacEigOpts.from_buffer_copy(bytes(o))
        setattr(o2, field, v)
        a = args(); a[0] = C.byref(o2)
        assert call(tr, a) == bad and "eigenray options" in msg(tr), field
    assert (rows == -7.0).all() and n_rows.value == -1 and bytes(tr.params) == before
    tr2 = g.Tracer(abi.GEOAC_2D, 0)
    tr2.set_atmosphere_1d(*g.load_met_1d(util.TOY))
    assert call(tr2, args()) == bad and "3-D" in msg(tr2)
    bare = g.Tracer(abi.GEOAC_3D, 0)
    assert call(bare, args()) == abi.GEOAC_ERR_NO_ATMO
    # no searches: GEOAC_OK, zero rows, nothing written
    a = args(); a[3] = 0; a[2] = None; a[4] = None; a[5] = None
    assert call(tr, a) == abi.GEOAC_OK and n_rows.value == 0 and (rows == -7.0).all() and bytes(tr.params) == before
    # the timing of the last search
    ms = tr.last_eigenray_ms()
    assert ms["kernel_ms"] >= 0.0 and ms["replay_ms"] >= 0.0 and ms["call_ms"] >= ms["replay_ms"]
