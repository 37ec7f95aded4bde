"""GPU parity tests (run on a real B200 with `-m gpu`): the CUDA path, called through the C ABI, against
 (1) the committed golden vectors dumped from the unmodified reference, and
 (2) the CPU oracle on freshly seeded launch angles,
discrete outputs bit-exact, continuous outputs within RTOL = 1e-9 relative (tests/util.py)."""
import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, nearthreshold as nt
from tests import util

pytestmark = pytest.mark.gpu


def _tracer_for(variant, kv, case=None):
    tr = g.Tracer(variant, 0)
    if util.is_rngdep(variant):
        tr.set_atmosphere_3d(*util.load_grid(case))
    else:
        z, T, u, v, rho = g.load_met_1d(util.profile_path(case) if case is not None else util.TOY, global_taper=util.is_global(variant))
        tr.set_atmosphere_1d(z, T, u, v, rho)
    tr.params = util.apply_keys(variant, tr.params, kv)
    return tr


# Amplitude, Jacobian and the auxiliary (launch-angle derivative) states are ill-conditioned near caustic-forming rays (their
# condition number with respect to the launch angle reaches 1e9): such an entry may differ from the reference by more than
# 1e-9 ONLY where a 1e-10 rad change of the launch angle moves it by more than a tenth of that difference, and is then
# listed with |D| (geoac_b200/nearthreshold.py).  Everything else -- positions, eikonal, travel time, attenuation, turning
# height, inclination, back azimuth, celerity -- is held to 1e-9 on every arrival, discrete outputs to equality.
AMP_RTOL = 1e-6          # raypath rows only (amplitude sampled along the path passes through caustics)


def _verdict(tr, variant, th, ph, out, want, label, capsys=None):
    calc_amp = tr.params.calc_amp
    cond = nt.conditioning(tr.trace, th, ph, out, variant, calc_amp)
    tainted, _ = nt.margin_flags(out, variant, tr.params)
    problems, listed, stats, n_disc = nt.check_against(out, want, variant, calc_amp, tainted, cond, rtol=util.RTOL, label=label)
    if capsys is not None:
        with capsys.disabled():
            print(f"\n[{label}] max rel diff per field: " + ", ".join(f"{k}:{v:.1e}" for k, v in sorted(stats.items())))
            for i, b, name, rel, resp, D in listed:
                print(f"   listed: ray {i} bounce {b}: {name} differs {rel:.2e} (moves {resp:.2e} under a 1e-10 rad change of the launch angle; |D| = {D:.3e})")
    return problems, listed, n_disc, tainted


@pytest.mark.parametrize("name", util.golden_cases())
def test_cuda_matches_reference_golden(name, capsys):
    d, kv = util.load_case(name)
    variant = int(d["variant"])
    tr = _tracer_for(variant, kv, d)
    th, ph = util.angles_rad(d["theta_deg"], d["phi_deg"])
    out = tr.trace(th, ph)
    want = {"rec": d["rec"], "status": d["status"], "n_steps": d["n_steps"]}
    problems, listed, n_disc, tainted = _verdict(tr, variant, th, ph, out, want, name, capsys)
    assert not problems, "\n".join(problems)
    assert n_disc == 0 and not tainted.any()          # the golden sets hold no near-threshold ray: discrete outputs equal everywhere


@pytest.mark.parametrize("name", util.path_cases())
def test_cuda_raypath_rows_match_reference(name):
    """WriteRays=True rows through geoac_trace_paths: row counts / bounce / step indices exact, positions and sums to 1e-9,
    the amplitude along the path (singular at caustics) to 1e-6."""
    d, kv = util.load_case(name)
    variant = int(d["variant"])
    tr = _tracer_for(variant, kv, d)
    th, ph = util.angles_rad(d["theta_deg"], d["phi_deg"])
    cap = 2000
    out = tr.trace_paths(th, ph, int(kv["path_stride"]), cap, caustic_cap=32)
    want_path, want_rows = util.golden_paths(d, cap)
    problems = util.compare_paths(out["path"], out["path_rows"], want_path, want_rows, util.RTOL, 1e-6, name)
    want_c, want_crows = util.golden_caustics(d, 32)                     # WriteCaustics=True events
    problems += util.compare_caustics(out["caustic"], out["caustic_rows"], want_c, want_crows, util.RTOL, name)
    only_c = tr.trace_paths(th, ph, 0, 0, caustic_cap=32)               # events without raypath rows
    assert np.array_equal(only_c["caustic"], out["caustic"]) and np.array_equal(only_c["caustic_rows"], out["caustic_rows"])
    want = {"rec": d["rec"], "status": d["status"], "n_steps": d["n_steps"]}
    rp, _, _, _ = _verdict(tr, variant, th, ph, out, want, name)
    assert not (problems + rp), "\n".join((problems + rp)[:10])
    # compacted rows (geoac_trace_paths_compact): the same rows, ray after ray, with offsets; a too-small buffer is reported and retried
    cp = tr.trace_paths_compact(th, ph, int(kv["path_stride"]), cap, caustic_cap=32, total_rows=7)
    assert np.array_equal(np.diff(cp["path_offset"]), out["path_rows"]) and np.array_equal(np.diff(cp["caustic_offset"]), out["caustic_rows"])
    for i in range(len(th)):
        assert np.array_equal(cp["path"][cp["path_offset"][i]:cp["path_offset"][i + 1]], out["path"][i, :out["path_rows"][i]])
        assert np.array_equal(cp["caustic"][cp["caustic_offset"][i]:cp["caustic_offset"][i + 1]], out["caustic"][i, :out["caustic_rows"][i]])
    assert np.array_equal(cp["rec"], out["rec"]) and np.array_equal(cp["status"], out["status"])
    # a row capacity that is too small drops the surplus rows but still reports how many were produced
    small = tr.trace_paths(th, ph, int(kv["path_stride"]), 5)
    assert np.array_equal(small["path_rows"], want_rows) and np.array_equal(small["path"][:, :5], out["path"][:, :5])


def test_cuda_matches_oracle_seeded(oracle, capsys):
    """Freshly seeded launch angles, the three stratified variants on ToyAtmo (the range-dependent ones are seeded on the
    full config-4 / config-5 grids in tests/test_gpu_scale_parity.py)."""
    rng = np.random.default_rng(20251018)
    n = 96
    theta_deg = rng.uniform(2.0, 55.0, n)
    phi_deg = rng.uniform(-180.0, 180.0, n)
    th, ph = util.angles_rad(theta_deg, phi_deg)
    for variant in (abi.GEOAC_3D, abi.GEOAC_2D, abi.GEOAC_GLOBAL):
        tr = _tracer_for(variant, {"bounces": 1})
        out = tr.trace(th, ph)
        glob = variant == abi.GEOAC_GLOBAL
        at = oracle.atmo1d(glob, *oracle.load_met_1d(util.TOY, global_taper=glob))
        want = util.oracle_trace_parallel(oracle, variant, at, tr.params, th, ph)
        problems, listed, n_disc, tainted = _verdict(tr, variant, th, ph, out, want, f"seeded variant {variant}", capsys)
        assert not problems, "\n".join(problems)
        assert n_disc == 0


def test_edge_cases():
    tr = _tracer_for(abi.GEOAC_3D, {"bounces": 0})
    # empty batch
    out = tr.trace(np.zeros(0), np.zeros(0))
    assert out["status"].shape == (0, 1)
    # a single ray, and a ragged batch that is not a multiple of the warp size
    for n in (1, 33):
        th, ph = util.angles_rad(np.linspace(5, 30, n), np.full(n, -90.0))
        out = tr.trace(th, ph)
        assert (out["status"][:, 0] != abi.ST_NONE).all()
    # a ray shot straight up leaves the region: BREAK, no arrival record (SURVEY App. A-19)
    th, ph = util.angles_rad([89.0], [-90.0])
    out = tr.trace(th, ph)
    assert out["status"][0, 0] == abi.ST_BREAK and out["rec"][abi.F_TRAVELTIME, 0, 0] == 0.0


def test_batch_order_independence_and_determinism():
    """Rays are claimed dynamically by whichever lane is free; results must not depend on that (bitwise)."""
    tr = _tracer_for(abi.GEOAC_3D, {"bounces": 1})
    _, _, th, ph = g.prop_angles(1, 60.5, 1, 0, 359, 40)
    a = tr.trace(th, ph)
    perm = np.random.default_rng(1).permutation(len(th))
    b = tr.trace(th[perm], ph[perm])
    assert np.array_equal(a["status"][perm], b["status"])
    assert np.array_equal(a["n_steps"][perm], b["n_steps"])
    assert np.array_equal(a["rec"][:, perm, :], b["rec"])


def test_longest_ray_first_schedule_is_result_neutral(monkeypatch):
    """The cost scout + counting sort only change the order in which lanes claim rays: records must be bitwise identical
    with the schedule forced on (knob lpt = 2) and off (=0), for a stratified and a range-dependent variant."""
    for case in ("3d_sub", "globalrngdep_sub"):
        d, kv = util.load_case(case)
        variant = int(d["variant"])
        th, ph = util.angles_rad(d["theta_deg"], d["phi_deg"])
        outs = []
        for mode in ("0", "2"):
            tr = _tracer_for(variant, kv, d)
            tr.set_knob("lpt", int(mode))
            outs.append(tr.trace(th, ph))
            n_k = tr.last_kernel_launches()          # scout (+ cost dilation) + sort kernels (+ long-region launch) + trace kernel
            assert n_k == 1 if mode == "0" else (n_k >= 5 if util.is_rngdep(variant) else n_k == 10)
        assert np.array_equal(outs[0]["status"], outs[1]["status"]) and np.array_equal(outs[0]["n_steps"], outs[1]["n_steps"])
        assert np.array_equal(outs[0]["rec"], outs[1]["rec"])


def test_multi_context_sharding_is_bitwise_identical():
    """SURVEY 8e: the batch split over several contexts (here two contexts on the one GPU of the test box, driven from
    host threads like a multi-GPU front end) gives bitwise the records of a single-context trace."""
    from geoac_b200 import sharding
    kv = {"bounces": 1}
    _, _, th, ph = g.prop_angles(1, 60.5, 1, 0, 359, 24)
    one = _tracer_for(abi.GEOAC_3D, kv).trace(th, ph)
    two = sharding.trace_multi([_tracer_for(abi.GEOAC_3D, kv), _tracer_for(abi.GEOAC_3D, kv)], th, ph, block=64)
    assert np.array_equal(one["status"], two["status"]) and np.array_equal(one["n_steps"], two["n_steps"])
    assert np.array_equal(one["rec"], two["rec"])


def test_library_multi_device_path_is_bitwise_identical():
    """geoac_trace_multi (host threads, interleaved 4096-ray blocks, pinned staging and merge INSIDE the library -- what a C++
    front end with one context per GPU calls): three contexts on the one GPU of the test box == one context, bit for bit; a
    ragged tail block, the geoac_create_multi / geoac_multi_set_* helpers, and the mismatch error path."""
    from geoac_b200 import api
    _, _, th, ph = g.prop_angles(1, 60.5, 1, 0, 359.9, 1.7)          # 12 720 rays: 3 full blocks + a ragged one
    kv = {"bounces": 1}
    one = _tracer_for(abi.GEOAC_3D, kv).trace(th, ph)
    trs = [_tracer_for(abi.GEOAC_3D, kv) for _ in range(3)]
    multi = api.trace_multi(trs, th, ph)
    for k in ("status", "n_steps", "rec"):
        assert np.array_equal(one[k], multi[k]), k
    mt = api.MultiTracer(abi.GEOAC_3D, [0, 0])
    mt.set_atmosphere_1d(*g.load_met_1d(util.TOY))
    mt.params = util.apply_keys(abi.GEOAC_3D, mt.params, kv)
    two = mt.trace(th[:5000], ph[:5000])
    for k in ("status", "n_steps"):
        assert np.array_equal(one[k][:5000], two[k]), k
    assert np.array_equal(one["rec"][:, :5000], two["rec"])
    assert mt.trace(th[:0], ph[:0])["status"].shape == (0, 2)
    bad = _tracer_for(abi.GEOAC_3D, {"bounces": 2})
    with pytest.raises(g.GeoAcError):
        api.trace_multi([trs[0], bad], th[:10], ph[:10])
    mt.close()


def test_reciprocity_at_scale():
    """Size-independent property at a config-2-like scale slice: in a stratified medium the n-th bounce range of
    the 2-D solver is (n+1) times the first (SURVEY 8c) -- checked on 4k rays without any oracle."""
    tr = _tracer_for(abi.GEOAC_2D, {"bounces": 2})
    _, _, th, ph = g.prop_angles(0.5, 45.0, 0.011, -90.0, -90.0, 1.0)
    out = tr.trace(th, ph)
    ok = (out["status"] == abi.ST_ARRIVAL).all(axis=1)
    r = out["rec"][0][ok]
    assert ok.sum() > 2000
    d2, d3 = np.abs(r[:, 1] / r[:, 0] / 2.0 - 1.0), np.abs(r[:, 2] / r[:, 0] / 3.0 - 1.0)
    # the reflection restarts from an approximate intercept, so the periodicity holds to ~1e-6, except for the few rays
    # that sit on the edge between two ducts (a tiny perturbation at the bounce sends them to another turning height)
    assert np.quantile(d2, 0.99) < 1e-4 and np.quantile(d3, 0.99) < 1e-4
    assert (d3 > 2e-3).sum() <= 0.005 * len(d3)


def test_branch_free_math_primitives():
    """The hot loop's own reciprocal / rsqrt / sqrt / exp / 10^x / sincos (core.cuh) against the CUDA math library on
    random operands: <= 4 ulp (9e-16 relative; absolute for sin / cos) -- seven orders inside the 1e-9 parity budget."""
    tr = g.Tracer(abi.GEOAC_3D, 0)
    errs = tr.selftest_math(4000)
    assert all(0.0 <= e < 9e-16 for e in errs.values()), errs
