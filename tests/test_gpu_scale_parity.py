"""GPU parity at BASELINE.json scale: the CUDA path (through the C ABI) against the CPU oracle (bit-exact restatement of
the reference, tests/test_oracle_golden.py) on

  * config 2: every 100th ray of the 216 000-ray grid (2 160 rays),
  * config 3: every 1 000th ray of the 500 000-ray grid (500 rays),
  * config 4: 64 seeded rays on the FULL 200 x 200 x 300 node grid,
  * config 5: 64 seeded rays on the FULL 181 x 361 x 300 global grid (step limit lowered so ducted rays end on LIMIT),

with the near-threshold listing (geoac_b200/nearthreshold.py) applied; the same angles traced through geoac_trace_device (torch
buffers, the default stream) with the claim order forced on must give bitwise the records held to the oracle, which carries the
verdict over to the scheduled path the benchmark times -- the stratified sort and whole-warp refill, and for configs 4 and 5
the long region, its exclusive launch and the quarter claims.  The parity bar is discrete outputs bit-exact except on slots the
listing flags; ray position, eikonal, travel time, attenuation, turning height, inclination, back azimuth, celerity to
1e-9 on every arrival; amplitude / Jacobian / auxiliary states to 1e-9 except where a 1e-10 rad change of the launch angle
moves them by more than that (listed with |D|).  The oracle runs one process per host core (fork: the children share the
node tables and never touch CUDA)."""
import os
import sys

import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, nearthreshold as nt
from tests import util
from tests.test_gpu_device_path import assert_bitwise, trace_device

sys.path.insert(0, util.ROOT)
import bench            # noqa: E402  (workload definitions only)

pytestmark = pytest.mark.gpu

def _report(capsys, label, problems, listed, stats, n_disc, lines, n_arr):
    with capsys.disabled():
        print(f"\n[{label}] {n_arr} arrivals; max rel diff per field: " + ", ".join(f"{k}:{v:.1e}" for k, v in sorted(stats.items())))
        print(f"[{label}] listed: {n_disc} discrete differences on flagged slots, {len(listed)} amplitude / auxiliary entries beyond 1e-9 "
              f"(each within 10x its response to a 1e-10 rad change of the launch angle)")
        for i, b, name, rel, resp, D in sorted(listed, key=lambda t: -t[3])[:8]:
            print(f"    ray {i} bounce {b}: {name} differs {rel:.2e}; perturbation response {resp:.2e}; |D| = {D:.3e}")
        for ln in lines[:12]:
            print("    flagged:", ln)


def _scheduled_device_trace_equals(workload, p, th, ph, got):
    tr, _ = bench.setup_tracer(workload, 0)
    tr.params = p
    tr.set_knob("lpt", 2)
    dev = trace_device(tr, th, ph)
    assert_bitwise(dev, got, f"{workload}: geoac_trace_device, claim order forced on")
    assert tr.last_kernel_launches() > 1
    if util.is_rngdep(bench.WORKLOADS[workload][0]):
        s = tr.last_schedule()
        assert s["long_packets"] > 0 and s["long_ctas"] > 0 and s["quarter_packets"] > 0, s
    tr.close()


def _run(workload, th_deg, ph_deg, th, ph, oracle, capsys, label, chunk, ray_limit=None):
    variant = bench.WORKLOADS[workload][0]
    tr, p = bench.setup_tracer(workload, 0)
    if ray_limit:
        p.ray_limit = ray_limit
        tr.params = p
    p = tr.params
    got = tr.trace(th, ph)
    _scheduled_device_trace_equals(workload, p, th, ph, got)
    cond = nt.conditioning(tr.trace, th, ph, got, variant, p.calc_amp)
    tainted, reasons = nt.margin_flags(got, variant, p)
    # oracle on the same inputs (atmosphere built once, before the fork)
    from geoac_b200 import synth
    atmo = bench.WORKLOADS[workload][3]
    if atmo == "toy":
        at = oracle.atmo1d(False, *oracle.load_met_1d(util.TOY))
    elif atmo == "c3":
        import tempfile
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "c3.met")
            synth.write_met(path, synth.config3_profile())
            at = oracle.atmo1d(True, *oracle.load_met_1d(path, global_taper=True))
    elif atmo == "c4":
        at = oracle.atmo3d(False, *synth.config4_grid())
    else:
        at = oracle.atmo3d(True, *synth.config5_grid())
    want = util.oracle_trace_parallel(oracle, variant, at, p, th, ph, chunk)
    problems, listed, stats, n_disc = nt.check_against(got, want, variant, p.calc_amp, tainted, cond, rtol=util.RTOL, label=label)
    lines = nt.listing(got, variant, p, th_deg, ph_deg, cond=None)
    n_arr = int((got["status"] == abi.ST_ARRIVAL).sum())
    _report(capsys, label, problems, listed, stats, n_disc, lines, n_arr)
    assert not problems, "\n".join(problems)
    # sanity next to the verdict: the bulk of the amplitudes agrees far below the tolerance (the tail is the listed, ill-conditioned
    # class -- it grows with the number of reflections: config 3 traces five bounces over 3 000 km)
    m = (got["status"] == abi.ST_ARRIVAL) & (want["status"] == abi.ST_ARRIVAL) & ~tainted & ~cond["flips"]
    if p.calc_amp and m.any():
        a, b = got["rec"][abi.F_AMPLITUDE][m], want["rec"][abi.F_AMPLITUDE][m]
        rel = np.abs(a - b) / np.abs(b)
        with capsys.disabled():
            print(f"[{label}] amplitude rel diff: median {np.median(rel):.1e}, 90 % {np.quantile(rel, 0.9):.1e}, max {rel.max():.1e}; "
                  f"{int((rel <= util.RTOL).sum())} of {rel.size} within 1e-9")
        assert np.median(rel) <= util.RTOL, np.median(rel)
    assert n_disc <= max(2, 0.001 * got["status"].size)
    return got, want


def test_config2_every_100th_ray_matches_the_oracle(oracle, capsys):
    _, th_deg, ph_deg, th, ph = bench.workload_angles("config2")
    idx = np.arange(0, len(th), 100)
    got, _ = _run("config2", th_deg[idx], ph_deg[idx], th[idx].copy(), ph[idx].copy(), oracle, capsys, "config 2 / 2160 rays", chunk=16)
    assert (got["status"] == abi.ST_ARRIVAL).sum() > 4000


def test_config3_every_1000th_ray_matches_the_oracle(oracle, capsys):
    _, th_deg, ph_deg, th, ph = bench.workload_angles("config3")
    idx = np.arange(0, len(th), 1000)
    got, _ = _run("config3", th_deg[idx], ph_deg[idx], th[idx].copy(), ph[idx].copy(), oracle, capsys, "config 3 / 500 rays", chunk=4)
    assert (got["status"] == abi.ST_ARRIVAL).sum() > 500


def _seeded(n, seed, th_lo=1.0, th_hi=50.95):
    rng = np.random.default_rng(seed)
    th_deg, ph_deg = rng.uniform(th_lo, th_hi, n), rng.uniform(0.0, 360.0, n)
    return th_deg, ph_deg, th_deg * util.PI / 180.0, util.PI / 2.0 - ph_deg * util.PI / 180.0


def test_config4_full_grid_seeded_rays_match_the_oracle(oracle, capsys):
    th_deg, ph_deg, th, ph = _seeded(64, 20251101)
    got, _ = _run("config4", th_deg, ph_deg, th, ph, oracle, capsys, "config 4 / full 200x200x300 grid / 64 rays", chunk=1)
    assert (got["status"] == abi.ST_ARRIVAL).sum() > 64


def test_config5_full_grid_seeded_rays_match_the_oracle(oracle, capsys):
    th_deg, ph_deg, th, ph = _seeded(64, 20251102)
    got, _ = _run("config5", th_deg, ph_deg, th, ph, oracle, capsys, "config 5 / full 181x361x300 grid / 64 rays", chunk=1, ray_limit=300.0)
    st = got["status"]
    assert (st == abi.ST_ARRIVAL).sum() > 32 and (st != abi.ST_NONE).any(axis=1).all()
