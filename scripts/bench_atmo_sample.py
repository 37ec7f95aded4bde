"""Throughput of geoac_sample_atmosphere: 1e7 seeded points, uniform in the domain, on ToyAtmo (3D), the config-3 profile
(Global), the full config-4 grid (200 x 200 x 300) and the full config-5 grid (181 x 361 x 300).

For each atmosphere, after one warm-up call of the same size:
  e2e     host clock around the synchronous call (coordinates in, 38 rows out through pageable memory)
  kernel  sum of the sample_atmosphere_kernel durations of a second call, from torch.profiler (CUDA activities)
The oracle's single-core rate on 2000 of the points is printed for scale (on the committed config-4 / config-5 fixtures for
the grids: the same formulas on a smaller horizontal grid; its per-point cost does not depend on the grid size).

    python scripts/bench_atmo_sample.py [--points 10000000] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import geoac_b200 as g                          # noqa: E402
from geoac_b200 import abi, synth               # noqa: E402

R_EARTH = 6370.0


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def atmospheres(tmp):
    c3 = os.path.join(tmp, "c3.met")
    synth.write_met(c3, synth.config3_profile())
    toy = os.path.join(ROOT, "tests", "golden", "ToyAtmo.met")
    return [
        ("toy_3d", abi.GEOAC_3D, "profile", lambda: g.load_met_1d(toy), "grid_none"),
        ("config3_global", abi.GEOAC_GLOBAL, "profile", lambda: g.load_met_1d(c3, global_taper=True), "grid_none"),
        ("config4_grid", abi.GEOAC_3D_RNGDEP, "grid", lambda: synth.config4_grid(), "grid_c4"),
        ("config5_grid", abi.GEOAC_GLOBAL_RNGDEP, "grid", lambda: synth.config5_grid(), "grid_c5"),
    ]


def domain_points(variant, kind, arrays, n, seed):
    rng = np.random.default_rng(seed)
    glob = variant in (abi.GEOAC_GLOBAL, abi.GEOAC_GLOBAL_RNGDEP)
    if kind == "profile":
        z = np.asarray(arrays[0])
        if glob:
            lo, hi = [z[0] + R_EARTH, -1.2, -3.0], [z[-1] + R_EARTH, 1.2, 3.0]
        else:
            lo, hi = [-800.0, -800.0, z[0]], [800.0, 800.0, z[-1]]
    else:
        ax0, ax1, axz = arrays[:3]
        if glob:
            lo, hi = [axz[0] + R_EARTH, ax0[0], ax1[0]], [axz[-1] + R_EARTH, ax0[-1], ax1[-1]]
        else:
            lo, hi = [ax0[0], ax1[0], axz[0]], [ax0[-1], ax1[-1], axz[-1]]
    return [np.ascontiguousarray(rng.uniform(lo[j], hi[j], n)) for j in range(3)]


def kernel_ms(tr, pts):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        tr.sample_atmosphere(*pts)
        torch.cuda.synchronize()
    us = [e.device_time for e in prof.events() if "sample_atmosphere_kernel" in e.name]
    return (sum(us) / 1000.0, len(us)) if us else (None, 0)


def oracle_rate(variant, kind, arrays, fixture, pts):
    from oracle import pyoracle as po
    from tests import atmo_sample_cases as S
    po.build()
    glob = variant in (abi.GEOAC_GLOBAL, abi.GEOAC_GLOBAL_RNGDEP)
    if kind == "grid":
        arrays = S.grid(fixture)
        pts = domain_points(variant, kind, arrays, 2000, 11)
    p = po.default_params(variant)
    at = po.atmo1d(glob, *arrays) if kind == "profile" else po.atmo3d(glob, *arrays)
    sub = [a[:2000] for a in pts]
    t0 = time.perf_counter()
    S.oracle_rows(po, at, sub, p.freq)
    return len(sub[0]) / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=10_000_000)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import tempfile
    tmp = tempfile.mkdtemp(prefix="atmo_bench")
    res = {"card": card(), "points": a.points, "cases": []}
    print("card (name, power limit, max SM clock):", res["card"], flush=True)
    for label, variant, kind, load, fixture in atmospheres(tmp):
        arrays = load()
        tr = g.Tracer(variant, 0)
        if kind == "profile":
            tr.set_atmosphere_1d(*arrays)
        else:
            tr.set_atmosphere_3d(*arrays)
        pts = domain_points(variant, kind, arrays, a.points, a.seed)
        tr.sample_atmosphere(*pts)                                   # warm-up: module load, staging allocation
        t0 = time.perf_counter()
        tr.sample_atmosphere(*pts)
        e2e = time.perf_counter() - t0
        kms, launches = kernel_ms(tr, pts)
        orc = oracle_rate(variant, kind, arrays, fixture, pts)
        r = {"case": label, "e2e_s": e2e, "e2e_points_per_s": a.points / e2e, "kernel_ms": kms, "kernel_launches": launches,
             "kernel_points_per_s": (a.points / (kms * 1e-3)) if kms else None, "oracle_1core_points_per_s": orc}
        res["cases"].append(r)
        print(json.dumps(r), flush=True)
        tr.close()
        del arrays, pts
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
