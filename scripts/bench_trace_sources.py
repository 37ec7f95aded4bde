"""geoac_trace_sources against one geoac_set_params + geoac_trace per source, on the same context and rays.

  (a) small fans, many sources: 3D on ToyAtmo, 256 sources on a 16 x 16 grid of (x, y) within +-200 km, each with
      theta = 1..60 deg step 1 x 30 azimuths (1 800 rays; 460 800 in all).  Host clock around each side; both end in a
      device synchronise (the host-buffer calls do).
  (b) the cost of per-ray invariants: config 2 (216 000 rays) from one source, geoac_trace_sources vs geoac_trace,
      by kernel_ms of geoac_last_trace_stats (the trace launches only).
  (c) range dependent: config-4 grid (synth), 16 sources on a 4 x 4 grid within +-300 km, 1 000 rays each
      (theta = 1..50 deg step 1 x 20 azimuths), host clock as in (a).
Each comparison checks that both sides' records are bitwise equal.  Every shape is warmed up once, then the two sides are
alternated 5 times; the JSON gives each side's median and spread (min, max).  The card's name, power limit and max SM
clock are read (nvidia-smi --query-gpu) in the same run.

    python scripts/bench_trace_sources.py --out DIR [--reps 5] [--parts abc]
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
import bench                                    # noqa: E402  (workload set-up of config 2)

TOY = os.path.join(ROOT, "tests", "golden", "ToyAtmo.met")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def with_source(tr, s):
    p = tr.params
    p.src[0], p.src[1], p.src[2] = s
    tr.params = p


def loop_per_source(tr, src, th1, ph1):
    """One set_params + trace per source; records concatenated source by source (the batched call's layout)."""
    outs = []
    for s in src:
        with_source(tr, s)
        outs.append(tr.trace(th1, ph1))
    return {"rec": np.concatenate([o["rec"] for o in outs], axis=1), "status": np.concatenate([o["status"] for o in outs]),
            "n_steps": np.concatenate([o["n_steps"] for o in outs])}


def bitwise(a, b):
    return (np.array_equal(a["status"], b["status"]) and np.array_equal(a["n_steps"], b["n_steps"])
            and np.array_equal(np.ascontiguousarray(a["rec"]).view(np.uint64), np.ascontiguousarray(b["rec"]).view(np.uint64)))


def summary(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "all": [float(x) for x in xs]}


def alternate(reps, sides):
    """sides: {name: f() -> (value, records)}.  One warm-up call each, then reps rounds of the sides in turn."""
    recs = {k: f()[1] for k, f in sides.items()}
    names = list(sides)
    assert bitwise(recs[names[0]], recs[names[1]]), "records differ between the two sides"
    vals = {k: [] for k in names}
    for _ in range(reps):
        for k in names:
            v, r = sides[k]()
            assert bitwise(r, recs[k]), f"{k}: records changed between repetitions"
            vals[k].append(v)
    return {k: summary(v) for k, v in vals.items()}


def host_timed(f):
    t0 = time.perf_counter()
    r = f()
    return time.perf_counter() - t0, r


def many_sources(tr, src, th1, ph1, reps):
    n1 = len(th1)
    th, ph = np.tile(th1, len(src)), np.tile(ph1, len(src))
    sid = np.repeat(np.arange(len(src), dtype=np.int32), n1)
    res = alternate(reps, {"trace_sources_s": lambda: host_timed(lambda: tr.trace_sources(src, sid, th, ph)),
                           "loop_s": lambda: host_timed(lambda: loop_per_source(tr, src, th1, ph1))})
    res.update(n_sources=len(src), rays_per_source=n1, rays=len(th),
               speedup_median=res["loop_s"]["median"] / res["trace_sources_s"]["median"])
    return res


def small_fans(result, reps):
    tr = g.Tracer(abi.GEOAC_3D, 0)
    tr.set_atmosphere_1d(*g.load_met_1d(TOY))
    xy = np.linspace(-200.0, 200.0, 16)
    src = np.array([(x, y, 0.0) for x in xy for y in xy])
    _, _, th1, ph1 = g.prop_angles(1.0, 60.0, 1.0, 0.0, 348.0, 12.0)
    result["a_small_fans_3d_toy"] = many_sources(tr, src, th1, ph1, reps)
    print("(a)", json.dumps(result["a_small_fans_3d_toy"]), flush=True)
    tr.close()


def invariants_overhead(result, reps):
    tr, _ = bench.setup_tracer("config2", 0)
    _, _, th, ph = g.prop_angles(*bench.WORKLOADS["config2"][1])
    one = np.array([tr.params.src[:]])
    sid = np.zeros(len(th), np.int32)

    def kernel_ms(f):
        r = f()
        return tr.last_stats()[1], r
    res = alternate(reps, {"trace_sources_kernel_ms": lambda: kernel_ms(lambda: tr.trace_sources(one, sid, th, ph)),
                           "trace_kernel_ms": lambda: kernel_ms(lambda: tr.trace(th, ph))})
    res.update(rays=len(th), overhead_median=res["trace_sources_kernel_ms"]["median"] / res["trace_kernel_ms"]["median"] - 1.0)
    result["b_config2_one_source"] = res
    print("(b)", json.dumps(res), flush=True)
    tr.close()


def range_dependent(result, reps):
    tr = g.Tracer(abi.GEOAC_3D_RNGDEP, 0)
    tr.set_atmosphere_3d(*synth.config4_grid())
    p = tr.params
    p.bounces, p.calc_amp, p.accum_per_segment = bench.WORKLOADS["config4"][2], 1, 0
    tr.params = p
    xy = np.linspace(-300.0, 300.0, 4)
    src = np.array([(x, y, 0.0) for x in xy for y in xy])
    _, _, th1, ph1 = g.prop_angles(1.0, 50.0, 1.0, 0.0, 342.0, 18.0)
    result["c_config4_grid_16_sources"] = many_sources(tr, src, th1, ph1, reps)
    print("(c)", json.dumps(result["c_config4_grid_16_sources"]), flush=True)
    tr.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for trace_sources_<parts>.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", default="abc", help="which of the comparisons (a), (b), (c) to run")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    result = {"card": card()}
    if "a" in args.parts:
        small_fans(result, args.reps)
    if "b" in args.parts:
        invariants_overhead(result, args.reps)
    if "c" in args.parts:
        range_dependent(result, args.reps)
    with open(os.path.join(args.out, f"trace_sources_{args.parts}.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
