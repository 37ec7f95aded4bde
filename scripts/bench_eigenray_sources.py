"""geoac_eigenray_search_sources against the loop of geoac_set_params + geoac_eigenray_search per source, on the same context.

  (a) 3D on ToyAtmo: 64 sources on an 8 x 8 grid of (x, y) within +-200 km, 16 receivers on a ring of radius 250 km
      around the origin searched from every source (1 024 searches), bounce counts 0-2.
  (b) 3D.RngDep on the config-4 grid fixture of the tests (tests/golden/grid_c4.npz): 4 sources on a 2 x 2 grid within
      +-100 km, 8 receivers on a ring of radius 220 km, bounce counts 0-1.
Both sides end in a device synchronise (the host-buffer calls do); host clock around each.  Each comparison checks that the
rows of the two sides are bitwise equal (the search index of column 0 aside), warms up once, then alternates the two sides
--reps times; the JSON gives each side's median and spread (min, max), the rounds and rays of each side, and for the
many-source call where its time went (geoac_last_eigenray_ms: host time replaying the searches, kernel time of its traces
summed, the whole call).  The card's name, power limit and max SM clock are read (nvidia-smi --query-gpu) in the same run.

    python scripts/bench_eigenray_sources.py --out DIR [--reps 5] [--parts ab]
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
from geoac_b200 import abi                      # noqa: E402
from tests import util                          # noqa: E402  (the grid fixture)

TOY = os.path.join(ROOT, "tests", "golden", "ToyAtmo.met")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    return q[0] if q else "unknown"


def ring(n, radius):
    a = np.arange(n) * 2.0 * np.pi / n
    return np.stack([radius * np.cos(a), radius * np.sin(a)], axis=1)


def stats_of(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs))}


def compare(tr, src, rcv, opts, reps):
    """One many-source call against the per-source loop; each source searches every receiver."""
    sid = np.repeat(np.arange(len(src), dtype=np.int32), len(rcv))
    rcv_all = np.tile(rcv, (len(src), 1))
    cap = len(sid) * (opts["bnc_max"] - opts["bnc_min"] + 1) * 16

    def batched():
        rows, st = tr.eigenray_search_sources(src, sid, rcv_all, cap_rows=cap, **opts)
        return rows, st, tr.last_eigenray_ms()

    def loop():
        p0 = tr.params
        rows, rounds, rays, found, kms = [], 0, 0, 0, 0.0
        for s in range(len(src)):
            p = tr.params
            p.src[0], p.src[1], p.src[2] = src[s]
            tr.params = p
            r, st = tr.eigenray_search(rcv, cap_rows=cap, **opts)
            r[:, 0] += s * len(rcv)                    # receiver index -> search index of the batched call
            rows.append(r)
            rounds, rays, found = rounds + st["rounds"], rays + st["rays"], found + st["found"]
            kms += tr.last_eigenray_ms()["kernel_ms"]
        tr.params = p0
        return np.concatenate(rows), {"rounds": rounds, "rays": rays, "found": found}, {"kernel_ms": kms}

    rb, sb, _ = batched()                              # warm-up, and the equality check
    rl, sl, _ = loop()
    equal = rb.shape == rl.shape and np.array_equal(rb.view(np.uint64), rl.view(np.uint64))
    assert equal, "rows of the many-source call differ from the per-source loop"
    t_b, t_l, ms_b, kms_l = [], [], [], []
    for _ in range(reps):
        t0 = time.perf_counter(); _, _, ms = batched(); t_b.append(time.perf_counter() - t0); ms_b.append(ms)
        t0 = time.perf_counter(); _, _, km = loop(); t_l.append(time.perf_counter() - t0); kms_l.append(km["kernel_ms"])
    res = {"searches": len(sid), "rows": len(rb), "eigenrays": int(sb["found"]), "bitwise_equal": bool(equal),
           "batched_s": stats_of(t_b), "loop_s": stats_of(t_l), "speedup_median": float(np.median(t_l) / np.median(t_b)),
           "batched_rounds": int(sb["rounds"]), "loop_rounds": int(sl["rounds"]), "batched_rays": int(sb["rays"]), "loop_rays": int(sl["rays"]),
           "batched_replay_ms": stats_of([m["replay_ms"] for m in ms_b]), "batched_kernel_ms": stats_of([m["kernel_ms"] for m in ms_b]),
           "batched_call_ms": stats_of([m["call_ms"] for m in ms_b]), "loop_kernel_ms": stats_of(kms_l)}
    return res


def toy_3d(result, reps):
    tr = g.Tracer(abi.GEOAC_3D, 0)
    tr.set_atmosphere_1d(*g.load_met_1d(TOY))
    xy = np.linspace(-200.0, 200.0, 8)
    src = np.array([(x, y, 0.0) for x in xy for y in xy])
    result["a_3d_toy_64_sources_16_receivers"] = compare(tr, src, ring(16, 250.0), dict(bnc_min=0, bnc_max=2), reps)
    print("(a)", json.dumps(result["a_3d_toy_64_sources_16_receivers"]), flush=True)
    tr.close()


def grid_c4(result, reps):
    d, _ = util.load_case("3drngdep_c4")
    tr = g.Tracer(abi.GEOAC_3D_RNGDEP, 0)
    tr.set_atmosphere_3d(*util.load_grid(d))
    xy = np.linspace(-100.0, 100.0, 2)
    src = np.array([(x, y, 0.0) for x in xy for y in xy])
    result["b_3drngdep_grid_c4_4_sources_8_receivers"] = compare(tr, src, ring(8, 220.0), dict(bnc_min=0, bnc_max=1), reps)
    print("(b)", json.dumps(result["b_3drngdep_grid_c4_4_sources_8_receivers"]), flush=True)
    tr.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for eigenray_sources_<parts>.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", default="ab", help="which of the comparisons (a), (b) to run")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    result = {"card": card()}
    if "a" in args.parts:
        toy_3d(result, args.reps)
    if "b" in args.parts:
        grid_c4(result, args.reps)
    with open(os.path.join(args.out, f"eigenray_sources_{args.parts}.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
