"""geoac_trace_ensemble against one geoac_set_atmosphere_1d + geoac_set_params + geoac_trace per member, on the same rays.

  (a) small fans, many atmospheres: 3D, 256 members made from ToyAtmo (16 wind scales 0.5..1.5 x 16 temperature offsets
      -7.5..+7.5 K, no random numbers), each with theta = 1..60 deg step 1 x 30 azimuths (1 800 rays; 460 800 in all).
      Host clock around each side; both end in a device synchronise (the host-buffer calls do).
  (b) the cost of tables in global memory: config 2 (216 000 rays) as a one-member ensemble vs geoac_trace on the same
      profile, by kernel_ms of geoac_last_trace_stats (the trace launches only).
  (c) Global: 64 members made from the config-3 profile (8 wind scales x 8 temperature offsets), 2 000 rays each
      (theta = 1..50 deg step 1 x 40 azimuths) with the config-3 parameters, host clock as in (a).
Each comparison checks that both sides' records are bitwise equal.  Every shape is warmed up once, then the two sides are
alternated 5 times; the JSON gives each side's median and spread (min, max).  The card's name, power limit and max SM
clock are read (nvidia-smi --query-gpu) in the same run.

    python scripts/bench_trace_ensemble.py --out DIR [--reps 5] [--parts abc]
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import geoac_b200 as g                                          # noqa: E402
from geoac_b200 import abi, synth                               # noqa: E402
import bench                                                    # noqa: E402  (workload set-up of configs 2 and 3)
from bench_trace_sources import alternate, card, host_timed    # noqa: E402  (same measurement protocol)

TOY = os.path.join(ROOT, "tests", "golden", "ToyAtmo.met")


def members_from(prof, winds, offsets):
    """One member per (wind scale, temperature offset [K]): the profile's winds scaled, its temperatures shifted."""
    z, T, u, v, rho = prof
    return [(z, T + dT, u * w, v * w, rho) for w in winds for dT in offsets]


def loop_per_member(tr, members, p, th1, ph1):
    """One set_atmosphere_1d + set_params + trace per member; records concatenated member by member (the batched call's layout)."""
    outs = []
    for m in members:
        tr.set_atmosphere_1d(*m)
        tr.params = p
        outs.append(tr.trace(th1, ph1))
    return {"rec": np.concatenate([o["rec"] for o in outs], axis=1), "status": np.concatenate([o["status"] for o in outs]),
            "n_steps": np.concatenate([o["n_steps"] for o in outs])}


def many_members(variant, members, p, th1, ph1, reps):
    ens, loop = g.Tracer(variant, 0), g.Tracer(variant, 0)
    ens.set_ensemble_1d(members)
    ens.params = p
    n1 = len(th1)
    th, ph = np.tile(th1, len(members)), np.tile(ph1, len(members))
    aid = np.repeat(np.arange(len(members), dtype=np.int32), n1)
    res = alternate(reps, {"trace_ensemble_s": lambda: host_timed(lambda: ens.trace_ensemble(aid, th, ph)),
                           "loop_s": lambda: host_timed(lambda: loop_per_member(loop, members, p, th1, ph1))})
    res.update(n_members=len(members), rays_per_member=n1, rays=len(th),
               speedup_median=res["loop_s"]["median"] / res["trace_ensemble_s"]["median"])
    ens.close(); loop.close()
    return res


def small_fans(result, reps):
    prof = g.load_met_1d(TOY)
    members = members_from(prof, np.linspace(0.5, 1.5, 16), np.linspace(-7.5, 7.5, 16))
    tr = g.Tracer(abi.GEOAC_3D, 0)
    tr.set_ensemble_1d(members)                 # the parameters as an ensemble of these members leaves them
    p = tr.params
    tr.close()
    _, _, th1, ph1 = g.prop_angles(1.0, 60.0, 1.0, 0.0, 348.0, 12.0)
    result["a_small_fans_3d_toy_256_members"] = many_members(abi.GEOAC_3D, members, p, th1, ph1, reps)
    print("(a)", json.dumps(result["a_small_fans_3d_toy_256_members"]), flush=True)


def tables_in_global_memory(result, reps):
    tr, _ = bench.setup_tracer("config2", 0)
    _, _, th, ph = g.prop_angles(*bench.WORKLOADS["config2"][1])
    p = tr.params
    tr.set_ensemble_1d([g.load_met_1d(TOY)])    # the profile bench.setup_tracer set; its parameters put back
    tr.params = p
    aid = np.zeros(len(th), np.int32)

    def kernel_ms(f):
        r = f()
        return tr.last_stats()[1], r
    res = alternate(reps, {"trace_ensemble_kernel_ms": lambda: kernel_ms(lambda: tr.trace_ensemble(aid, th, ph)),
                           "trace_kernel_ms": lambda: kernel_ms(lambda: tr.trace(th, ph))})
    res.update(rays=len(th), overhead_median=res["trace_ensemble_kernel_ms"]["median"] / res["trace_kernel_ms"]["median"] - 1.0)
    result["b_config2_one_member"] = res
    print("(b)", json.dumps(res), flush=True)
    tr.close()


def global_members(result, reps):
    tr, _ = bench.setup_tracer("config3", 0)
    p = tr.params                               # config-3 parameters (range limit, source at 30 N)
    tr.close()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "c3.met")
        synth.write_met(path, synth.config3_profile())
        prof = g.load_met_1d(path, global_taper=True)
    members = members_from(prof, np.linspace(0.6, 1.4, 8), np.linspace(-6.0, 6.0, 8))
    _, _, th1, ph1 = g.prop_angles(1.0, 50.0, 1.0, 0.0, 351.0, 9.0)
    result["c_global_config3_64_members"] = many_members(abi.GEOAC_GLOBAL, members, p, th1, ph1, reps)
    print("(c)", json.dumps(result["c_global_config3_64_members"]), flush=True)


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="directory for trace_ensemble_<parts>.json")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--parts", default="abc", help="which of the comparisons (a), (b), (c) to run")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    result = {"card": card()}
    if "a" in args.parts:
        small_fans(result, args.reps)
    if "b" in args.parts:
        tables_in_global_memory(result, args.reps)
    if "c" in args.parts:
        global_members(result, args.reps)
    with open(os.path.join(args.out, f"trace_ensemble_{args.parts}.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
