#!/usr/bin/env python
"""bench.py -- throughput of the batched ray-tracing hot path.  Default workload: BASELINE.json's config 2
(GeoAc3D, ToyAtmo.met, theta 1-60 deg step 1 x azimuth 0-359.9 deg step 0.1 = 216 000 rays, 2 bounces, CalcAmp on,
WriteRays=False); one pass over the whole launch-angle grid = one "step".

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

Workloads: config1 ... config5 are BASELINE.json's five configurations (SURVEY.md section 8d); config4s / config5s are the
same range-dependent runs on a coarser node grid with fewer rays (quick checks); smallgrid / midgrid are reduced config-2
launch grids.  N > 1 is launched by torchrun, one rank per GPU, no data-path collective (rays are independent, SURVEY 8e):
  * config 5 (the "1e6 rays sharded across 1/2/4/8 B200" configuration) splits its ray list across ranks in interleaved
    4096-ray blocks -> "scaling": "strong";
  * every other workload replicates the launch grid per rank with a rank-specific azimuth rotation -> "scaling": "weak".
Rank 0 prints ONE JSON line.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOY = os.path.join(ROOT, "tests", "golden", "ToyAtmo.met")
PI = 3.141592653589793238462643

V2D, V3D, VGLOBAL, V3DRD, VGLOBALRD = 0, 1, 2, 3, 4
KERNEL_NAMES = {V2D: "geoac::trace_kernel<Eq2D<true>,512,true>", V3D: "geoac::trace_kernel<Eq3D<true>,384,true>",
                VGLOBAL: "geoac::trace_kernel<EqGlobal<true>,384,true>", V3DRD: "geoac::trace_kernel<Eq3DRD<true>,128,false>",
                VGLOBALRD: "geoac::trace_kernel<EqGlobalRD<true>,128,false>"}
# ALGORITHMIC FP64 operations per RK4 step of each variant (CalcAmp on, incl. the travel-time + absorption bookkeeping of
# the step; add/sub/mul/div/sqrt/transcendental = 1, fma = 2, compares 0 -- SURVEY 8d).
#  * ALGO_FLOPS_PER_STEP: counted on THIS repo's de-duplicated formulation by running the per-ray code with an op-counting
#    scalar (tests/flopcount/run_flopcount.py -> tests/flopcount/flops.jsonl), as SURVEY 8d (i) asks.  `roofline.achieved`
#    uses these: they are the operations the kernel's algorithm needs, each libm call counted once.
#  * SURVEY_FLOPS_PER_STEP: SURVEY 8d's provisional hand de-duplication of the REFERENCE's formulation (+-25 %); reported
#    next to it as `achieved_survey_figure`.  The range-dependent figures differ most: the tensor-product sampler needs
#    17-19 k operations where the reference's five-bicubic-patch scheme, de-duplicated, needs ~39 k.
ALGO_FLOPS_PER_STEP = {V2D: 739.6, V3D: 1220.2, VGLOBAL: 2126.3, V3DRD: 16922.0, VGLOBALRD: 18202.6}
# the same count on the round-1 formulation (before the common factor of the right-hand sides moved into the step factors, the
# nu^2 interpolant and the step-size shortcut removed ~6 % of the operations): reported next to it so that rounds stay comparable
ALGO_FLOPS_PER_STEP_R1 = {V2D: 766.0, V3D: 1295.0, VGLOBAL: 2225.2, V3DRD: 16988.7, VGLOBALRD: 18613.4}
NCU_DRAM_BYTES_PER_RAY = {"config2": 502.0}       # measured with ncu --set full, see roofline.traffic_source
SURVEY_FLOPS_PER_STEP = {V2D: 1400.0, V3D: 2200.0, VGLOBAL: 2800.0, V3DRD: 39000.0, VGLOBALRD: 40000.0}

#               variant    theta_min, theta_max, theta_step, phi_min, phi_max, phi_step   bounces  atmosphere
WORKLOADS = {
    "config1":   (V2D,       (0.5, 45.0, 0.5, -90.0, -90.0, 1.0),       2, "toy"),
    "config2":   (V3D,       (1.0, 60.5, 1.0, 0.0, 359.95, 0.1),        2, "toy"),
    "smallgrid": (V3D,       (1.0, 60.5, 1.0, 0.0, 359.5, 5.0),         2, "toy"),
    "midgrid":   (V3D,       (1.0, 60.5, 1.0, 0.0, 359.75, 0.5),        2, "toy"),
    "config3":   (VGLOBAL,   (0.5, 50.45, 0.1, 0.0, 359.8, 0.36),       5, "c3"),
    "config4":   (V3DRD,     (1.0, 50.975, 0.05, 0.0, 358.0, 3.6),      2, "c4"),
    "config4s":  (V3DRD,     (1.0, 50.75, 0.5, 0.0, 358.0, 3.6),        2, "c4s"),
    "config5":   (VGLOBALRD, (1.0, 50.975, 0.05, 0.0, 359.8, 0.36),     2, "c5"),
    "config5s":  (VGLOBALRD, (1.0, 50.75, 0.5, 0.0, 358.0, 3.6),        2, "c5s"),
}
DESCRIPTIONS = {
    "config1": "BASELINE config 1: GeoAc2D, ToyAtmo.met, theta 0.5..45 step 0.5, azimuth -90 (90 rays), bounces=2",
    "config2": "BASELINE config 2: GeoAc3D stratified, ToyAtmo.met, theta 1..60 step 1 x azimuth 0..359.9 step 0.1 (216000 rays), bounces=2, CalcAmp on, WriteRays=False",
    "smallgrid": "reduced grid for debugging: GeoAc3D, theta 1..60 x azimuth 0..355 step 5 (4320 rays)",
    "midgrid": "reduced grid for ncu captures: GeoAc3D, theta 1..60 x azimuth 0..359.5 step 0.5 (43200 rays)",
    "config3": "BASELINE config 3: GeoAcGlobal, synthetic stratified profile to 150 km (SURVEY 8d), source lat 30 lon 0, theta 0.5..50.4 step 0.1 x azimuth 0..359.64 step 0.36 (500000 rays), bounces=5, rng_max=3000",
    "config4": "BASELINE config 4: GeoAc3D.RngDep, synthetic 200x200x300 node grid (SURVEY 8d), theta 1..50.95 step 0.05 x azimuth 0..356.4 step 3.6 (100000 rays), bounces=2, CalcAmp on",
    "config4s": "config 4 on a 50x50x300 node grid with 10000 rays (quick check)",
    "config5": "BASELINE config 5: GeoAcGlobal.RngDep, synthetic 181x361x300 global grid (SURVEY 8d), source lat 35 lon 0, theta 1..50.95 step 0.05 x azimuth 0..359.64 step 0.36 (1000000 rays), bounces=2",
    "config5s": "config 5 on a 46x91x300 node grid with 10000 rays (quick check)",
}
SHARDED = {"config5"}            # strong scaling: one ray list split across ranks (geoac_b200/sharding.py)


def workload_angles(name, rank=0):
    from geoac_b200 import api
    variant, grid, _, _ = WORKLOADS[name]
    th_deg, ph_deg, _, _ = api.prop_angles(*grid)
    if name not in SHARDED and variant != V2D:
        ph_deg = ph_deg + 0.05 * rank / 8.0                          # weak scaling: same grid, rank-specific rotation
    return grid, th_deg, ph_deg, th_deg * PI / 180.0, PI / 2.0 - ph_deg * PI / 180.0


def shard_indices(n, rank, world):
    from geoac_b200 import sharding
    return sharding.shard_indices(n, rank, world, int(os.environ.get("GEOAC_BENCH_SHARD_BLOCK", sharding.SHARD_BLOCK)))


def setup_tracer(name, device):
    """Create the context of a workload on `device` with its atmosphere and parameters; returns (tracer, params)."""
    import geoac_b200 as g
    from geoac_b200 import synth
    variant, _, bounces, atmo = WORKLOADS[name]
    tr = g.Tracer(variant, device)
    if atmo == "toy":
        tr.set_atmosphere_1d(*g.load_met_1d(TOY))
    elif atmo == "c3":
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "c3.met")
            synth.write_met(path, synth.config3_profile())
            tr.set_atmosphere_1d(*g.load_met_1d(path, global_taper=True))
    elif atmo in ("c4", "c4s"):
        tr.set_atmosphere_3d(*(synth.config4_grid() if atmo == "c4" else synth.config4_grid(50, 50, 300)))
    elif atmo in ("c5", "c5s"):
        tr.set_atmosphere_3d(*(synth.config5_grid() if atmo == "c5" else synth.config5_grid(46, 91, 300)))
    p = tr.params
    p.bounces, p.calc_amp, p.accum_per_segment = bounces, 1, (1 if variant == V2D else 0)
    if name == "config3":
        p.range_limit = 3000.0
        p.src[0], p.src[1], p.src[2] = 0.0, 30.0 * PI / 180.0, 0.0
    if variant == VGLOBALRD:
        p.src[0], p.src[1], p.src[2] = 0.0, 35.0 * PI / 180.0, 0.0
    tr.params = p
    return tr, p


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason sampling DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if not self.nv:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ CPU reference arm
def _theta_count(th_deg):
    """Number of inclinations of the launch grid, taken from the ENUMERATED angles (theta is the fast axis of the mains'
    loops); never recomputed from (max - min) / step, which is off by one for loop maxima placed half a step past the end."""
    th_deg = np.asarray(th_deg)
    change = np.nonzero(th_deg[1:] < th_deg[:-1])[0]
    return int(change[0]) + 1 if len(change) else len(th_deg)


def _sample_stride(total, want_rays, n_theta):
    """Stride of a subsample `index = offset + k * stride` that is STRATIFIED in inclination: consecutive sample points step
    through the theta axis by about 0.382 n_theta (golden-section spacing, coprime with n_theta), so any run of consecutive
    points -- the whole sample as well as one process's share of it -- covers the inclinations evenly.  Ray lifetimes depend
    on theta (14x between theta = 1 and 60 deg), so an unstratified sample misestimates rays/s by that much."""
    stride = max(1, total // max(1, want_rays))
    if n_theta <= 1 or total <= want_rays:
        return stride
    want_mod = max(1, int(round(0.381966 * n_theta)))
    while math.gcd(want_mod, n_theta) != 1:
        want_mod += 1
    stride += (want_mod - stride) % n_theta
    return stride


def _sample_sets(total, want_rays, n_proc, n_theta):
    """Disjoint index sets, one per process: process i takes the sample points k = i, i + n_proc, i + 2 n_proc, ..."""
    stride = _sample_stride(total, want_rays, n_theta)
    pts = np.arange(0, total, stride, dtype=np.int64)[: max(n_proc, want_rays)]
    return stride, [pts[i::n_proc] for i in range(n_proc)]


def cpu_reference_run(workload, target_rays, n_proc, as_shipped=False):
    """Time the reference's own CPU implementation on a theta-stratified subsample of the workload, split over n_proc
    processes with disjoint ray sets.  Stratified workloads run oracle/_ref/ref_<variant> (the unmodified reference sources +
    a driver main; kind "reference", built -O2; `as_shipped` runs the -O0 build the reference's makefile produces, kind
    "reference-as-shipped"); when it is not built, and for the range-dependent workloads (whose reference input is
    40 000+ node files), the C restatement in oracle/ is timed instead (kind "port").
    Returns dict(rays, steps, seconds, rate, kind, cores, sample)."""
    from geoac_b200 import abi, synth
    variant, grid, bounces, atmo = WORKLOADS[workload]
    _, th_deg, _, _, _ = workload_angles(workload)
    total = len(th_deg)
    n_theta = _theta_count(th_deg)
    stride, sets = _sample_sets(total, target_rays, n_proc, n_theta)
    ref_bin = os.path.join(ROOT, "oracle", "_ref", "ref_" + abi.VARIANT_NAMES[variant] + ("_O0" if as_shipped else ""))
    keys = dict(theta_min=grid[0], theta_max=grid[1], theta_step=grid[2], bounces=bounces)
    if variant != V2D:
        keys.update(phi_min=grid[3], phi_max=grid[4], phi_step=grid[5], accum_mode=0)
    if workload == "config3":
        keys.update(lat_src=30, lon_src=0, rng_max=3000)
    if os.path.exists(ref_bin) and atmo in ("toy", "c3"):
        kind = "reference-as-shipped" if as_shipped else "reference"
        with tempfile.TemporaryDirectory() as td:
            prof = TOY
            if atmo == "c3":
                prof = os.path.join(td, "c3.met")
                synth.write_met(prof, synth.config3_profile())
            procs = []
            for i in range(n_proc):
                # the driver takes rays with index % stride_i == offset_i: process i's points are offset i*stride, spaced n_proc*stride
                cmd = [ref_bin, os.path.join(td, f"o{i}.bin"), prof] + [f"{k}={v}" for k, v in keys.items()] \
                    + [f"stride={stride * n_proc}", f"offset={(i * stride) % (stride * n_proc)}"]
                procs.append(subprocess.Popen(cmd, stdout=subprocess.PIPE, text=True))
            outs = [p.communicate()[0] for p in procs]
        infos = [json.loads(o.strip().splitlines()[-1]) for o in outs]
        per = [(i["rays"], i["steps"], i["t_trace_s"]) for i in infos]          # excluding profile load
    else:
        if as_shipped:
            return None
        kind = "port"
        from multiprocessing import Pool
        with Pool(n_proc) as pool:
            per = pool.starmap(_port_worker, [(workload, s) for s in sets])       # excluding atmosphere set-up
    rays = sum(r[0] for r in per)
    steps = sum(r[1] for r in per)
    secs = max(r[2] for r in per)
    # steady-state throughput of n_proc busy cores: sum of the per-process rates (dividing by the slowest process instead
    # would charge the sample's residual imbalance -- a few dozen rays per process -- to the reference)
    rate = sum(r[0] / r[2] for r in per if r[2] > 0)
    step_rate = sum(r[1] / r[2] for r in per if r[2] > 0)
    return {"rays": rays, "steps": steps, "seconds": secs, "rate": rate, "step_rate": step_rate, "kind": kind, "cores": n_proc,
            "steps_per_ray": steps / max(1, rays),
            "sample": f"every {stride}th ray of {workload}, theta-stratified ({rays} of {total} rays, {steps} RK4 steps, "
                      f"{steps / max(1, rays):.0f} steps/ray), {n_proc} process(es), sum of per-process rates"}


def _port_worker(workload, idx):
    from geoac_b200 import synth
    from oracle import pyoracle as po
    variant, _, bounces, atmo = WORKLOADS[workload]
    _, _, _, th, ph = workload_angles(workload)
    if atmo == "toy":
        at = po.atmo1d(False, *po.load_met_1d(TOY))
    elif atmo == "c3":
        with tempfile.TemporaryDirectory() as td:
            path = os.path.join(td, "c3.met")
            synth.write_met(path, synth.config3_profile())
            at = po.atmo1d(True, *po.load_met_1d(path, global_taper=True))
    elif atmo in ("c4", "c4s"):
        at = po.atmo3d(False, *(synth.config4_grid() if atmo == "c4" else synth.config4_grid(50, 50, 300)))
    else:
        at = po.atmo3d(True, *(synth.config5_grid() if atmo == "c5" else synth.config5_grid(46, 91, 300)))
    p = po.default_params(variant, at)
    p.bounces, p.calc_amp, p.accum_per_segment = bounces, 1, (1 if variant == V2D else 0)
    if workload == "config3":
        p.range_limit = 3000.0
        p.src[0], p.src[1], p.src[2] = 0.0, 30.0 * PI / 180.0, 0.0
    if variant == VGLOBALRD:
        p.src[0], p.src[1], p.src[2] = 0.0, 35.0 * PI / 180.0, 0.0
    t0 = time.perf_counter()
    out = po.trace(variant, at, p, th[idx], ph[idx])
    return len(idx), out["total_steps"], time.perf_counter() - t0


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0))
    if WORKLOADS[args.workload][3] in ("c4", "c5"):
        cores = min(cores, 8)                                    # every process holds its own copy of the node tables
    per_step = []
    res = None
    rays_per_core = 24 if WORKLOADS[args.workload][0] in (V2D, V3D, VGLOBAL) else 1
    for i in range(args.warmup + args.steps):
        res = cpu_reference_run(args.workload, target_rays=cores * rays_per_core, n_proc=cores)
        if i >= args.warmup:
            per_step.append(res)
    secs = sum(r["seconds"] for r in per_step)
    val = float(np.mean([r["rate"] for r in per_step]))
    step_rate = float(np.mean([r["step_rate"] for r in per_step]))
    line = {"impl": "reference", "metric": "rays/sec", "value": val, "unit": "rays/s", "rk4_steps_per_sec": step_rate,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.workload in SHARDED else "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic launch-angle grid; " + ("ToyAtmo.met profile" if WORKLOADS[args.workload][3] == "toy" else "synthetic G2S atmosphere (SURVEY 8d)"),
            "config": {"workload": DESCRIPTIONS[args.workload], "sample": res["sample"]},
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": res["cores"], "kind": res["kind"], "sample": res["sample"],
                             "rk4_steps_per_sec": step_rate, "steps_per_ray": res["steps_per_ray"]},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from geoac_b200 import abi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        cpu_group = dist.new_group(backend="gloo")                    # host-side barrier: an NCCL barrier spins ON the waiting ranks' GPUs
    dev = torch.device("cuda", local)

    variant = WORKLOADS[args.workload][0]
    _, th_deg, ph_deg, th, ph = workload_angles(args.workload, rank)
    sharded = args.workload in SHARDED
    if sharded and world > 1:
        mine = shard_indices(len(th), rank, world)
        th, ph = np.ascontiguousarray(th[mine]), np.ascontiguousarray(ph[mine])
    elif sharded and args.shard_of:                                      # development aid: rank R's share of a W-way split on ONE GPU
        r_, w_ = (int(x) for x in args.shard_of.split("/"))
        mine = shard_indices(len(th), r_, w_)
        th, ph = np.ascontiguousarray(th[mine]), np.ascontiguousarray(ph[mine])
    if args.rays_cap > 0:
        th, ph = np.ascontiguousarray(th[: args.rays_cap]), np.ascontiguousarray(ph[: args.rays_cap])
    n = len(th)
    tr, p = setup_tracer(args.workload, local)
    if args.bounces >= 0:
        p.bounces = args.bounces
        tr.params = p
    if args.ray_limit > 0:
        p.ray_limit = args.ray_limit
        tr.params = p
    n_rec = p.bounces + 1
    n_slots = n * n_rec

    # ---- device-resident leg: inputs already in HBM, outputs stay in HBM ----
    d_th = torch.from_numpy(th).to(dev)
    d_ph = torch.from_numpy(ph).to(dev)
    d_rec = torch.empty((abi.NFIELDS, n_slots), dtype=torch.float64, device=dev)
    d_status = torch.empty(n_slots, dtype=torch.int32, device=dev)
    d_nsteps = torch.empty(n_slots, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)        # > 126 MB L2
    stream = torch.cuda.current_stream(dev)

    def one_pass():
        flush.zero_()                                                    # L2 flush between iterations
        tr.trace_device(n, d_th.data_ptr(), d_ph.data_ptr(), d_rec.data_ptr(), d_status.data_ptr(), d_nsteps.data_ptr(), stream.cuda_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        one_pass()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        ev[i][0].record(stream)
        flush.zero_()
        kev[i][0].record(stream)
        tr.trace_device(n, d_th.data_ptr(), d_ph.data_ptr(), d_rec.data_ptr(), d_status.data_ptr(), d_nsteps.data_ptr(), stream.cuda_stream)
        kev[i][1].record(stream)
        ev[i][1].record(stream)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, n, n_rec, d_rec, d_status, d_nsteps)
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    kern_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps        # scheduling pass + trace kernel (+4 memsets) per pass
    total_steps, _ = tr.last_stats()                                    # RK4 steps of one pass on this rank
    lane_occ = tr.last_lane_occupancy()
    launches_per_pass = tr.last_kernel_launches()
    arrivals = int((d_status == abi.ST_ARRIVAL).sum().item())

    t = torch.tensor([dev_ms, float(total_steps), float(n), float(arrivals)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        dev_ms_max, steps_all, rays_all, arrivals_all = tmax[0].item(), tsum[1].item(), tsum[2].item(), tsum[3].item()
    else:
        dev_ms_max, steps_all, rays_all, arrivals_all = dev_ms, float(total_steps), float(n), float(arrivals)
    secs = dev_ms_max * 1e-3
    rays_per_s = rays_all * args.steps / secs
    steps_per_s = steps_all * args.steps / secs

    # ---- end-to-end leg: HOST (pinned) buffers through the public C-ABI call, H2D + D2H inside the timed region ----
    h_th = torch.from_numpy(th).pin_memory(); h_ph = torch.from_numpy(ph).pin_memory()
    h_rec = torch.empty((abi.NFIELDS, n, n_rec), dtype=torch.float64).pin_memory()
    h_status = torch.empty((n, n_rec), dtype=torch.int32).pin_memory()
    h_nsteps = torch.empty((n, n_rec), dtype=torch.int32).pin_memory()
    out = {"rec": h_rec.numpy(), "status": h_status.numpy(), "n_steps": h_nsteps.numpy()}
    long_run = args.workload in ("config3", "config4", "config5") and not args.e2e_full
    e2e_k = 1 if long_run else max(1, min(args.steps, 3))
    if args.no_e2e:
        e2e_k = 0
    else:
        tr.reserve(n)                                                   # device staging allocated outside the timed region
        if not long_run:
            tr.trace(h_th.numpy(), h_ph.numpy(), out)                   # warm-up pass
    barrier()
    e0 = time.perf_counter()
    for _ in range(e2e_k):
        tr.trace(h_th.numpy(), h_ph.numpy(), out)                       # synchronous: returns with results on the host
    barrier()
    e2e_s = max(time.perf_counter() - e0, 1e-9)
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_rays = rays_all * e2e_k / te.item()
    h2d = 2 * n * 8
    d2h = abi.NFIELDS * n_slots * 8 + 2 * n_slots * 4 + 16

    multi = None
    if world > 1 and args.workload in ("config1", "config2") and not args.rays_cap:
        barrier()
        if rank == 0:                                                    # the other ranks wait on the HOST (gloo): their GPUs stay idle for rank 0
            try:
                multi = single_process_multi_record(args, world)
            except Exception as e:                                       # reported, never fatal for the bench line
                multi = {"error": str(e)}
        dist.barrier(group=cpu_group)
        barrier()
    strong = None
    if not args.no_strong and args.workload == "config2" and not args.rays_cap:
        tr_keep = tr
        strong = strong_scaling_record(world, rank, local, dev, barrier)
        tr = tr_keep
    if rank == 0:
        peak_tf, peak_ms = tr.measure_fp64_peak()
        flops_step = ALGO_FLOPS_PER_STEP[variant]
        achieved_tf = flops_step * total_steps / (kern_ms * 1e-3) / 1e12
        atmo = WORKLOADS[args.workload][3]
        line = {
            "metric": "rays/sec", "value": rays_per_s, "unit": "rays/s", "rk4_steps_per_sec": steps_per_s,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
            "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic launch-angle grid; " + ("ToyAtmo.met profile (the reference's shipped fixture)" if atmo == "toy"
                                                        else "synthetic G2S atmosphere generated as SURVEY 8d specifies"),
            "config": {"workload": DESCRIPTIONS[args.workload], "rays_per_gpu": n, "rk4_steps_per_pass_per_gpu": total_steps,
                       "arrival_records_per_pass": int(arrivals_all), "lane_occupancy": round(lane_occ, 4),
                       "l2": "256 MiB buffer written between iterations (L2 flush)",
                       "multi_gpu": "one ray list split across ranks in interleaved 4096-ray blocks" if sharded else "replicated grid per rank, azimuth offset by rank"},
            "e2e": {"value": e2e_rays, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "passes": e2e_k},
            "gpu_launches": args.steps * launches_per_pass,
            "clocks": sampler.summary(),
            "roofline": {"bound": "fp64", "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf if peak_tf > 0 else None,
                         "traffic": (NCU_DRAM_BYTES_PER_RAY[args.workload] * n if args.workload in NCU_DRAM_BYTES_PER_RAY else None),
                         "traffic_source": ("bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture "
                                            "(profiles/r1_ncu_full_trace_kernel_Eq3D_final2.txt, 86 400-ray slice: 43.4 MB = 502 B per ray), scaled "
                                            "to this launch's rays; algorithmic: 16 B of angles in + 216 B per arrival record out"
                                            if args.workload in NCU_DRAM_BYTES_PER_RAY else None),
                         "kernel": KERNEL_NAMES[variant], "kernel_ms_per_launch": kern_ms,
                         "algorithmic_flops_per_rk4_step": flops_step,
                         "frac_with_round1_flop_count": (ALGO_FLOPS_PER_STEP_R1[variant] * total_steps / (kern_ms * 1e-3) / 1e12 / peak_tf) if peak_tf > 0 else None,
                         "round1_flops_per_rk4_step": ALGO_FLOPS_PER_STEP_R1[variant],
                         "achieved_survey_figure": SURVEY_FLOPS_PER_STEP[variant] * total_steps / (kern_ms * 1e-3) / 1e12,
                         "survey_flops_per_rk4_step": SURVEY_FLOPS_PER_STEP[variant],
                         "peak_source": "DFMA micro-benchmark run in this process (MEASURED_PEAKS.json has no FP64 entry); "
                                        "HBM is not the bound: ~0.03 B/step of record traffic"},
            "wall_s_timed_region": t_wall,
        }
        if multi is not None:
            line["single_process_multi"] = multi
        if strong is not None:
            strong["roofline_frac"] = strong["roofline_frac"] / peak_tf if peak_tf > 0 else None
            line["strong"] = strong
        if variant in (V3DRD, VGLOBALRD):
            line["config"]["schedule"] = tr.last_schedule()
        if world == 1 and not args.no_cpu_baseline:
            rngdep = variant in (V3DRD, VGLOBALRD)
            cb = cpu_reference_run(args.workload, target_rays=(8 if rngdep else 120), n_proc=1)
            grid_spr = total_steps / max(1, n)
            line["cpu_baseline"] = {"value": cb["rate"], "unit": "rays/s", "cores": 1, "kind": cb["kind"],
                                    "sample": cb["sample"], "rk4_steps_per_sec": cb["step_rate"],
                                    "steps_per_ray": cb["steps_per_ray"], "workload_steps_per_ray": grid_spr,
                                    # the sample's rays/s rescaled to the workload's mean ray length (they agree within a few per cent
                                    # when the sample is representative; the stratified sample makes it so)
                                    "value_at_workload_steps_per_ray": cb["step_rate"] / grid_spr if grid_spr > 0 else None}
            if not rngdep:
                sh = cpu_reference_run(args.workload, target_rays=60, n_proc=1, as_shipped=True)
                if sh is not None:
                    line["cpu_baseline_as_shipped"] = {"value": sh["rate"], "unit": "rays/s", "cores": 1, "kind": sh["kind"],
                                                       "sample": sh["sample"] + "; g++ -O0 as the reference's makefile builds it",
                                                       "rk4_steps_per_sec": sh["step_rate"], "steps_per_ray": sh["steps_per_ray"]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, n, n_rec, d_rec, d_status, d_nsteps):
    """Write the records of the last timed pass as float64 .npy files under out_dir, shaped as Tracer.trace returns them:
    rec [NFIELDS][rays][n_rec], status and n_steps [rays][n_rec], plus ray_index [rays] (the rays' positions in the traced
    batch).  When all rays would exceed DUMP_BYTES, a fixed seeded sample of rays is written, every bounce of each, so that
    runs of two builds with the same arguments can be compared file for file."""
    import torch
    nf = d_rec.shape[0]
    per_ray = 8 * ((nf + 2) * n_rec + 1)
    k = min(n, (DUMP_BYTES - 4 * 4096) // per_ray)                       # 4096 bytes per file left for the .npy header
    idx = np.arange(n) if k == n else np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    sel = torch.from_numpy(idx).to(d_rec.device)
    arrays = {"rec": d_rec.view(nf, n, n_rec).index_select(1, sel),
              "status": d_status.view(n, n_rec).index_select(0, sel),
              "n_steps": d_nsteps.view(n, n_rec).index_select(0, sel)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.to(torch.float64).cpu().numpy())
    np.save(os.path.join(out_dir, "ray_index.npy"), idx.astype(np.float64))


def single_process_multi_record(args, world):
    """Rank 0 only, the other ranks idle at a barrier: ONE process drives all `world` devices through the product's own multi-device
    entry point (geoac_create_multi + geoac_trace_multi: host threads, interleaved 4096-ray blocks, pinned staging, merge by ray
    index) -- the path a C++ front end uses -- on the concatenation of every rank's batch, host buffers in and out."""
    from geoac_b200 import api, abi
    variant, _, bounces, atmo = WORKLOADS[args.workload]
    ths, phs = [], []
    for r in range(world):
        _, _, _, th, ph = workload_angles(args.workload, r)
        ths.append(th); phs.append(ph)
    th, ph = np.concatenate(ths), np.concatenate(phs)
    mt = api.MultiTracer(variant, list(range(world)))
    try:
        if atmo == "toy":
            mt.set_atmosphere_1d(*api.load_met_1d(TOY))
        else:
            return None
        p = mt.params
        p.bounces, p.calc_amp, p.accum_per_segment = bounces, 1, (1 if variant == V2D else 0)
        mt.params = p
        out = mt.trace(th, ph)                                           # warm-up: staging allocated, kernels loaded
        t0 = time.perf_counter()
        k = 2
        for _ in range(k):
            mt.trace(th, ph, out)
        secs = (time.perf_counter() - t0) / k
        return {"devices": world, "rays": int(len(th)), "rays_per_sec": len(th) / secs, "ms_per_pass": 1e3 * secs,
                "arrival_records": int((out["status"] == abi.ST_ARRIVAL).sum()),
                "api": "geoac_create_multi + geoac_multi_set_* + geoac_trace_multi (one process, one host thread per device, host buffers)"}
    finally:
        mt.close()


def strong_scaling_record(world, rank, local, dev, barrier):
    """Config 5 (the "1e6 rays sharded across 1/2/4/8 B200" configuration of BASELINE.json) in FULL, one timed pass, the ray list
    split across the ranks in interleaved 4096-ray blocks (geoac_b200/sharding.py) -- carried in every bench line so that the
    strong-scaling curve N = 1, 2, 4, 8 is in the driver's own record.  Device-resident angles, CUDA events, max over ranks."""
    import torch
    import torch.distributed as dist
    from geoac_b200 import abi
    _, _, _, th, ph = workload_angles("config5")
    n_total = len(th)
    if world > 1:
        mine = shard_indices(n_total, rank, world)
        th, ph = np.ascontiguousarray(th[mine]), np.ascontiguousarray(ph[mine])
    n = len(th)
    t0 = time.perf_counter()
    tr, p = setup_tracer("config5", local)
    setup_s = time.perf_counter() - t0
    n_slots = n * (p.bounces + 1)
    d_th, d_ph = torch.from_numpy(th).to(dev), torch.from_numpy(ph).to(dev)
    d_rec = torch.empty((abi.NFIELDS, n_slots), dtype=torch.float64, device=dev)
    d_status = torch.empty(n_slots, dtype=torch.int32, device=dev)
    d_nsteps = torch.empty(n_slots, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream(dev)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    tr.trace_device(n, d_th.data_ptr(), d_ph.data_ptr(), d_rec.data_ptr(), d_status.data_ptr(), d_nsteps.data_ptr(), stream.cuda_stream)
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    steps, _ = tr.last_stats()
    occ = tr.last_lane_occupancy()
    sched = tr.last_schedule()
    arrivals = int((d_status == abi.ST_ARRIVAL).sum().item())
    checksum = int(d_nsteps.to(torch.int64).sum().item())
    t = torch.tensor([ms, float(steps), float(n), float(arrivals), float(checksum), occ], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tmin = t.clone(); dist.all_reduce(tmin, op=dist.ReduceOp.MIN)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    else:
        tmax = tmin = tsum = t
    tr.close()
    per_rank = [ms]
    if world > 1:
        gathered = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([ms], dtype=torch.float64, device=dev))
        per_rank = [g.item() for g in gathered]
    secs = tmax[0].item() * 1e-3
    return {"workload": DESCRIPTIONS["config5"], "scaling": "strong", "n_gpus": world, "passes": 1, "ms": tmax[0].item(), "ms_fastest_rank": tmin[0].item(),
            "ms_per_rank": [round(x, 1) for x in per_rank],
            "rays": int(tsum[2].item()), "rays_per_sec": tsum[2].item() / secs, "rk4_steps": int(tsum[1].item()), "rk4_steps_per_sec": tsum[1].item() / secs,
            "arrival_records": int(tsum[3].item()), "n_steps_checksum": int(tsum[4].item()),
            "lane_occupancy_min_rank": tmin[5].item(), "setup_s_rank0": setup_s,
            "schedule_rank0": sched,
            "roofline_frac": ALGO_FLOPS_PER_STEP[VGLOBALRD] * tsum[1].item() / secs / 1e12 / max(1, world),   # divided by the measured peak below
            "note": "whole-job time = slowest rank; one ray list split across ranks, atmosphere replicated, no collective on the data path"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="config2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-full", action="store_true", help="warm the end-to-end leg up even on the long workloads")
    ap.add_argument("--rays-cap", type=int, default=0, help="profiling aid: keep only the first N rays of the workload")
    ap.add_argument("--bounces", type=int, default=-1, help="profiling aid: override the workload's bounce count")
    ap.add_argument("--shard-of", default="", help="development aid: 'R/W' traces rank R's share of a W-way split of a sharded workload on one GPU")
    ap.add_argument("--no-e2e", action="store_true", help="development aid: skip the end-to-end leg")
    ap.add_argument("--no-strong", action="store_true", help="skip the config-5 strong-scaling sub-record")
    ap.add_argument("--ray-limit", type=float, default=0.0, help="profiling aid: override ray_limit (RK4 step limit per segment = 100 x ray_limit)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write rank 0's records of the last timed pass to DIR/*.npy (float64, at most 64 MB: a seeded sample of rays beyond that)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's records (--impl ours)")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
