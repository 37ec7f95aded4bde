"""Scheduling of the range-dependent sets is result neutral, bit for bit: Eq3DRD on the config-4 grid fixture and EqGlobalRD
on the config-5 one.  The reference is the natural claim order (knob lpt = 0: one launch, no long region).  Every scheduling
configuration -- long region, exclusive long-region launch, quarter claims, cost dilation, cost scout step -- must give the
same records, and each test asserts from geoac_last_schedule / the kernel count that the mechanism it exercises ran.  Also:
the cooperative four-lanes-per-ray mode against the serial path, and the capture kernels under a claim order."""
import numpy as np
import pytest
import torch

from geoac_b200 import abi
from tests import util
from tests.test_gpu_device_path import assert_bitwise, make_tracer, seeded_angles

pytestmark = pytest.mark.gpu

SETS = ["3drngdep_c4", "globalrngdep_c5"]
WARPS_PER_CTA = 4          # the range-dependent trace kernels run 128-lane CTAs (capi.cu: dispatch_trace)
BOUNCES = 1                # one reflection per ray: reflections are exercised at two thirds of the GPU time of the fixtures' two


def mixed_angles(n, n_long, seed=7):
    """n_long seeded rays at trace-length inclinations, then steep ones that leave through the top of the grid within a few
    hundred steps.  The first packets are long, the rest cost far less than the average work of a lane: a long region and
    a non-empty main region next to it, at a small cost in GPU time."""
    th1, ph1 = seeded_angles(n_long, seed)
    rng = np.random.default_rng(seed + 1)
    th2, ph2 = util.angles_rad(rng.uniform(84.0, 89.0, n - n_long), rng.uniform(-180.0, 180.0, n - n_long))
    return np.concatenate([th1, th2]), np.concatenate([ph1, ph2])


def run(case, th, ph, **knobs):
    tr = make_tracer(case, knobs=knobs, bounces=BOUNCES)
    out = tr.trace(th, ph)
    return out, tr.last_schedule(), tr


def check_slots(out):
    assert (out["status"][:, 0] != abi.ST_NONE).all(), "a ray produced no first-segment outcome"


def lane_count(case):
    """Lanes of the full trace launch on this GPU: the claim order is automatic (lpt = 1) exactly when a batch has more rays
    than that.  Found with steep, short rays; the lane count is a whole number of CTAs per SM."""
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    for per_sm in range(1, 17):
        lanes = sm * per_sm * 32 * WARPS_PER_CTA
        th, ph = util.angles_rad(np.full(lanes + 1, 88.0), np.linspace(-180.0, 180.0, lanes + 1))
        _, s, tr = run(case, th, ph, lpt=1)
        if tr.last_kernel_launches() > 1:
            return lanes
    raise AssertionError("the automatic claim order never engaged")


@pytest.mark.parametrize("case", SETS)
def test_ragged_batches_are_schedule_neutral(case):
    """Partial last packets (claim-order entries 0xffffffff), 8 / 9 rays around the switch into the cooperative mode, and a
    batch one ray above the lane count, where the automatic claim order engages with a main region beside the long one."""
    th, ph = seeded_angles(65, 11)
    for n in (1, 7, 8, 9, 31, 33, 65):
        want, _, _ = run(case, th[:n], ph[:n], lpt=0)
        got, s, _ = run(case, th[:n], ph[:n], lpt=2)
        assert_bitwise(got, want, f"{case} n={n}")
        check_slots(want)
        assert s["long_packets"] > 0 and s["long_ctas"] > 0, (n, s)
    n = lane_count(case) + 1
    th, ph = mixed_angles(n, max(320, n // 32))          # the long rays hold the average lane work well above a steep packet's
    want, s0, t0 = run(case, th, ph, lpt=0)
    assert t0.last_kernel_launches() == 1 and s0["long_packets"] == 0
    got, s, tr = run(case, th, ph)                                          # lpt = 1, as the benchmark runs
    assert_bitwise(got, want, f"{case} n={n}")
    check_slots(want)
    assert tr.last_kernel_launches() > 1 and 0 < s["long_packets"] < (n + 31) // 32 and s["long_ctas"] > 0, s


@pytest.mark.parametrize("case", SETS)
def test_every_scheduling_configuration_is_result_neutral(case):
    th, ph = mixed_angles(1000, 320)
    packets = (len(th) + 31) // 32
    want, s, _ = run(case, th, ph, lpt=0)
    assert s["long_packets"] == 0 and s["long_ctas"] == 0
    check_slots(want)

    def same(label, th=th, ph=ph, want=want, **knobs):
        got, s, tr = run(case, th, ph, lpt=2, **knobs)
        assert_bitwise(got, want, f"{case} {label}")
        return s, tr

    base, tr = same("defaults")
    assert base["long_packets"] > 0 and base["quarter_packets"] > 0 and base["long_ctas"] > 0, base
    assert base["long_packets"] < packets, base                          # the main region is not empty
    launches = tr.last_kernel_launches()
    s, _ = same("quarter = 0", quarter=0)
    assert s["long_packets"] > 0 and s["long_ctas"] > 0 and s["quarter_packets"] == 0, s
    s, t = same("exclusive = 0", exclusive=0)                             # one launch: main region first, then the long one
    assert s["long_packets"] > 0 and s["long_ctas"] == 0 and t.last_kernel_launches() == launches - 1, s
    s, _ = same("coop = 0", coop=0)
    assert s["long_packets"] == 0 and s["long_ctas"] == 0 and s["quarter_packets"] == 0, s
    _, t = same("dilate = 0", dilate=0)
    assert t.last_kernel_launches() == launches - 1
    _, t = same("dilate = 90 deg", dilate=90000)
    assert t.last_kernel_launches() == launches
    s, _ = same("long_alpha = 1", long_alpha=1)                           # every packet long
    assert s["long_packets"] == packets and s["long_ctas"] > 0, s
    s, _ = same("long_alpha huge", long_alpha=1 << 30)                     # none
    assert s["long_packets"] == 0 and s["long_ctas"] == 0 and s["quarter_packets"] == 0, s
    # one CTA for the long region: its four warps cap the quarter claims (three more warps per quarter packet)
    s, _ = same("quarter_alpha = 1, long_sm_pct = 1", quarter_alpha=1, long_sm_pct=1)
    assert s["long_ctas"] == 1 and s["quarter_packets"] == min(s["long_packets"], max(0, WARPS_PER_CTA - s["long_packets"]) // 3), s
    one, _, _ = run(case, th[:32], ph[:32], lpt=0)
    s, _ = same("one packet, quarter_alpha = 1, long_sm_pct = 1", th=th[:32], ph=ph[:32], want=one, quarter_alpha=1, long_sm_pct=1)
    assert s["long_packets"] == 1 and s["quarter_packets"] == 1 and s["long_ctas"] == 1, s
    costs = []
    for coarse in (1, 64):
        s, t = same(f"scout_coarse = {coarse}", scout_coarse=coarse)
        assert s["long_packets"] > 0, s
        costs.append(t.predicted_costs(len(th)))
    assert not np.array_equal(costs[0], costs[1])                         # the knob reached the cost scout


@pytest.mark.parametrize("case", SETS + ["3d_sub"])
def test_ray_alone_equals_ray_in_a_batch(case):
    """Range-dependent sets: a packet is traced serially, one lane per ray, until 8 or fewer of its rays are live, then four
    lanes per ray; a ray traced alone is in the cooperative mode from its first step.  The records must not depend on the
    mode.  The stratified 3-D set has no cooperative mode: a lane's result must not depend on its neighbours."""
    d, _ = util.load_case(case)
    if util.is_rngdep(int(d["variant"])):
        th, ph = seeded_angles(32, 23)
    else:
        th, ph = util.angles_rad(d["theta_deg"][:64], d["phi_deg"][:64])
    tr = make_tracer(case, knobs={"lpt": 0}, bounces=BOUNCES)
    batch = tr.trace(th, ph)
    check_slots(batch)
    assert (batch["status"][:, 0] == abi.ST_ARRIVAL).any()                # some rays reflect
    for i in range(len(th)):
        one = tr.trace(th[i:i + 1], ph[i:i + 1])
        assert_bitwise(one, {k: (v[:, i:i + 1] if k == "rec" else v[i:i + 1]) for k, v in batch.items()}, f"{case} ray {i}")


@pytest.mark.parametrize("case", ["3drngdep_path", "globalrngdep_path", "3drngdep_c4"])
def test_capture_kernels_are_schedule_neutral(case):
    """geoac_trace_paths (dense) under the claim order: one launch claims the whole order (main region, long region,
    quarter packets), and the raypath rows, row counts and caustic events equal those of the natural order."""
    d, kv = util.load_case(case)
    if "path_stride" in kv:
        th, ph = util.angles_rad(d["theta_deg"], d["phi_deg"])
        stride = int(kv["path_stride"])
    else:
        th, ph = seeded_angles(96, 31)
        stride = 25
    outs = []
    for lpt in (0, 2):
        tr = make_tracer(case, knobs={"lpt": lpt}, accum_per_segment=1)
        outs.append(tr.trace_paths(th, ph, stride, 4000, caustic_cap=64))
        s = tr.last_schedule()
        if lpt:
            assert tr.last_kernel_launches() > 1 and s["long_packets"] > 0 and s["long_ctas"] == 0, s
    a, b = outs
    assert_bitwise(b, a, case)
    for k in ("path_rows", "caustic_rows"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("path", "caustic"):
        assert np.array_equal(a[k].view(np.uint64), b[k].view(np.uint64)), k
    assert a["path_rows"].min() > 0 and a["path_rows"].max() < 4000
