"""geoac_trace_device -- the entry point bench.py times: torch device buffers, the caller's stream, no synchronisation --
against geoac_trace of the same batch on a fresh context, bit for bit (status, n_steps and every record field), for all ten
trace kernels (five variants x calc_amp).  The host trace is the path the golden and oracle parity tests check, so the
equality carries their verdict over to the device path.  Also: outputs filled with garbage beforehand, the legacy default
stream and a side stream, the long-region fork / join, parameter changes, back-to-back calls, the reported counters and
kernel time, and the argument checks."""
import math

import numpy as np
import pytest
import torch

import geoac_b200 as g
from geoac_b200 import abi, api
from tests import util

pytestmark = pytest.mark.gpu

# stratified sets: golden angles on their profiles; range-dependent sets: a seeded batch on the committed config-4 / config-5
# grid fixtures with the parameters of the golden cases traced on them
CASES = {abi.GEOAC_2D: "2d_config1", abi.GEOAC_3D: "3d_sub", abi.GEOAC_GLOBAL: "global_sub",
         abi.GEOAC_3D_RNGDEP: "3drngdep_c4", abi.GEOAC_GLOBAL_RNGDEP: "globalrngdep_c5"}


def make_tracer(case, calc_amp=1, knobs=None, **params):
    """A context with the atmosphere and parameters of golden case `case`; `params` override fields of geoac_params."""
    d, kv = util.load_case(case)
    variant = int(d["variant"])
    tr = g.Tracer(variant, 0)
    for k, v in (knobs or {}).items():
        tr.set_knob(k, v)
    if util.is_rngdep(variant):
        tr.set_atmosphere_3d(*util.load_grid(d))
    else:
        tr.set_atmosphere_1d(*g.load_met_1d(util.profile_path(d), global_taper=util.is_global(variant)))
    p = util.apply_keys(variant, tr.params, kv)
    p.calc_amp = calc_amp
    for k, v in params.items():
        setattr(p, k, v)
    tr.params = p
    return tr


def seeded_angles(n, seed, th_lo=1.0, th_hi=51.0):
    rng = np.random.default_rng(seed)
    return util.angles_rad(rng.uniform(th_lo, th_hi, n), rng.uniform(-180.0, 180.0, n))


def case_angles(case, n_rngdep=160, seed=20261021):
    d, _ = util.load_case(case)
    if util.is_rngdep(int(d["variant"])):
        return seeded_angles(n_rngdep, seed)
    return util.angles_rad(d["theta_deg"], d["phi_deg"])


class DeviceBuffers:
    """Angles and outputs of one batch as torch tensors on cuda:0, the outputs filled with 0xFF bytes (NaN records,
    status / n_steps -1) so that a slot the call does not write shows."""

    def __init__(self, th, ph, n_rec):
        dev = torch.device("cuda", 0)
        self.n, self.n_rec = len(th), n_rec
        self.th = torch.from_numpy(np.ascontiguousarray(th)).to(dev)
        self.ph = torch.from_numpy(np.ascontiguousarray(ph)).to(dev)
        self.rec = torch.empty((abi.NFIELDS, self.n * n_rec), dtype=torch.float64, device=dev)
        self.status = torch.empty(self.n * n_rec, dtype=torch.int32, device=dev)
        self.n_steps = torch.empty(self.n * n_rec, dtype=torch.int32, device=dev)
        self.rec.view(torch.int64).fill_(-1)
        self.status.fill_(-1)
        self.n_steps.fill_(-1)

    def trace(self, tr, stream):
        tr.trace_device(self.n, self.th.data_ptr(), self.ph.data_ptr(), self.rec.data_ptr(), self.status.data_ptr(),
                        self.n_steps.data_ptr(), stream.cuda_stream)

    def snapshot(self):
        """Copies of the outputs enqueued on the current stream (no synchronisation), as a dict of tensors."""
        return {"rec": self.rec.clone(), "status": self.status.clone(), "n_steps": self.n_steps.clone()}

    def host(self, snap):
        n, r = self.n, self.n_rec
        return {"rec": snap["rec"].cpu().numpy().reshape(abi.NFIELDS, n, r), "status": snap["status"].cpu().numpy().reshape(n, r),
                "n_steps": snap["n_steps"].cpu().numpy().reshape(n, r)}


def trace_device(tr, th, ph, stream=None):
    """One geoac_trace_device call on `stream` (default: the current stream, i.e. the legacy default stream as bench.py
    uses it) into garbage-filled buffers; the outputs are cloned on the same stream right after the call returns, and only
    then is the stream synchronised.  Returns host copies shaped like Tracer.trace's."""
    stream = stream if stream is not None else torch.cuda.current_stream()
    with torch.cuda.stream(stream):
        buf = DeviceBuffers(th, ph, tr.params.bounces + 1)
        buf.trace(tr, stream)
        snap = buf.snapshot()
    stream.synchronize()
    return buf.host(snap)


def assert_bitwise(got, want, label=""):
    for k in ("status", "n_steps"):
        assert np.array_equal(got[k], want[k]), f"{label}: {k} differs at {np.argwhere(got[k] != want[k])[:5].tolist()}"
    bad = np.argwhere(np.ascontiguousarray(got["rec"]).view(np.uint64) != np.ascontiguousarray(want["rec"]).view(np.uint64))
    assert bad.size == 0, f"{label}: {len(bad)} record values differ, first [field, ray, slot] {bad[:5].tolist()}"


@pytest.mark.parametrize("side_stream", [False, True], ids=["default_stream", "side_stream"])
@pytest.mark.parametrize("calc_amp", [1, 0])
@pytest.mark.parametrize("variant", sorted(CASES), ids=[abi.VARIANT_NAMES[v] for v in sorted(CASES)])
def test_trace_device_equals_host_trace(variant, calc_amp, side_stream):
    """Range-dependent sets with the claim order forced on: the long region gets its exclusive launch on the context's
    second stream, forked from and joined back into the caller's stream -- the outputs are cloned right after the call on
    that stream, so a missing join would show as records not yet written."""
    case = CASES[variant]
    th, ph = case_angles(case)
    want = make_tracer(case, calc_amp).trace(th, ph)
    rd = util.is_rngdep(variant)
    tr = make_tracer(case, calc_amp, knobs={"lpt": 2} if rd else None)
    got = trace_device(tr, th, ph, torch.cuda.Stream() if side_stream else None)
    assert_bitwise(got, want, case)
    assert (want["status"][:, 0] != abi.ST_NONE).all() and (want["status"] == abi.ST_ARRIVAL).any()
    if rd:
        s = tr.last_schedule()
        assert s["long_packets"] > 0 and s["long_ctas"] > 0, s


@pytest.mark.parametrize("case", ["3d_sub", "3drngdep_c4"])
def test_parameter_change_is_ordered_into_the_callers_stream(case):
    """New parameters are turned into launch invariants on the context's own stream; the call orders that work into the
    caller's stream.  A side stream, a trace with the old parameters, then new freq and bounces and an immediate call."""
    th, ph = case_angles(case, n_rngdep=64)
    tr = make_tracer(case)
    s = torch.cuda.Stream()
    trace_device(tr, th, ph, s)
    p = tr.params
    p.freq, p.bounces = 0.73, p.bounces + 1
    tr.params = p
    got = trace_device(tr, th, ph, s)
    want = make_tracer(case, freq=0.73, bounces=p.bounces).trace(th, ph)
    assert_bitwise(got, want, case)
    assert got["status"].shape[1] == p.bounces + 1


@pytest.mark.parametrize("case", ["3d_sub", "3drngdep_c4"])
def test_back_to_back_calls_on_one_stream_equal_a_single_call(case):
    """bench.py's loop: a 256 MB memset, then geoac_trace_device, three times on the legacy default stream without a
    synchronisation in between, into the same buffers.  The claim order is forced on, so the range-dependent calls each fork
    and join a long-region launch and reset the claim counters the previous call's launches used."""
    th, ph = case_angles(case)
    want = make_tracer(case).trace(th, ph)
    tr = make_tracer(case, knobs={"lpt": 2})
    stream = torch.cuda.current_stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    buf = DeviceBuffers(th, ph, tr.params.bounces + 1)
    for _ in range(3):
        flush.zero_()
        buf.trace(tr, stream)
    snap = buf.snapshot()
    stream.synchronize()
    assert_bitwise(buf.host(snap), want, case)


def test_counters_and_kernel_time_after_a_device_trace():
    """After geoac_trace_device and a synchronisation the step count is the one a host trace of the batch reports, and
    kernel_ms is the duration of this call's work, not the time of an earlier host trace."""
    th, ph = util.angles_rad(np.linspace(84.0, 88.0, 8), np.linspace(-90.0, 90.0, 8))   # steep rays: a short trace
    host = make_tracer("3d_sub")
    host.trace(th, ph)
    steps_host, _ = host.last_stats()
    tr = make_tracer("3d_sub")
    lth, lph = case_angles("3d_sub")                                          # shallow rays too: a much longer trace
    tr.trace(lth, lph)
    _, ms_long = tr.last_stats()
    stream = torch.cuda.current_stream()
    with torch.cuda.stream(stream):
        buf = DeviceBuffers(th, ph, tr.params.bounces + 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        buf.trace(tr, stream)
        e1.record(stream)
    stream.synchronize()
    steps, ms = tr.last_stats()
    assert steps == steps_host > 0
    assert math.isfinite(ms) and 0.0 < ms <= e0.elapsed_time(e1) + 0.01, (ms, e0.elapsed_time(e1))
    assert ms < ms_long, (ms, ms_long)
    assert tr.last_stats() == (steps, ms)                                    # stable once read
    tr.trace(lth, lph)                                                      # a host trace reports its own time again
    assert tr.last_stats()[1] > ms


def test_argument_checks():
    """Refused before anything is enqueued: NULL buffers with n_rays > 0, n_rays < 0 (GEOAC_ERR_BAD_ARG with a message),
    no atmosphere (GEOAC_ERR_NO_ATMO); n_rays == 0 is GEOAC_OK whatever the pointers.  The context then traces as before."""
    L = api.lib()
    th, ph = case_angles("3d_sub")
    tr = make_tracer("3d_sub")
    buf = DeviceBuffers(th, ph, tr.params.bounces + 1)
    ptrs = [buf.th.data_ptr(), buf.ph.data_ptr(), buf.rec.data_ptr(), buf.status.data_ptr(), buf.n_steps.data_ptr()]
    stream = torch.cuda.current_stream().cuda_stream
    call = lambda t, n, p: L.geoac_trace_device(t._h, n, *p, stream)
    for i in range(5):
        p = list(ptrs)
        p[i] = None
        assert call(tr, buf.n, p) == abi.GEOAC_ERR_BAD_ARG, i
        assert "geoac_trace_device: null buffer" in L.geoac_last_error(tr._h).decode(), i
    assert call(tr, -1, ptrs) == abi.GEOAC_ERR_BAD_ARG and "n_rays < 0" in L.geoac_last_error(tr._h).decode()
    assert call(tr, 0, [None] * 5) == abi.GEOAC_OK
    assert L.geoac_trace_device(None, buf.n, *ptrs, stream) == abi.GEOAC_ERR_BAD_ARG
    bare = g.Tracer(abi.GEOAC_3D, 0)
    assert call(bare, buf.n, ptrs) == abi.GEOAC_ERR_NO_ATMO and "atmosphere" in L.geoac_last_error(bare._h).decode()
    assert call(bare, 0, ptrs) == abi.GEOAC_OK
    torch.cuda.synchronize()
    assert (buf.host(buf.snapshot())["status"] == -1).all()                  # none of the refused calls wrote anything
    assert_bitwise(trace_device(tr, th, ph), make_tracer("3d_sub").trace(th, ph), "after the refusals")
