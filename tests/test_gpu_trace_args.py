"""Capture arguments of geoac_trace_paths and geoac_trace_paths_compact (called through the C ABI on a 3-D context with
ToyAtmo): each single invalid input is refused with its return code and message, the empty batch and a too-small compacted
buffer are answered as include/geoac_b200.h documents, and a context that refused all of them still traces exactly like a
fresh one."""
import ctypes as C

import numpy as np
import pytest

import geoac_b200 as g
from geoac_b200 import abi, api
from tests import util

pytestmark = pytest.mark.gpu

N, STRIDE, CAP, CCAP = 24, 25, 400, 8
DP, IP, LP = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int64)


def _tracer():
    tr = g.Tracer(abi.GEOAC_3D, 0)
    tr.set_atmosphere_1d(*api.load_met_1d(util.TOY))
    p = tr.params
    p.bounces, p.accum_per_segment = 1, 1            # capture rows need the per-segment accumulation
    tr.params = p
    return tr


def _set(tr, **kv):
    p = tr.params
    for k, v in kv.items():
        setattr(p, k, v)
    tr.params = p


def _ptr(a, t):
    return None if a is None else a.ctypes.data_as(t)


def _call(tr, compact, n=N, stride=STRIDE, cap=CAP, ccap=CCAP, total=N * CAP, ctotal=N * CCAP, **null):
    """One call with valid buffers for N rays; `n`, the capture sizes and (set to None) any buffer can be overridden."""
    th, ph = util.angles_rad(np.linspace(4.0, 44.0, N), np.linspace(-120.0, 60.0, N))
    n_rec = tr.params.bounces + 1
    b = {"theta": th, "phi": ph, "rec": np.zeros((abi.NFIELDS, N, n_rec)), "status": np.zeros((N, n_rec), np.int32),
         "n_steps": np.zeros((N, n_rec), np.int32)}
    if compact:
        b.update(path=np.zeros((max(total, 1), abi.PATH_NF)), path_index=np.full(N + 1, -1, np.int64),
                 caustic=np.zeros((max(ctotal, 1), abi.CAUSTIC_NF)), caustic_index=np.full(N + 1, -1, np.int64))
    else:
        b.update(path=np.zeros((N, CAP, abi.PATH_NF)), path_index=np.zeros(N, np.int32),
                 caustic=np.zeros((N, CCAP, abi.CAUSTIC_NF)), caustic_index=np.zeros(N, np.int32))
    keep = dict(b)
    b.update(null)
    head = (tr._h, n, _ptr(b["theta"], DP), _ptr(b["phi"], DP), _ptr(b["rec"], DP), _ptr(b["status"], IP), _ptr(b["n_steps"], IP))
    if compact:
        rc = api.lib().geoac_trace_paths_compact(*head, stride, cap, total, _ptr(b["path"], DP), _ptr(b["path_index"], LP),
                                                 ccap, ctotal, _ptr(b["caustic"], DP), _ptr(b["caustic_index"], LP))
    else:
        rc = api.lib().geoac_trace_paths(*head, stride, cap, _ptr(b["path"], DP), _ptr(b["path_index"], IP),
                                         ccap, _ptr(b["caustic"], DP), _ptr(b["caustic_index"], IP))
    return rc, keep


def _error(tr):
    return api.lib().geoac_last_error(tr._h).decode()


@pytest.mark.parametrize("compact", [False, True], ids=["dense", "compact"])
def test_each_invalid_capture_argument_is_refused(compact):
    tr = _tracer()
    bad = abi.GEOAC_ERR_BAD_ARG
    ask = "ask for raypath rows"
    path_msg = "raypath capture needs its buffers and a positive per-ray capacity" if compact else \
        "raypath capture needs path buffers and a positive row capacity"
    cases = [
        (dict(stride=-1), ask),
        (dict(ccap=-1), ask),
        (dict(stride=0, ccap=0), ask),
        (dict(cap=0), path_msg),
        (dict(path=None), path_msg),
        (dict(path_index=None), path_msg),
        (dict(caustic=None), "caustic capture needs its buffers"),
        (dict(caustic_index=None), "caustic capture needs its buffers"),
    ]
    for kw, msg in cases:
        rc, _ = _call(tr, compact, **kw)
        assert rc == bad and msg in _error(tr), (kw, rc, _error(tr))
    _set(tr, calc_amp=0)
    rc, _ = _call(tr, compact)
    assert rc == bad and "caustic capture needs calc_amp = 1" in _error(tr)
    _set(tr, calc_amp=1, accum_per_segment=0)
    rc, _ = _call(tr, compact)
    assert rc == bad and "need accum_per_segment = 1" in _error(tr)
    _set(tr, accum_per_segment=1)
    # refused without a message of their own: the last one stays
    before = _error(tr)
    for kw in (dict(n=-1), dict(theta=None), dict(phi=None), dict(rec=None), dict(status=None), dict(n_steps=None)):
        rc, _ = _call(tr, compact, **kw)
        assert rc == bad and _error(tr) == before, kw
    # after all of that the context traces like a fresh one
    rc, got = _call(tr, compact)
    fresh = _tracer()
    rc2, want = _call(fresh, compact)
    assert rc == rc2 == abi.GEOAC_OK
    for k in ("rec", "status", "n_steps", "path", "path_index", "caustic", "caustic_index"):
        assert np.array_equal(got[k], want[k]), k
    assert (want["status"] == abi.ST_ARRIVAL).any() and want["path"].any()
    assert tr.last_stats()[0] == fresh.last_stats()[0]


def test_empty_batch_and_too_small_compacted_buffer():
    tr = _tracer()
    rc, b = _call(tr, True, n=0)
    assert rc == abi.GEOAC_OK and b["path_index"][0] == 0 and b["caustic_index"][0] == 0
    rc, _ = _call(tr, False, n=0)
    assert rc == abi.GEOAC_OK
    # a too-small row buffer: TOO_LARGE, with the records and the raypath offsets written (the last one is the size needed)
    _, dense = _call(tr, False)
    kept = np.minimum(dense["path_index"], CAP)                  # rows past the per-ray capacity are counted, not kept
    rc, b = _call(tr, True, total=7)
    assert rc == abi.GEOAC_ERR_TOO_LARGE and "rows produced" in _error(tr)
    assert np.array_equal(np.diff(b["path_index"]), kept) and b["path_index"][-1] > 7
    for k in ("rec", "status", "n_steps"):
        assert np.array_equal(b[k], dense[k]), k
    rc, b = _call(tr, True, total=int(kept.sum()))
    assert rc == abi.GEOAC_OK and np.array_equal(np.diff(b["path_index"]), kept)
