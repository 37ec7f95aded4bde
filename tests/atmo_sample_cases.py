"""Atmospheres, seeded point sets and per-column tolerances shared by the geoac_sample_atmosphere tests (host emulation on the
CPU, the device on a B200).  Every case is evaluated against the oracle's row (tests/atmo_sample/oracle_row.c, linked against
the CPU oracle): the reference's c / u / v / rho, *_diff, SuthBass_Alpha and Eval_Spline_AllOrder2 with every spline cursor
reset first.  The two helper libraries are compiled into a temporary directory on first use."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from geoac_b200 import abi
from tests import util

R_EARTH = 6370.0
SEED = 20261020
MEDIUM = {"freq": 0.5, "tweak_abs": 0.7, "z_grnd": 0.35}     # a non-default absorption set-up
DP = C.POINTER(C.c_double)


HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "atmo_sample")
_LIBS = {}


def _p(a):
    return a.ctypes.data_as(DP)


def _helper(name):
    """Compile one helper library (once per process): 'emul' (host_sample.cpp with the flags of tests/emul.py) or 'oracle'
    (oracle_row.c with the oracle's flags, linked against oracle/liboracle.so)."""
    if name not in _LIBS:
        out = os.path.join(tempfile.mkdtemp(prefix="atmo_sample"), f"lib{name}.so")
        if name == "emul":
            cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-mfma", "-ffp-contract=fast", os.path.join(HERE, "host_sample.cpp")]
        else:
            from oracle import pyoracle as po
            odir = os.path.dirname(po.build())
            cmd = ["gcc", "-O2", "-ffp-contract=off", "-fPIC", "-std=c11", "-shared", os.path.join(HERE, "oracle_row.c"),
                   "-L" + odir, "-loracle", "-Wl,-rpath," + odir, "-lm"]
        subprocess.check_call(cmd + ["-o", out])
        _LIBS[name] = C.CDLL(out)
    return _LIBS[name]


# ---------------------------------------------------------------- atmospheres
def profile(po, name):
    """z, T, u, v, rho of a stratified profile: 'toy' (ToyAtmo.met, Cartesian taper) or 'config3' (Global taper)."""
    if name == "toy":
        return po.load_met_1d(util.TOY)
    from geoac_b200 import synth
    path = os.path.join(tempfile.mkdtemp(prefix="c3"), "c3.met")
    synth.write_met(path, synth.config3_profile())
    return po.load_met_1d(path, global_taper=True)


def grid(name):
    """ax0, ax1, axz, T, u, v, rho of a committed grid fixture (tests/golden/<name>.npz)."""
    g = np.load(os.path.join(util.GOLD, name + ".npz"))
    return [np.ascontiguousarray(g[k]) for k in ("ax0", "ax1", "axz", "T", "u", "v", "rho")]


# (label, variant, kind, source): kind 'profile' or 'grid'
CPU_CASES = [
    ("toy_3d", abi.GEOAC_3D, "profile", "toy"),
    ("config3_global", abi.GEOAC_GLOBAL, "profile", "config3"),
    ("grid_cart", abi.GEOAC_3D_RNGDEP, "grid", "grid_cart"),
    ("grid_glob", abi.GEOAC_GLOBAL_RNGDEP, "grid", "grid_glob"),
]
GPU_CASES = [("toy_2d", abi.GEOAC_2D, "profile", "toy")] + CPU_CASES + [
    ("grid_c4", abi.GEOAC_3D_RNGDEP, "grid", "grid_c4"),
    ("grid_c5", abi.GEOAC_GLOBAL_RNGDEP, "grid", "grid_c5"),
]


def params(po, variant, medium=None):
    p = po.default_params(variant)
    for k, v in (medium or {}).items():
        setattr(p, k, v)
    return p


def load(kind, source, po):
    return profile(po, source) if kind == "profile" else grid(source)


def axes(variant, kind, arrays):
    """Knots of the three coordinates in the variant's order.  A stratified atmosphere has knots in the vertical only; its
    horizontal coordinates get a plain range (they are not read)."""
    glob = util.is_global(variant)
    if kind == "profile":
        z = np.asarray(arrays[0], dtype=np.float64) + (R_EARTH if glob else 0.0)
        if glob:
            return [z, np.array([-1.2, 1.2]), np.array([-3.0, 3.0])]
        return [np.array([-800.0, 800.0]), np.array([-800.0, 800.0]), z]
    ax0, ax1, axz = arrays[:3]
    if glob:
        return [np.asarray(axz) + R_EARTH, np.asarray(ax0), np.asarray(ax1)]
    return [np.asarray(ax0), np.asarray(ax1), np.asarray(axz)]


# ---------------------------------------------------------------- points
def points(ax, seed, n=2000):
    """About n points (p0, p1, p2) from a fixed seed: uniform in the domain, exactly on knots / grid nodes, on the cell edges
    of each axis separately, on the first and last knot of each axis, and outside the domain in each coordinate (by up to 5 %
    of the axis span, which keeps the altitude inside the absorption model's polynomial range)."""
    rng = np.random.default_rng(seed)
    lo, hi = [a[0] for a in ax], [a[-1] for a in ax]
    m = n // 10

    def uniform(k):
        return np.column_stack([rng.uniform(lo[j], hi[j], k) for j in range(3)])

    def knots(j, k):
        return rng.choice(ax[j], k)

    blocks = [uniform(3 * m)]
    blocks.append(np.column_stack([knots(j, m) for j in range(3)]))           # grid nodes
    for j in range(3):                                                        # cell edges of axis j
        b = uniform(m); b[:, j] = knots(j, m); blocks.append(b)
    for j in range(3):                                                        # first / last knot of axis j
        b = uniform(m // 2); b[:, j] = np.where(rng.random(m // 2) < 0.5, lo[j], hi[j]); blocks.append(b)
    for j in range(3):                                                        # outside in coordinate j
        b = uniform(m // 2)
        d = rng.uniform(0.0, 0.05, m // 2) * (hi[j] - lo[j])
        b[:, j] = np.where(rng.random(m // 2) < 0.5, lo[j] - d, hi[j] + d); blocks.append(b)
    P = np.concatenate(blocks)
    return [np.ascontiguousarray(P[:, j]) for j in range(3)]


# ---------------------------------------------------------------- the oracle
def oracle_atmo(po, variant, kind, arrays, params):
    L = _helper("oracle")
    L.orc_row_set_medium.argtypes = [C.c_void_p, C.c_double, C.c_double]
    at = po.atmo1d(util.is_global(variant), *arrays) if kind == "profile" else po.atmo3d(util.is_global(variant), *arrays)
    L.orc_row_set_medium(at.h, params.z_grnd, params.tweak_abs)
    return at


def oracle_rows(po, at, pts, freq):
    L = _helper("oracle")
    L.orc_row_sample.argtypes = [C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_double, DP]
    n = len(pts[0])
    out = np.zeros((abi.ATM_NF, n))
    row = np.zeros(abi.ATM_NF)
    for i in range(n):
        L.orc_row_sample(at.h, float(pts[0][i]), float(pts[1][i]), float(pts[2][i]), freq, _p(row))
        out[:, i] = row
    return out


# ---------------------------------------------------------------- the bar
# Per output column: max|got - oracle| <= TOL[col] * scale[col].  TOL_MEASURED is the largest deviation measured over the host
# emulation and the device (one B200) on every atmosphere of GPU_CASES, medium cases included; TOL is 10x that, rounded up to
# 1, 2 or 5 times a power of ten, and at least 1e-15 where nothing was measured (the absorption column beyond its allowance).
# The loosest is 5e-12 (second derivatives of T on the Global grids, in their scaled units); none is looser than 1e-10.
TOL_MEASURED = np.array([
    2.2e-15, 2.5e-15, 5.6e-16, 3.5e-16, 5.1e-15, 4.3e-15, 6.0e-16, 0.0e+00, 2.8e-15, 1.7e-15,
    1.2e-13, 1.7e-13, 1.1e-15, 1.7e-13, 3.0e-13, 6.6e-15, 6.4e-15, 2.5e-13, 2.5e-15, 2.6e-16,
    4.0e-15, 4.4e-15, 1.7e-14, 4.2e-14, 3.8e-14, 3.5e-15, 3.5e-15, 4.8e-14, 6.7e-16, 2.5e-16,
    1.1e-16, 1.7e-15, 7.9e-15, 3.3e-17, 4.1e-14, 2.7e-17, 2.3e-16, 5.9e-16,
])
TOL = np.array([
    5e-14, 5e-14, 1e-14, 5e-15, 1e-13, 5e-14, 1e-14, 1e-15, 5e-14, 2e-14,
    2e-12, 2e-12, 2e-14, 2e-12, 5e-12, 1e-13, 1e-13, 5e-12, 5e-14, 5e-15,
    5e-14, 5e-14, 2e-13, 5e-13, 5e-13, 5e-14, 5e-14, 5e-13, 1e-14, 5e-15,
    2e-15, 2e-14, 1e-13, 1e-15, 5e-13, 1e-15, 5e-15, 1e-14,
])


def column_scales(want):
    """max|oracle column|, except that a derivative of T, u or v is measured against the largest of its siblings of the same
    order (the three first or the six second derivatives of that field).  A derivative that vanishes identically -- a wind that
    does not vary along an axis, as in the synthetic grids -- comes out as rounding noise (~1e-21) from the oracle's 16x16
    patch fits and as an exact or near zero from the tensor-product form; against its own noise it has no scale at all."""
    scale = np.abs(want).max(axis=1)
    for b in (abi.ATM_T, abi.ATM_UF, abi.ATM_VF):
        for lo, hi in ((b + 1, b + 4), (b + 4, b + 10)):
            scale[lo:hi] = scale[lo:hi].max()
    return scale


def alpha_allowance(params, c):
    """Absolute slack of the absorption column.  The classical term carries sqrt(1 + nu^2) - 1; at low altitude nu^2 is below
    one ulp of 1, so that factor is a staircase of rounding steps of size ~2^-52 in the reference itself (DESIGN section 3,
    "Lean Sutherland-Bass").  Two steps of it: 2 x 8.685889 x tweak_abs x (2 pi freq / c) x sqrt(0.5 x 2^-52)."""
    return 2.0 * 8.685889 * params.tweak_abs * (2.0 * np.pi * params.freq / c) * np.sqrt(0.5 * 2.0 ** -52)


def check(got, want, params, label):
    """Problems (empty = pass) and the measured deviation of every column relative to its scale (absolute where the scale
    is 0: the columns a stratified atmosphere leaves at 0)."""
    scale = column_scales(want)
    err = np.abs(got - want)
    err[abi.ATM_ALPHA] = np.maximum(err[abi.ATM_ALPHA] - alpha_allowance(params, want[abi.ATM_C]), 0.0)
    rel = err.max(axis=1) / np.where(scale > 0, scale, 1.0)
    problems = []
    for f in range(abi.ATM_NF):
        if not np.all(np.isfinite(got[f])):
            problems.append(f"{label}: column {f} has non-finite values")
        elif rel[f] > TOL[f]:
            i = int(np.argmax(err[f]))
            problems.append(f"{label}: column {f}: {rel[f]:.3e} > {TOL[f]:g} (point {i}: got {got[f, i]!r}, want {want[f, i]!r})")
    return problems, rel


# ---------------------------------------------------------------- the host emulation (tests/atmo_sample/host_sample.cpp, g++)
def emul_rows(variant, kind, arrays, params, pts):
    from tests import emul
    L = _helper("emul")
    n = len(pts[0])
    out = np.zeros((abi.ATM_NF, n))
    P = [np.ascontiguousarray(a, dtype=np.float64) for a in pts]
    if kind == "profile":
        L.emul_sample_1d.argtypes = [C.c_int, C.POINTER(abi.GeoacParams), C.c_int, DP, C.c_long, DP, DP, DP]
        tab, nt = emul.make_table(util.is_global(variant), *arrays)
        tab = np.ascontiguousarray(tab)
        L.emul_sample_1d(variant, C.byref(params), nt, _p(tab), n, _p(P[0]), _p(P[2]), _p(out))
    else:
        L.emul_sample_3d.argtypes = [C.c_int, C.POINTER(abi.GeoacParams), C.c_int, C.c_int, C.c_int] + [DP] * 7 + [C.c_long, DP, DP, DP, DP]
        A = [np.ascontiguousarray(a, dtype=np.float64) for a in arrays]
        L.emul_sample_3d(variant, C.byref(params), len(A[0]), len(A[1]), len(A[2]), *[_p(a) for a in A], n, *[_p(a) for a in P], _p(out))
    return out
