"""CPU tests of geoac_sample_atmosphere's per-point code (geoac_b200/csrc/atmo_sample.cuh) compiled with g++ through
tests/atmo_sample/host_sample.cpp, against the oracle's row (tests/atmo_sample/oracle_row.c): seeded points uniform in the
domain, on knots / grid nodes, on the cell edges of each axis, on the first and last knots and outside the domain, on ToyAtmo
(3D), the config-3 profile (Global) and the two committed grid fixtures.  Also the NULL-context return of the C entry point."""
import ctypes as C

import numpy as np
import pytest

from geoac_b200 import abi, api
from tests import atmo_sample_cases as S

CASES = [(c[0], c[1], c[2], c[3], {}) for c in S.CPU_CASES] + [
    ("toy_3d_medium", abi.GEOAC_3D, "profile", "toy", S.MEDIUM),
    ("grid_cart_medium", abi.GEOAC_3D_RNGDEP, "grid", "grid_cart", S.MEDIUM),
]


@pytest.mark.parametrize("label,variant,kind,source,medium", CASES, ids=[c[0] for c in CASES])
def test_host_emulation_matches_oracle(oracle, label, variant, kind, source, medium):
    arrays = S.load(kind, source, oracle)
    p = S.params(oracle, variant, medium)
    pts = S.points(S.axes(variant, kind, arrays), seed=S.SEED)
    want = S.oracle_rows(oracle, S.oracle_atmo(oracle, variant, kind, arrays, p), pts, p.freq)
    got = S.emul_rows(variant, kind, arrays, p, pts)
    problems, _ = S.check(got, want, p, label)
    assert not problems, "\n".join(problems)


def test_sample_refuses_a_null_context(built_lib):
    x = np.zeros(4)
    d = x.ctypes.data_as(C.POINTER(C.c_double))
    assert api.lib().geoac_sample_atmosphere(None, 1, d, d, d, d) == abi.GEOAC_ERR_BAD_ARG
    assert api.lib().geoac_sample_atmosphere(None, 0, None, None, None, None) == abi.GEOAC_ERR_BAD_ARG
