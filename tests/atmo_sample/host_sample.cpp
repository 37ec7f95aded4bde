// tests/atmo_sample/host_sample.cpp -- TEST-ONLY: geoac_sample_atmosphere's per-point code (geoac_b200/csrc/atmo_sample.cuh)
// compiled with g++, so that it can be checked against the oracle where there is no GPU.  Tables are built with the host
// recurrences the device build is bit-identical to (host_tables.hpp); the invariants are filled as refresh_consts fills them.
// Rows: out[f * n_pts + i].
#include <algorithm>
#include <cstring>
#include <vector>
#include "../../geoac_b200/csrc/core.cuh"
#include "../../geoac_b200/csrc/mspline.cuh"
#include "../../geoac_b200/csrc/eq_rngdep.cuh"
#include "../../geoac_b200/csrc/trace_kernel.cuh"
#include "../../geoac_b200/csrc/atmo_sample.cuh"
#include "../../geoac_b200/csrc/host_tables.hpp"

using namespace geoac;

// Only the medium parameters (z_grnd, tweak_abs, freq) and the source reach the sampler.
static LaunchConsts sample_consts(int variant, const geoac_params* p) {
    LaunchConsts L; std::memset(&L, 0, sizeof L);
    L.z_grnd = p->z_grnd; L.tweak_abs = p->tweak_abs; L.freq = p->freq;
    for (int i = 0; i < 3; i++) L.src[i] = p->src[i];
    if (variant == GEOAC_2D || variant == GEOAC_3D || variant == GEOAC_3D_RNGDEP) L.src[2] = std::max(p->z_grnd, p->src[2]);
    else L.src[0] = std::max(p->z_grnd, p->src[0]);
    return L;
}

// stratified: `table` is the device layout of core.cuh (one TAB_NARR record per level)
extern "C" void emul_sample_1d(int variant, const geoac_params* p, int n, const double* table, long n_pts,
                               const double* p0, const double* p2, double* out) {
    Table1D T; T.base = table; T.n = n; T.xmin = table[TAB_X]; T.xmax = table[(size_t)(n - 1) * TAB_NARR + TAB_X]; T.jump_scale = 0.0;
    LaunchConsts L = sample_consts(variant, p);
    fill_launch_consts_1d(L, T, variant);
    for (long i = 0; i < n_pts; i++) {
        if (variant == GEOAC_GLOBAL) sample_point_1d<true>(L, T, p0[i], p2[i], out + i, n_pts);
        else sample_point_1d<false>(L, T, p0[i], p2[i], out + i, n_pts);
    }
}

// range-dependent: fields dense [n0][n1][nz] exactly as geoac_set_atmosphere_3d receives them
extern "C" void emul_sample_3d(int variant, const geoac_params* p, int n0, int n1, int nz, const double* ax0, const double* ax1, const double* axz,
                               const double* Tf, const double* uf, const double* vf, const double* rhof, long n_pts,
                               const double* p0, const double* p1, const double* p2, double* out) {
    const bool glob = variant == GEOAC_GLOBAL_RNGDEP;
    std::vector<double> z, tuv, rh;
    build_grid_tables(glob, n0, n1, nz, ax0, ax1, axz, Tf, uf, vf, rhof, z, tuv, rh);
    std::vector<double> r0, r1, rz;
    build_axis_records(ax0, n0, r0); build_axis_records(ax1, n1, r1); build_axis_records(z.data(), nz, rz);
    Grid3D g; g.tuv = tuv.data(); g.rho = rh.data(); g.ax0 = r0.data(); g.ax1 = r1.data(); g.axz = rz.data(); g.n0 = n0; g.n1 = n1; g.nz = nz;
    g.amin = ax0[0]; g.amax = ax0[n0 - 1]; g.bmin = ax1[0]; g.bmax = ax1[n1 - 1]; g.zmin = z[0]; g.zmax = z[nz - 1];
    g.scratch = nullptr; g.role = 0; g.nrole = 1; g.glane0 = 0; g.gmask = 0;
    LaunchConsts L = sample_consts(variant, p);
    fill_launch_consts_3d(L, g, variant);
    for (long i = 0; i < n_pts; i++) {
        if (glob) sample_point_grid<true>(L, g, p0[i], p1[i], p2[i], out + i, n_pts);
        else sample_point_grid<false>(L, g, p0[i], p1[i], p2[i], out + i, n_pts);
    }
}
