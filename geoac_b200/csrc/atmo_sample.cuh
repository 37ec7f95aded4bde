// atmo_sample.cuh -- the atmosphere as the kernels evaluate it, at arbitrary points (geoac_sample_atmosphere).
//
// One point = one row of GEOAC_ATM_NF values (include/geoac_b200.h): c, u, v, rho and the vertical derivatives of c, u, v as
// travel time, absorption, amplitude and reflection see them (the 1-D spline, or the range-dependent scalar wrappers
// ms_wrappers), the Sutherland-Bass coefficient with the full model, and the value, gradient and Hessian of T, u, v as the
// right-hand side sees them (the 1-D spline's f, f', f'', or ms_sample_tuv with the reference's slips, App. A-8 / A-9).
//
// Every point is evaluated as the reference evaluates it from COLD cursors (accel = 0), so a row does not depend on the
// points evaluated before it.  That matters on the grids, where the bicubic patch is only C1 across cell edges: on a grid
// line the Hessian columns depend on the cell the search picks.  The device kernel (capi.cu) and tests/atmo_sample run this
// same code.
#pragma once
#include "core.cuh"
#include "mspline.cuh"

namespace geoac {

// Find_Segment of the 1-D spline from cursor 0 (G2S_Spline1D.cpp:202-243) for a point already clamped into the table: the
// interval [x_k, x_k+1] that holds it, by bisection.  On an interior knot m the reference's first tests (cursor interval 0,
// then interval 1) and its two-ended scan pick interval m-1 when m <= 2 or m lies in the lower half (2m <= n-1), else m.
GEOAC_HD int seg_find_cold(const Table1D& t, double xc) {
    int lo = 0, hi = t.n - 1;                                  // invariant: x[lo] <= xc, and xc < x[hi] unless hi = n-1
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (t.lvl(mid)[TAB_X] <= xc) lo = mid; else hi = mid;
    }
    if (lo > 0 && xc == t.lvl(lo)[TAB_X] && (lo <= 2 || 2 * lo <= t.n - 1)) --lo;
    return lo;
}

// Output row of one point: out[f * stride], f = 0 .. GEOAC_ATM_NF-1.  T/u/v blocks in the variant's coordinate order.
GEOAC_HD void sample_store_block(double* out, int64_t stride, int first, const double (&d)[10]) {
#pragma unroll
    for (int i = 0; i < 10; i++) out[(int64_t)(first + i) * stride] = d[i];
}

// Stratified atmospheres (2D / 3D: vertical coordinate p2 [km]; Global: p0 = r [km from the Earth's centre]).
template <bool GLOBAL>
GEOAC_HD void sample_point_1d(const LaunchConsts& L, const Table1D& T, double p0, double p2, double* out, int64_t stride) {
    const double xq = GLOBAL ? p0 : p2;
    int k = seg_find_cold(T, clampd(xq, T.xmin, T.xmax));
    const SegPos sp = seg_locate(T, xq, k);                    // the cursor already holds the point: no walk
    double Tv, dT, ddT, u, du, ddu, v, dv, ddv;
    spl_f2(T, TAB_T, sp, Tv, dT, ddT);
    spl_f2(T, TAB_U, sp, u, du, ddu);
    spl_f2(T, TAB_V, sp, v, dv, ddv);
    const double rho = spl_f(T, TAB_RHO, sp);
    const double c = sqrt(kGamR * Tv);                         // as fill_launch_consts_1d
    const double gT = kGamR * Tv, inv_c = g_rsqrt(gT);         // as the segment routines hand c to the absorption model
    const double alpha = suthbass_alpha(L, L.sb, GLOBAL ? xq - kREarth : xq, gT * inv_c, inv_c, rho);
    const double row[8] = { c, u, v, rho, kGamR / (2.0 * c) * dT, du, dv, alpha };
#pragma unroll
    for (int i = 0; i < 8; i++) out[(int64_t)i * stride] = row[i];
    // f, d0, d1, d2, d00, d11, d22, d01, d02, d12: only the vertical entries are non-zero
    const int d1 = GLOBAL ? 1 : 3, d2 = GLOBAL ? 4 : 6;
    const double f[3] = { Tv, u, v }, df[3] = { dT, du, dv }, ddf[3] = { ddT, ddu, ddv };
#pragma unroll
    for (int F = 0; F < 3; F++) {
        double blk[10];
#pragma unroll
        for (int i = 0; i < 10; i++) blk[i] = 0.0;
        blk[0] = f[F]; blk[d1] = df[F]; blk[d2] = ddf[F];
        sample_store_block(out, stride, GEOAC_ATM_T + 10 * F, blk);
    }
}

// Range-dependent atmospheres: Cartesian (x, y, z) = grid axes (ax0, ax1, vertical); Global (r, lat, lon) = (vertical, ax0, ax1).
template <bool GLOBAL>
GEOAC_HD void sample_point_grid(const LaunchConsts& L, const Grid3D& g, double p0, double p1, double p2, double* out, int64_t stride) {
    const double a = GLOBAL ? p1 : p0, b = GLOBAL ? p2 : p1, z = GLOBAL ? p0 : p2;
    Cur3 cold;
    cold.ka = ms_find_cold(g.ax0, g.n0, clampd(a, g.amin, g.amax));
    cold.kb = ms_find_cold(g.ax1, g.n1, clampd(b, g.bmin, g.bmax));
    cold.kz = ms_find_cold(g.axz, g.nz, clampd(z, g.zmin, g.zmax));
    Cur3 cur = cold;
    double w[4], dz[3];
    ms_wrappers<GLOBAL, true, true>(g, a, b, z, cur, w, dz);
    const double c = sqrt(kGamR * w[0]);                        // as fill_launch_consts_3d
    const double gT = kGamR * w[0], inv_c = g_rsqrt(gT);
    double alpha;
    if (GLOBAL) {
        // reference state under the point at the lowest level (EqGlobalRD::segment, App. A-14)
        double wr[4], dzr[3];
        Cur3 cg = cold; cg.kz = 0;
        ms_wrappers<true, true, false, true>(g, a, b, L.z_grnd, cg, wr, dzr);
        SBRef ref; suthbass_ref(ref, sqrt(kGamR * wr[0]), wr[3]);
        alpha = suthbass_alpha(L, ref, z - kREarth, gT * inv_c, inv_c, w[3]);
    } else {
        alpha = suthbass_alpha(L, L.sb, z, gT * inv_c, inv_c, w[3]);
    }
    const double row[8] = { c, w[1], w[2], w[3], kGamR / (2.0 * c) * dz[0], dz[1], dz[2], alpha };
#pragma unroll
    for (int i = 0; i < 8; i++) out[(int64_t)i * stride] = row[i];
    // ms_sample_tuv slots (0 f, 1 a, 2 b, 3 z, 4 aa, 5 bb, 6 zz, 7 ab, 8 az, 9 bz) -> f, d0, d1, d2, d00, d11, d22, d01, d02, d12
    // of the variant's coordinates; Global (r, lat, lon) = (z, a, b), as orc_mspline_allorder2 reorders them
    double S[3][10];
    cur = cold;
    ms_sample_tuv<GLOBAL, true>(g, a, b, z, cur, S);
#pragma unroll
    for (int F = 0; F < 3; F++) {
        double blk[10];
        if (GLOBAL) {
            const double* s = S[F];
            blk[0] = s[0]; blk[1] = s[3]; blk[2] = s[1]; blk[3] = s[2]; blk[4] = s[6];
            blk[5] = s[4]; blk[6] = s[5]; blk[7] = s[8]; blk[8] = s[9]; blk[9] = s[7];
        } else {
#pragma unroll
            for (int i = 0; i < 10; i++) blk[i] = S[F][i];
        }
        sample_store_block(out, stride, GEOAC_ATM_T + 10 * F, blk);
    }
}

}  // namespace geoac
