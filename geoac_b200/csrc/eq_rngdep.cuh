// eq_rngdep.cuh -- per-ray physics of the two range-dependent variants, de-duplicated for one thread per ray.
//
//   Eq3DRD     : 3-D Cartesian moving medium over a G2S node grid  (reference Code/GeoAc/GeoAc.EquationSets.3DRngDep.cpp)
//   EqGlobalRD : spherical-earth moving medium over a lat/lon grid (reference Code/GeoAc/GeoAc.EquationSets.GlobalRngDep.cpp)
//
// Both integrate all three eikonal components: y = [x(3), nu(3), X_theta(3), mu_theta(3), X_phi(3), mu_phi(3)]
// (Global: coordinates (r, lat, lon), wind order (w, v, u), w = 0).  One call of ms_sample_tuv per RK4 stage replaces
// the reference's three Eval_Spline_AllOrder2 calls; travel time / absorption / amplitude / reflection use the scalar
// wrappers' arithmetic (ms_wrappers), exactly like the reference does (SURVEY App. E-5).
#pragma once
#include "core.cuh"
#include "mspline.cuh"

namespace geoac {

// c, grad c and the launch-angle derivative of grad c from T and its derivatives (3DRngDep.cpp:277-293)
struct RdSound { double c, inv_c, hg, hg2; };
GEOAC_HD RdSound rd_sound(double T) {
    RdSound s; const double gT = kGamR * T;
    s.inv_c = g_rsqrt(gT); s.c = gT * s.inv_c;
    s.hg = 0.5 * kGamR * s.inv_c;             // gamR/(2c)
    s.hg2 = s.hg * s.hg * s.inv_c;            // gamR^2/(4c^3)
    return s;
}

// ======================================================= 3-D Cartesian, range dependent =======================
template <bool AMP>
struct Eq3DRD {
    using Scout = Eq3DRD<false>;           // amplitude-free set used by the cost scout (trace_kernel.cuh)
    static constexpr int NEQ = AMP ? 18 : 6;
    using Atmo = Grid3D;
    using Cursor = Cur3;
    static constexpr int VARIANT = GEOAC_3D_RNGDEP;

    struct RayC { double sth, cth, sph, cph; };

    GEOAC_HD static double altitude(const double* y) { return y[2]; }

    // GeoAc_SetInitialConditions, 3DRngDep.cpp:70-136
    GEOAC_HD static void init(const LaunchConsts& L, const Grid3D& G, double theta, double phi, RayC& rc, double* y, Cur3& cur) {
        sincos(theta, &rc.sth, &rc.cth); sincos(phi, &rc.sph, &rc.cph);
        const double inv_c0 = 1.0 / L.c_src;
        const double Mu = L.u_src * inv_c0, Mv = L.v_src * inv_c0;
        const double n0 = rc.cth * rc.cph, n1 = rc.cth * rc.sph, n2 = rc.sth;
        const double t0 = -rc.sth * rc.cph, t1 = -rc.sth * rc.sph, t2 = rc.cth;
        const double p0 = -rc.cth * rc.sph, p1 = rc.cth * rc.cph;
        const double MS = 1.0 + (n0 * Mu + n1 * Mv);
        const double iM = 1.0 / MS, iM2 = iM * iM;
        y[0] = L.src[0]; y[1] = L.src[1]; y[2] = L.src[2];
        y[3] = n0 * iM; y[4] = n1 * iM; y[5] = n2 * iM;
        if (AMP) {
            const double dMt = t0 * Mu + t1 * Mv, dMp = p0 * Mu + p1 * Mv;
            y[6] = y[7] = y[8] = 0.0; y[12] = y[13] = y[14] = 0.0;
            y[9]  = t0 * iM - n0 * iM2 * dMt; y[10] = t1 * iM - n1 * iM2 * dMt; y[11] = t2 * iM - n2 * iM2 * dMt;
            y[15] = p0 * iM - n0 * iM2 * dMp; y[16] = p1 * iM - n1 * iM2 * dMp; y[17] =         - n2 * iM2 * dMp;
        }
        // the reference resets its spline cursors here (:130-134): the first look-up is a cold search
        cur.ka = ms_find_cold(G.ax0, G.n0, clampd(y[0], G.amin, G.amax));
        cur.kb = ms_find_cold(G.ax1, G.n1, clampd(y[1], G.bmin, G.bmax));
        cur.kz = ms_find_cold(G.axz, G.nz, clampd(y[2], G.zmin, G.zmax));
    }

    GEOAC_HD static double step_size(const LaunchConsts& L, const double* y) { return step_size_z(L, y[2] - L.z_grnd); }       // 3DRngDep.cpp:206-213

    // GeoAc_UpdateSources + GeoAc_EvalSrcEq, 3DRngDep.cpp:218-393
    GEOAC_HD static double rhs(const LaunchConsts&, const Grid3D& G, const RayC&, const double* p, double* f, Cur3& cur) {
        double (&S)[3][10] = *reinterpret_cast<double (*)[3][10]>(G.scratch);      // per-thread block (shared memory on the device)
        ms_sample_tuv<false, AMP>(G, p[0], p[1], p[2], cur, S);
        const double* Tt = S[0]; const double* U = S[1]; const double* V = S[2];
        const RdSound s = rd_sound(Tt[0]);
        const double dc[3] = { s.hg * Tt[1], s.hg * Tt[2], s.hg * Tt[3] };
        const double nu0 = p[3], nu1 = p[4], nu2 = p[5];
        const double nm2 = nu0 * nu0 + nu1 * nu1 + nu2 * nu2;
        const double inv_nm = g_rsqrt(nm2), nm = nm2 * inv_nm;
        const double cn = s.c * inv_nm;
        const double g0 = cn * nu0 + U[0], g1 = cn * nu1 + V[0], g2 = cn * nu2;
        const double inv_cgm = g_rsqrt(g0 * g0 + g1 * g1 + g2 * g2);
        f[0] = g0; f[1] = g1; f[2] = g2;          // every right-hand side carries 1/|c_g|: returned as the common factor
        double E[3];
#pragma unroll
        for (int n = 0; n < 3; n++) { E[n] = nm * dc[n] + nu0 * U[1 + n] + nu1 * V[1 + n]; f[3 + n] = -E[n]; }
        if (AMP) {
            // symmetric second-derivative index: (n,m) -> slot in the sampler's output
            // 0 f, 1 a, 2 b, 3 z, 4 aa, 5 bb, 6 zz, 7 ab, 8 az, 9 bz
            const int H[3][3] = { { 4, 7, 8 }, { 7, 5, 9 }, { 8, 9, 6 } };
#pragma unroll
            for (int k = 0; k < 2; k++) {
                const double X0 = p[6 + 6 * k], X1 = p[7 + 6 * k], X2 = p[8 + 6 * k];
                const double m0 = p[9 + 6 * k], m1 = p[10 + 6 * k], m2 = p[11 + 6 * k];
                const double dck = X0 * dc[0] + X1 * dc[1] + X2 * dc[2];
                const double duk = X0 * U[1] + X1 * U[2] + X2 * U[3];
                const double dvk = X0 * V[1] + X1 * V[2] + X2 * V[3];
                const double XdT = X0 * Tt[1] + X1 * Tt[2] + X2 * Tt[3];
                const double dnm = (nu0 * m0 + nu1 * m1 + nu2 * m2) * inv_nm;
                const double q = inv_nm * (dck - cn * dnm);
                const double d0 = nu0 * q + cn * m0 + duk, d1 = nu1 * q + cn * m1 + dvk, d2 = nu2 * q + cn * m2;
                const double gg = (g0 * d0 + g1 * d1 + g2 * d2) * inv_cgm * inv_cgm;
                f[6 + 6 * k] = d0 - g0 * gg;
                f[7 + 6 * k] = d1 - g1 * gg;
                f[8 + 6 * k] = d2 - g2 * gg;
#pragma unroll
                for (int n = 0; n < 3; n++) {
                    const double ddc = s.hg * (X0 * Tt[H[n][0]] + X1 * Tt[H[n][1]] + X2 * Tt[H[n][2]]) - s.hg2 * Tt[1 + n] * XdT;
                    const double ddu = X0 * U[H[n][0]] + X1 * U[H[n][1]] + X2 * U[H[n][2]];
                    const double ddv = X0 * V[H[n][0]] + X1 * V[H[n][1]] + X2 * V[H[n][2]];
                    f[9 + 6 * k + n] = gg * E[n] - (dnm * dc[n] + nm * ddc + m0 * U[1 + n] + m1 * V[1 + n] + nu0 * ddu + nu1 * ddv);
                }
            }
        }
        return inv_cgm;
    }

    // GeoAc_BreakCheck / GeoAc_GroundCheck, 3DRngDep.cpp:451-472 (box from GeoAc_SetPropRegion)
    GEOAC_HD static bool left_region(const LaunchConsts& L, const RayC&, const double* y) {
        return (y[0] > L.box_max[0]) || (y[0] < L.box_min[0]) || (y[1] > L.box_max[1]) || (y[1] < L.box_min[1]) || (y[2] > L.vert_limit);
    }
    GEOAC_HD static bool below_ground(const LaunchConsts& L, const double* y) { return y[2] < L.z_grnd; }
    GEOAC_HD static double break_margin(const LaunchConsts& L, const RayC&, const double* ya, const double* yb) {
        double m = frac_beyond(ya[2] - L.vert_limit, yb[2] - L.vert_limit, 2.0);
#pragma unroll
        for (int i = 0; i < 2; i++) {
            m = frac_beyond(ya[i] - L.box_max[i], yb[i] - L.box_max[i], m);
            m = frac_beyond(L.box_min[i] - ya[i], L.box_min[i] - yb[i], m);
        }
        return m;
    }

    // one segment of GeoAc_TravelTime + GeoAc_SB_Atten, 3DRngDep.cpp:478-542, 597-635
    GEOAC_HD static void segment(const LaunchConsts& L, const Grid3D& G, const RayC&, const double* ya, const double* yb,
                                 Cur3& cur, double& dtt, double& datt) {
        const double dx = yb[0] - ya[0], dy = yb[1] - ya[1], dz = yb[2] - ya[2];
        const double ds = g_sqrt(fmax(dx * dx + dy * dy + dz * dz, 1e-290));
        const double xm = ya[0] + dx * 0.5, ym = ya[1] + dy * 0.5, zm = ya[2] + dz * 0.5;
        const double n0 = ya[3] + (yb[3] - ya[3]) * 0.5, n1 = ya[4] + (yb[4] - ya[4]) * 0.5, n2 = ya[5] + (yb[5] - ya[5]) * 0.5;
        double w[4], dzs[3];
        ms_wrappers<false, true, false>(G, xm, ym, zm, cur, w, dzs);
        const double gT = kGamR * w[0];
        const double inv_c = g_rsqrt(gT), c = gT * inv_c;
        const double cn = c * g_rsqrt(n0 * n0 + n1 * n1 + n2 * n2);
        const double c0 = cn * n0 + w[1], c1 = cn * n1 + w[2], c2 = cn * n2;
        dtt = ds * g_rsqrt(c0 * c0 + c1 * c1 + c2 * c2);
        datt = suthbass_alpha(L, L.sb, zm, c, inv_c, w[3]) * ds;
    }

    // GeoAc_ApproximateIntercept + GeoAc_SetReflectionConditions, 3DRngDep.cpp:142-201
    GEOAC_HD static void reflect(const LaunchConsts& L, const Grid3D& G, const RayC&, const double* ym2, const double* ym1,
                                 const double* yk, double* y0, Cur3& cur) {
        const double dz_k = yk[2] - ym1[2], dz_g = ym1[2] - L.z_grnd;
        const double a1 = dz_g / dz_k, a2 = 0.5 * a1 * a1;
        double pv[NEQ];
#pragma unroll
        for (int i = 0; i < NEQ; i++) pv[i] = ym1[i] + (ym1[i] - yk[i]) * a1 + (yk[i] + ym2[i] - 2.0 * ym1[i]) * a2;
        double w[4], dzs[3];
        ms_wrappers<false, false, true>(G, pv[0], pv[1], L.z_grnd, cur, w, dzs);
        const double cg = sqrt(kGamR * w[0]);
        const double dcg = kGamR / (2.0 * cg) * dzs[0];
        const double dnuz_ds = -1.0 / cg * (L.c_src / cg * dcg + pv[3] * dzs[1] + pv[4] * dzs[2]);
#pragma unroll
        for (int i = 0; i < NEQ; i++) y0[i] = pv[i];
        y0[2] = L.z_grnd;
        y0[5] = -pv[5];
        if (AMP) {
            const double den = 1.0 / (cg / L.c_src * pv[5]);
            y0[8] = -pv[8]; y0[14] = -pv[14];
            y0[11] = -pv[11] + 2.0 * dnuz_ds * pv[8] * den;
            y0[17] = -pv[17] + 2.0 * dnuz_ds * pv[14] * den;
        }
    }

    // GeoAc_Jacobian, 3DRngDep.cpp:547-565
    GEOAC_HD static double jacobian(const LaunchConsts&, const Grid3D& G, const RayC&, const double* yk, Cur3& cur) {
        if (!AMP) return 0.0;
        double w[4], dzs[3];
        ms_wrappers<false, false, false>(G, yk[0], yk[1], yk[2], cur, w, dzs);
        const double c = sqrt(kGamR * w[0]), u = w[1], v = w[2];
        const double nu0 = yk[3], nu1 = yk[4], nu2 = yk[5];
        const double nm = sqrt(nu0 * nu0 + nu1 * nu1 + nu2 * nu2);
        const double q0 = c * nu0 / nm + u, q1 = c * nu1 / nm + v, q2 = c * nu2 / nm;
        const double qm = sqrt(q0 * q0 + q1 * q1 + q2 * q2);
        const double xs = q0 / qm, ys = q1 / qm, zs = q2 / qm;
        return xs * (yk[7] * yk[14] - yk[13] * yk[8]) - yk[6] * (ys * yk[14] - zs * yk[13]) + yk[12] * (ys * yk[8] - zs * yk[7]);
    }

    // GeoAc_Amplitude at an arbitrary state (3DRngDep.cpp:547-592; also evaluated along the path for the raypath rows)
    GEOAC_HD static double amplitude(const LaunchConsts& L, const Grid3D& G, const RayC& rc, const double* yk, Cur3& cur) {
        if (!AMP) return 0.0;
        double w[4], dzs[3];
        ms_wrappers<false, true, false>(G, yk[0], yk[1], yk[2], cur, w, dzs);
        const double c = sqrt(kGamR * w[0]), u = w[1], v = w[2], rho = w[3];
        const double nu0 = yk[3], nu1 = yk[4], nu2 = yk[5];
        const double c0 = L.c_src, u0 = L.u_src, v0 = L.v_src;
        double D;
        {
            const double nm = sqrt(nu0 * nu0 + nu1 * nu1 + nu2 * nu2);
            const double q0 = c * nu0 / nm + u, q1 = c * nu1 / nm + v, q2 = c * nu2 / nm;
            const double qm = sqrt(q0 * q0 + q1 * q1 + q2 * q2);
            const double xs = q0 / qm, ys = q1 / qm, zs = q2 / qm;
            D = xs * (yk[7] * yk[14] - yk[13] * yk[8]) - yk[6] * (ys * yk[14] - zs * yk[13]) + yk[12] * (ys * yk[8] - zs * yk[7]);
        }
        const double nu_mag = (c0 - nu0 * u - nu1 * v) / c;
        const double nu_mag0 = 1.0 - nu0 * u0 / c0 - nu1 * v0 / c0;
        const double cp0 = c * nu0 / nu_mag + u, cp1 = c * nu1 / nu_mag + v, cp2 = c * nu2 / nu_mag;
        const double cs0 = c0 * rc.cth * rc.cph + u0, cs1 = c0 * rc.cth * rc.sph + v0, cs2 = c0 * rc.sth;
        const double cpm = sqrt(cp0 * cp0 + cp1 * cp1 + cp2 * cp2), csm = sqrt(cs0 * cs0 + cs1 * cs1 + cs2 * cs2);
        const double num = rho * nu_mag * (c * c * c) * csm * rc.cth;
        const double den = L.rho_src * nu_mag0 * (c0 * c0 * c0) * cpm * D;
        return 1.0 / (4.0 * kPi) * sqrt(fabs(num / den));
    }

    // GeoAc_Jacobian + GeoAc_Amplitude (3DRngDep.cpp:547-592) and the results row of GeoAc3D.RngDep_main.cpp:296-318
    GEOAC_HD static void arrival(const LaunchConsts& L, const Grid3D& G, const RayC& rc, const double* ym1, const double* yk,
                                 double tt, Cur3& cur, double& amp, double& incl, double& backaz, double& aux, double& margin) {
        (void)tt;
        double w[4], dzs[3];
        ms_wrappers<false, false, false>(G, yk[0], yk[1], L.z_grnd, cur, w, dzs);
        incl = -asin(sqrt(kGamR * w[0]) / L.c_src * yk[5]) * 180.0 / kPi;
        double b = 90.0 - atan2(-yk[4], -yk[3]) * 180.0 / kPi;
        while (b < -180.0) b += 360.0;
        while (b > 180.0) b -= 360.0;
        backaz = b; aux = 0.0;
        margin = (yk[2] - L.z_grnd) / fabs(yk[2] - ym1[2]);
        amp = amplitude(L, G, rc, yk, cur);
    }
};

// ======================================================= spherical, range dependent ===========================
// grid axes: ax0 = latitude, ax1 = longitude, vertical = r.  Sampler output slots (0 f, 1 a, 2 b, 3 z, 4 aa, 5 bb, 6 zz,
// 7 ab, 8 az, 9 bz) in coordinate order (r, lat, lon): first derivatives {3, 1, 2}; second derivatives below.
template <bool AMP>
struct EqGlobalRD {
    using Scout = EqGlobalRD<false>;           // amplitude-free set used by the cost scout (trace_kernel.cuh)
    static constexpr int NEQ = AMP ? 18 : 6;
    using Atmo = Grid3D;
    using Cursor = Cur3;
    static constexpr int VARIANT = GEOAC_GLOBAL_RNGDEP;

    struct RayC { double sth, cth, sph, cph, nu0, cos_lat_src; };

    GEOAC_HD static double altitude(const double* y) { return y[0] - kREarth; }

    // GeoAc_SetInitialConditions, GlobalRngDep.cpp:76-140 (same as Global.cpp; no cursor reset in this file)
    GEOAC_HD static void init(const LaunchConsts& L, const Grid3D& G, double theta, double phi, RayC& rc, double* y, Cur3& cur) {
        sincos(theta, &rc.sth, &rc.cth); sincos(phi, &rc.sph, &rc.cph);
        const double inv_c0 = 1.0 / L.c_src;
        const double Mv = L.v_src * inv_c0, Mu = L.u_src * inv_c0;
        const double n0 = rc.sth, n1 = rc.cth * rc.sph, n2 = rc.cth * rc.cph;
        const double t0 = rc.cth, t1 = -rc.sth * rc.sph, t2 = -rc.sth * rc.cph;
        const double p1 = rc.cth * rc.cph, p2 = -rc.cth * rc.sph;
        const double MS = 1.0 + (n1 * Mv + n2 * Mu);
        const double iM = 1.0 / MS, iM2 = iM * iM;
        rc.nu0 = iM;
        rc.cos_lat_src = cos(L.src[1]);
        y[0] = L.src[0] + kREarth; y[1] = L.src[1]; y[2] = L.src[2];
        y[3] = n0 * iM; y[4] = n1 * iM; y[5] = n2 * iM;
        if (AMP) {
            const double dMt = t1 * Mv + t2 * Mu, dMp = p1 * Mv + p2 * Mu;
            y[6] = y[7] = y[8] = 0.0; y[12] = y[13] = y[14] = 0.0;
            y[9]  = t0 * iM - n0 * iM2 * dMt; y[10] = t1 * iM - n1 * iM2 * dMt; y[11] = t2 * iM - n2 * iM2 * dMt;
            y[15] =         - n0 * iM2 * dMp; y[16] = p1 * iM - n1 * iM2 * dMp; y[17] = p2 * iM - n2 * iM2 * dMp;
        }
        cur.ka = ms_find_cold(G.ax0, G.n0, clampd(y[1], G.amin, G.amax));
        cur.kb = ms_find_cold(G.ax1, G.n1, clampd(y[2], G.bmin, G.bmax));
        cur.kz = ms_find_cold(G.axz, G.nz, clampd(y[0], G.zmin, G.zmax));
    }

    GEOAC_HD static double step_size(const LaunchConsts& L, const double* y) { return step_size_z(L, y[0] - L.ground); }       // GlobalRngDep.cpp:214-221

    // GeoAc_UpdateSources + GeoAc_EvalSrcEq, GlobalRngDep.cpp:226-460
    GEOAC_HD static double rhs(const LaunchConsts&, const Grid3D& G, const RayC&, const double* p, double* f, Cur3& cur) {
        double (&S)[3][10] = *reinterpret_cast<double (*)[3][10]>(G.scratch);      // per-thread block (shared memory on the device)
        ms_sample_tuv<true, AMP>(G, p[1], p[2], p[0], cur, S);
        const double* Tt = S[0]; const double* U = S[1]; const double* V = S[2];
        const int D1[3] = { 3, 1, 2 };                                   // d/dr, d/dlat, d/dlon
        const RdSound s = rd_sound(Tt[0]);
        const double u = U[0], v = V[0];
        double dc[3], du[3], dv[3];
#pragma unroll
        for (int n = 0; n < 3; n++) { dc[n] = s.hg * Tt[D1[n]]; du[n] = U[D1[n]]; dv[n] = V[D1[n]]; }
        const double r = p[0];
        const double nu0 = p[3], nu1 = p[4], nu2 = p[5];
        const double nm2 = nu0 * nu0 + nu1 * nu1 + nu2 * nu2;
        const double inv_nm = g_rsqrt(nm2), nm = nm2 * inv_nm;
        const double cn = s.c * inv_nm;
        const double g0 = cn * nu0, g1 = cn * nu1 + v, g2 = cn * nu2 + u;
        const double inv_cgm = g_rsqrt(g0 * g0 + g1 * g1 + g2 * g2);
        double st, ct; g_sincos(p[1], &st, &ct);
        const double inv_r = g_rcp(r), inv_ct = g_rcp(ct), tant = st * inv_ct;
        const double GC[3] = { 1.0, inv_r, inv_r * inv_ct };
        const double nug = nu1 * g1 + nu2 * g2;
        const double A = nu0 * ct + nu1 * st;
        const double B = nu1 * u - nu2 * v;
        const double GT[3] = { inv_r * nug, nu0 * v - nu0 * g1 + nu2 * g2 * tant, nu0 * u * ct + B * st - g2 * A };
        f[0] = g0; f[1] = GC[1] * g1; f[2] = GC[2] * g2;     // every right-hand side carries 1/|c_g|: returned as the common factor
        double E[3];
#pragma unroll
        for (int n = 0; n < 3; n++) { E[n] = nm * dc[n] + nu1 * dv[n] + nu2 * du[n]; f[3 + n] = -GC[n] * (E[n] + GT[n]); }
        if (AMP) {
            // second derivatives in (r, lat, lon) order from the sampler's (a = lat, b = lon, z = r) slots
            const int H[3][3] = { { 6, 8, 9 }, { 8, 4, 7 }, { 9, 7, 5 } };
            const double inv_r2 = inv_r * inv_r, inv_ct2 = inv_ct * inv_ct;
#pragma unroll
            for (int k = 0; k < 2; k++) {
                const double R0 = p[6 + 6 * k], R1 = p[7 + 6 * k], R2 = p[8 + 6 * k];
                const double m0 = p[9 + 6 * k], m1 = p[10 + 6 * k], m2 = p[11 + 6 * k];
                const double dck = R0 * dc[0] + R1 * dc[1] + R2 * dc[2];
                const double duk = R0 * du[0] + R1 * du[1] + R2 * du[2];
                const double dvk = R0 * dv[0] + R1 * dv[1] + R2 * dv[2];
                const double RdT = R0 * Tt[D1[0]] + R1 * Tt[D1[1]] + R2 * Tt[D1[2]];
                const double dnm = (nu0 * m0 + nu1 * m1 + nu2 * m2) * inv_nm;
                const double q = inv_nm * (dck - cn * dnm);
                const double d0 = nu0 * q + cn * m0, d1 = nu1 * q + cn * m1 + dvk, d2 = nu2 * q + cn * m2 + duk;
                const double gg = (g0 * d0 + g1 * d1 + g2 * d2) * inv_cgm * inv_cgm;
                const double dGC[3] = { 0.0, -R0 * inv_r2, -R0 * inv_r2 * inv_ct + st * R1 * inv_r * inv_ct2 };
                const double dGT[3] = {
                    dGC[1] * nug + inv_r * (m1 * g1 + nu1 * d1 + m2 * g2 + nu2 * d2),
                    m0 * v + nu0 * dvk - m0 * g1 - nu0 * d1 + (m2 * g2 + nu2 * d2) * tant + nu2 * g2 * R1 * inv_ct2,
                    (m0 * u + nu0 * duk) * ct - nu0 * u * R1 * st + (m1 * u + nu1 * duk - m2 * v - nu2 * dvk) * st + B * R1 * ct
                        - d2 * A - g2 * (m0 * ct - nu0 * R1 * st + m1 * st + nu1 * R1 * ct) };
                f[6 + 6 * k] = d0 - g0 * gg;
                f[7 + 6 * k] = dGC[1] * g1 + GC[1] * (d1 - g1 * gg);
                f[8 + 6 * k] = dGC[2] * g2 + GC[2] * (d2 - g2 * gg);
#pragma unroll
                for (int n = 0; n < 3; n++) {
                    const double ddc = s.hg * (R0 * Tt[H[n][0]] + R1 * Tt[H[n][1]] + R2 * Tt[H[n][2]]) - s.hg2 * Tt[D1[n]] * RdT;
                    const double ddu = R0 * U[H[n][0]] + R1 * U[H[n][1]] + R2 * U[H[n][2]];
                    const double ddv = R0 * V[H[n][0]] + R1 * V[H[n][1]] + R2 * V[H[n][2]];
                    // the second term carries E without GeoTerms, like the reference (GlobalRngDep.cpp EvalSrcEq)
                    f[9 + 6 * k + n] = GC[n] * gg * E[n] - dGC[n] * (E[n] + GT[n])
                                   - GC[n] * (dnm * dc[n] + nm * ddc + m1 * dv[n] + m2 * du[n] + nu1 * ddv + nu2 * ddu + dGT[n]);
                }
            }
        }
        return inv_cgm;
    }

    // GeoAc_BreakCheck, GlobalRngDep.cpp:523-535 (altitude + lat/lon box); GroundCheck :537-545
    GEOAC_HD static bool left_region(const LaunchConsts& L, const RayC&, const double* y) {
        return (y[0] > L.vert_limit) || (y[1] < L.box_min[0]) || (y[1] > L.box_max[0]) || (y[2] < L.box_min[1]) || (y[2] > L.box_max[1]);
    }
    GEOAC_HD static bool below_ground(const LaunchConsts& L, const double* y) { return y[0] < L.ground; }
    GEOAC_HD static double break_margin(const LaunchConsts& L, const RayC&, const double* ya, const double* yb) {
        double m = frac_beyond(ya[0] - L.vert_limit, yb[0] - L.vert_limit, 2.0);
#pragma unroll
        for (int i = 0; i < 2; i++) {
            m = frac_beyond(ya[1 + i] - L.box_max[i], yb[1 + i] - L.box_max[i], m);
            m = frac_beyond(L.box_min[i] - ya[1 + i], L.box_min[i] - yb[1 + i], m);
        }
        return m;
    }

    // one segment of GeoAc_TravelTime + GeoAc_SB_Atten (same arithmetic as Global.cpp:527-589, 634-670).  The absorption
    // model's reference state is sampled at (r = z_grnd -> lowest level, lat, lon) of the query point (App. A-14).
    GEOAC_HD static void segment(const LaunchConsts& L, const Grid3D& G, const RayC&, const double* ya, const double* yb,
                                 Cur3& cur, double& dtt, double& datt) {
        const double dr = yb[0] - ya[0], dt = yb[1] - ya[1], dp = yb[2] - ya[2];
        const double rm = ya[0] + dr * 0.5, tm = ya[1] + dt * 0.5, pm = ya[2] + dp * 0.5;
        double st, ct; g_sincos(tm, &st, &ct);
        const double a = rm * dt, bc = rm * ct * dp, bs = rm * st * dp;
        const double ds_tt = g_sqrt(fmax(dr * dr + a * a + bc * bc, 1e-290)), ds_sb = g_sqrt(fmax(dr * dr + a * a + bs * bs, 1e-290));
        const double n0 = ya[3] + (yb[3] - ya[3]) * 0.5, n1 = ya[4] + (yb[4] - ya[4]) * 0.5, n2 = ya[5] + (yb[5] - ya[5]) * 0.5;
        double w[4], wr[4], dzs[3];
        ms_wrappers<true, true, false>(G, tm, pm, rm, cur, w, dzs);
        const double gT = kGamR * w[0];
        const double inv_c = g_rsqrt(gT), c = gT * inv_c;
        const double cn = c * g_rsqrt(n0 * n0 + n1 * n1 + n2 * n2);
        const double c0 = cn * n0, c1 = cn * n1 + w[2], c2 = cn * n2 + w[1];
        dtt = ds_tt * g_rsqrt(c0 * c0 + c1 * c1 + c2 * c2);
        {   // reference state at the lowest levels under the query point: the vertical search starts from the bottom cell
            const int kz_ray = cur.kz;
            cur.kz = 0;
            ms_wrappers<true, true, false, true>(G, tm, pm, L.z_grnd, cur, wr, dzs);
            cur.kz = kz_ray;
        }
        SBRef ref; suthbass_ref(ref, sqrt(kGamR * wr[0]), wr[3]);
        datt = suthbass_alpha(L, ref, rm - kREarth, c, inv_c, w[3]) * ds_sb;
    }

    // first-order intercept + reflection, GlobalRngDep.cpp:144-209 (same as Global.cpp:140-205)
    GEOAC_HD static void reflect(const LaunchConsts& L, const Grid3D& G, const RayC&, const double*, const double* ym1,
                                 const double* yk, double* y0, Cur3& cur) {
        const double a1 = (ym1[0] - L.ground) / (yk[0] - ym1[0]);
        double pv[NEQ];
#pragma unroll
        for (int i = 0; i < NEQ; i++) pv[i] = ym1[i] + (ym1[i] - yk[i]) * a1;
        double w[4], dzs[3];
        ms_wrappers<true, false, true>(G, pv[1], pv[2], pv[0], cur, w, dzs);
        const double c = sqrt(kGamR * w[0]), dc = kGamR / (2.0 * c) * dzs[0];
        const double dnu_r_ds = -1.0 / c * (L.c_src / c * dc + pv[4] * dzs[2] + pv[5] * dzs[1] + c / pv[0] * (pv[4] * pv[4] + pv[5] * pv[5]));
#pragma unroll
        for (int i = 0; i < NEQ; i++) y0[i] = pv[i];
        y0[0] = L.ground;
        y0[3] = -pv[3];
        if (AMP) {
            const double den = 1.0 / (c / L.c_src * pv[3]);
            y0[6] = -pv[6]; y0[12] = -pv[12];
            y0[9]  = -pv[9]  + 2.0 * dnu_r_ds * pv[6] * den;
            y0[15] = -pv[15] + 2.0 * dnu_r_ds * pv[12] * den;
        }
    }

    // GeoAc_Jacobian (as Global.cpp:594-608)
    GEOAC_HD static double jacobian(const LaunchConsts&, const Grid3D& G, const RayC&, const double* yk, Cur3& cur) {
        if (!AMP) return 0.0;
        double w[4], dzs[3];
        ms_wrappers<true, false, false>(G, yk[1], yk[2], yk[0], cur, w, dzs);
        const double c = sqrt(kGamR * w[0]), u = w[1], v = w[2];
        const double r = yk[0], nu0 = yk[3], nu1 = yk[4], nu2 = yk[5];
        double sl, cl; sincos(yk[1], &sl, &cl);
        const double nm = sqrt(nu0 * nu0 + nu1 * nu1 + nu2 * nu2);
        const double q0 = c * nu0 / nm, q1 = c * nu1 / nm + v, q2 = c * nu2 / nm + u;
        const double qm = sqrt(q0 * q0 + q1 * q1 + q2 * q2);
        const double dr_ds = q0 / qm, dt_ds = 1.0 / r * q1 / qm, dp_ds = 1.0 / (r * sl) * q2 / qm;
        return r * r * cl * (dr_ds * (yk[7] * yk[14] - yk[13] * yk[8]) - yk[6] * (dt_ds * yk[14] - dp_ds * yk[13])
                             + yk[12] * (dt_ds * yk[8] - dp_ds * yk[7]));
    }

    // GeoAc_Amplitude at an arbitrary state (as Global.cpp:594-629; also evaluated along the path for the raypath rows)
    GEOAC_HD static double amplitude(const LaunchConsts& L, const Grid3D& G, const RayC& rc, const double* yk, Cur3& cur) {
        if (!AMP) return 0.0;
        double w[4], dzs[3];
        ms_wrappers<true, true, false>(G, yk[1], yk[2], yk[0], cur, w, dzs);
        const double c = sqrt(kGamR * w[0]);
        const double u = w[1], v = w[2], rho = w[3];
        const double r = yk[0];
        const double nu0 = yk[3], nu1 = yk[4], nu2 = yk[5];
        double sl, cl; sincos(yk[1], &sl, &cl);
        const double nm = sqrt(nu0 * nu0 + nu1 * nu1 + nu2 * nu2);
        const double q0 = c * nu0 / nm, q1 = c * nu1 / nm + v, q2 = c * nu2 / nm + u;
        const double qm = sqrt(q0 * q0 + q1 * q1 + q2 * q2);
        const double dr_ds = q0 / qm, dt_ds = 1.0 / r * q1 / qm, dp_ds = 1.0 / (r * sl) * q2 / qm;
        const double D = r * r * cl * (dr_ds * (yk[7] * yk[14] - yk[13] * yk[8]) - yk[6] * (dt_ds * yk[14] - dp_ds * yk[13])
                                       + yk[12] * (dt_ds * yk[8] - dp_ds * yk[7]));
        const double c0 = L.c_src;
        const double nu_mag = (c0 - nu1 * v - nu2 * u) / c, nu_mag0 = rc.nu0;
        const double cp0 = c * nu0 / nu_mag, cp1 = c * nu1 / nu_mag + v, cp2 = c * nu2 / nu_mag + u;
        const double cs0 = c0 * rc.sth / nu_mag0, cs1 = c0 * rc.cth * rc.sph / nu_mag + L.v_src, cs2 = c0 * rc.cth * rc.cph / nu_mag + L.u_src;
        const double cpm = sqrt(cp0 * cp0 + cp1 * cp1 + cp2 * cp2), csm = sqrt(cs0 * cs0 + cs1 * cs1 + cs2 * cs2);
        const double num = rho * nu_mag * (c * c * c) * csm * rc.cth;
        const double den = L.rho_src * nu_mag0 * (c0 * c0 * c0) * cpm * D;
        return 1.0 / (4.0 * kPi) * sqrt(fabs(num / den));
    }

    // Jacobian / amplitude (as Global.cpp:594-629) and the results row of GeoAcGlobal.RngDep_main.cpp:304-328 (+asin: App. A-16)
    GEOAC_HD static void arrival(const LaunchConsts& L, const Grid3D& G, const RayC& rc, const double* ym1, const double* yk,
                                 double tt, Cur3& cur, double& amp, double& incl, double& backaz, double& aux, double& margin) {
        double w[4], dzs[3];
        ms_wrappers<true, true, false>(G, yk[1], yk[2], yk[0], cur, w, dzs);
        const double c = sqrt(kGamR * w[0]);
        incl = asin(c / L.c_src * yk[3]) * 180.0 / kPi;
        double b = 90.0 - atan2(-yk[4], -yk[5]) * 180.0 / kPi;
        if (b < -180.0) b += 360.0;
        if (b > 180.0) b -= 360.0;
        backaz = b;
        const double s1 = sin((yk[1] - L.src[1]) / 2.0), s2 = sin((yk[2] - L.src[2]) / 2.0);
        const double h = s1 * s1 + rc.cos_lat_src * cos(yk[1]) * (s2 * s2);
        aux = 2.0 * kREarth * asin(sqrt(h)) / tt;
        margin = (yk[0] - L.ground) / fabs(yk[0] - ym1[0]);
        amp = amplitude(L, G, rc, yk, cur);
    }
};

// Per-launch invariants of the range-dependent variants: atmosphere at the source, Sutherland-Bass reference state at
// (0, 0, z_grnd) (Cartesian, Absorption.cpp:33-34).  Evaluated with the wrappers' arithmetic from cold cursors.
GEOAC_HD void fill_launch_consts_3d(LaunchConsts& L, const Grid3D& G, int variant) {
    const bool glob = (variant == GEOAC_GLOBAL_RNGDEP);
    L.ground = glob ? kREarth + L.z_grnd : L.z_grnd;
    double w[4], dzs[3];
    Cur3 cur;
    auto cold = [&](double a, double b, double z) {
        cur.ka = ms_find_cold(G.ax0, G.n0, clampd(a, G.amin, G.amax));
        cur.kb = ms_find_cold(G.ax1, G.n1, clampd(b, G.bmin, G.bmax));
        cur.kz = ms_find_cold(G.axz, G.nz, clampd(z, G.zmin, G.zmax));
    };
    if (glob) {
        cold(L.src[1], L.src[2], L.src[0] + kREarth);
        ms_wrappers<true, true, false>(G, L.src[1], L.src[2], L.src[0] + kREarth, cur, w, dzs);
    } else {
        cold(L.src[0], L.src[1], L.src[2]);
        ms_wrappers<false, true, false>(G, L.src[0], L.src[1], L.src[2], cur, w, dzs);
    }
    L.c_src = sqrt(kGamR * w[0]); L.u_src = w[1]; L.v_src = w[2]; L.rho_src = w[3];
    L.c_000 = 0.0; L.c_gnd = 0.0; L.rho_gnd = 0.0; L.dc_gnd = L.du_gnd = L.dv_gnd = 0.0;
    if (!glob) {
        cold(0.0, 0.0, L.z_grnd);
        ms_wrappers<false, true, false>(G, 0.0, 0.0, L.z_grnd, cur, w, dzs);
        suthbass_setup(L, sqrt(kGamR * w[0]), w[3]);
    } else {
        L.sb.invTo = L.sb.cbrtTo = L.sb.visc_num = L.sb.inv_visc_num = L.sb.invPo = 0.0;     // per step (see EqGlobalRD::segment)
        suthbass_tables(L);
    }
}

}  // namespace geoac
