// mspline.cuh -- range-dependent atmosphere sampler for one thread per ray.
//
// What the reference computes (Code/Atmo/G2S_MultiDimSpline3D.cpp:1156-1593, G2S_GlobalMultiDimSpline3D.cpp:1047-1461;
// behavioural spec in SURVEY App. E): natural cubic splines in the vertical at every horizontal node, and per query five
// bicubic Hermite patches whose corner data are centred finite differences of vertical-spline values, each pushed
// through a dense 16x16 matrix -- 148 vertical-spline calls and ~95 k floating-point operations per field triple.
//
// What this file does instead: the Hermite patch with finite-difference corner data is a TENSOR PRODUCT of 1-D
// operators, so every output is a small bilinear form over the 4x4 node block
//     HX(Q) = h00 Q1 + h01 Q2 + dx (h10 r0 (Q2-Q0) + h11 r1 (Q3-Q1))         (1-D Hermite with FD slopes)
//     FX(V,G) = h00 r0 (V2-V0) + h01 r1 (V3-V1) + dx (h10 r0 (G2-G0) + h11 r1 (G3-G1))   (values dV/dx, slopes dG/dx)
// applied along ax0 inside a row and accumulated over the four rows with the matching ax1 weights.  One pass over the
// 16 nodes yields the value, the gradient and the six second derivatives of T, u and v (~4 k flops instead of ~95 k),
// identical to the reference up to rounding.  The reference's formula slips are kept (SURVEY App. A-8, A-9): the
// Cartesian wrappers / d2f/dz2 block scale the ax1 slope data by dx, the Global vertical-derivative columns drop their
// leading term, and Global second derivatives are not divided by the cell size.
//
// Node data layout in HBM (read through L1/L2; a ray stays in one cell for tens of steps):
//     tuv[((i0*n1 + i1)*nz + k)*18 + 6*field + {0: f, 1: df/dz slope, 2: d(df/dax0)/dz slope, 3: d(df/dax1)/dz slope,
//                                              4: df/dax0, 5: df/dax1 (centred node differences, one-sided at the rim)}]
//     rho[((i0*n1 + i1)*nz + k)*2  + {0: f, 1: slope}]
// The node differences are what the reference's Eval_Vert_Spline_dfdx / dfdy recompute from the neighbouring columns on
// every query (G2S_MultiDimSpline3D.cpp:476-562); storing them with the node makes a column self-contained: three
// aligned 16-byte loads per field and level, no neighbour look-ups, and the two levels a column needs are 2 x 144
// contiguous bytes for all three fields.
#pragma once
#include "core.cuh"

namespace geoac {

struct Grid3D {
    const double* tuv;
    const double* rho;
    const double* ax0; const double* ax1; const double* axz;
    int n0, n1, nz;
    double amin, amax, bmin, bmax, zmin, zmax;
    double* scratch;        // per-thread sampler output block (MS_SCRATCH doubles): shared memory on the device
    // cooperative mode (trace_kernel.cuh, straggler acceleration): `nrole` = 4 lanes advance ONE ray together, lane `role`
    // evaluates row `role` of the 4x4 node block; lanes glane0 .. glane0+3 (mask gmask) form the group.  nrole = 1: serial.
    int role, nrole, glane0; unsigned gmask;
};
constexpr int MS_SCRATCH = 30;

// cursor of a ray: cell of the last look-up
struct Cur3 { int ka, kb, kz; };

// Axis tables: one 32-byte record per node index k,
//   { x[k], 1/(x[k+1]-x[k]), 1/(x[k+1]-x[max(k-1,0)]), 1/(x[min(k+2,n-1)]-x[k]) }
// i.e. the coordinate and the three reciprocals a query in cell k needs (cell width, and the spans of the node differences
// centred on nodes k and k+1).  The reference divides by these spans on every query; they depend on the cell only, so the
// host computes them once with the same divisions (host_tables.hpp: build_axis_records) and a query does no division.
constexpr int AX = 4;

constexpr int MS_STRIDE = 18;      // doubles per node and level in `tuv`
constexpr int MS_FIELD = 6;        // doubles per field inside a node record

// Find_Segment from a cold cursor (both reference files): alternate a search from the bottom and from the top, so a point
// exactly on knot m lands in cell m-1 in the lower half of the axis and in cell m in the upper half.
GEOAC_HD int ms_find_cold(const double* x, int n, double xq) {
    for (int i = 0; i < n; i++) {
        if (xq >= x[AX * i] && xq <= x[AX * (i + 1)]) return i;
        if (xq >= x[AX * (n - 2 - i)] && xq < x[AX * (n - 1 - i)]) return n - 2 - i;
    }
    return 0;
}
// warm cursor: stay in the current cell when the point is on one of its knots (the reference's first test)
GEOAC_HD int ms_find_warm(const double* x, int n, double xq, int k) {
    k = (k < 0) ? 0 : ((k > n - 2) ? n - 2 : k);
    while (xq < x[AX * k]) --k;
    while (xq > x[AX * (k + 1)]) ++k;
    return k;
}

struct MsAxis {
    unsigned off[4];                     // element offsets of the 4 slot nodes (k-1, k, k+1, k+2 clamped)
    double r0, r1;                       // 1 / (x[up] - x[dn]) of the finite differences centred on nodes k and k+1
    double d, inv_d, t;                  // cell width, its reciprocal, scaled coordinate
};

GEOAC_HD void ms_axis(MsAxis& A, const double* x, int n, int k, double xq, unsigned stride) {
    const int km = (k - 1 < 0) ? 0 : k - 1, kp = (k + 2 > n - 1) ? n - 1 : k + 2;
    A.off[0] = (unsigned)km * stride; A.off[1] = (unsigned)k * stride; A.off[2] = (unsigned)(k + 1) * stride; A.off[3] = (unsigned)kp * stride;
    const Pair xd = ld_pair(x + AX * k), rr = ld_pair(x + AX * k + 2);     // (x[k], 1/d), (r0, r1)
    A.r0 = rr.a; A.r1 = rr.b;
    A.d = x[AX * (k + 1)] - xd.a;
    A.inv_d = xd.b;
    A.t = (xq - xd.a) * xd.b;
}

// 1-D weights of one axis: Hermite basis at t (and its t-derivative) combined with the corner finite differences
struct MsW {
    double h00, h01, S0, S1;       // value basis; slope basis times the cell width
    double p, q, P, Q;             // h00 r0, h01 r1, S0 r0, S1 r1
    double e00, e01, T0, T1;       // derivatives of the above with respect to t
    double pd, qd, Pd, Qd;
};
GEOAC_HD void ms_weights(MsW& w, const MsAxis& A, double slope_scale) {
    const double t = A.t, u = 1.0 - t;
    w.h00 = (1.0 + 2.0 * t) * u * u; w.h01 = t * t * (3.0 - 2.0 * t);
    w.S0 = slope_scale * (t * u * u); w.S1 = slope_scale * (t * t * (t - 1.0));
    w.e00 = 6.0 * t * (t - 1.0); w.e01 = -w.e00;
    w.T0 = slope_scale * (u * (1.0 - 3.0 * t)); w.T1 = slope_scale * (t * (3.0 * t - 2.0));
    const double r0 = A.r0, r1 = A.r1;
    w.p = w.h00 * r0; w.q = w.h01 * r1; w.P = w.S0 * r0; w.Q = w.S1 * r1;
    w.pd = w.e00 * r0; w.qd = w.e01 * r1; w.Pd = w.T0 * r0; w.Qd = w.T1 * r1;
}
// row operators along one axis (Q0..Q3 = quantity on the four slot nodes)
GEOAC_HD double ms_HX(const MsW& w, double Q0, double Q1, double Q2, double Q3)  { return w.h00 * Q1 + w.h01 * Q2 + w.P * (Q2 - Q0) + w.Q * (Q3 - Q1); }
GEOAC_HD double ms_HXd(const MsW& w, double Q0, double Q1, double Q2, double Q3) { return w.e00 * Q1 + w.e01 * Q2 + w.Pd * (Q2 - Q0) + w.Qd * (Q3 - Q1); }

// vertical position shared by every column of a query.  The vertical Hermite spline is LINEAR in a column's four data
// (f_k, f_k+1, s_k, s_k+1), so its value / first / second derivative at this position are dot products with coefficient
// triples that depend on the position only -- computed once per query, 3 FMAs per column and quantity instead of ~9:
//     V   = f_k + cV1 (f_k+1 - f_k) + cVa s_k + cVb s_k+1          (same polynomial as G2S_MultiDimSpline3D.cpp:476-562)
//     V'  =       cD1 (f_k+1 - f_k) + cDa s_k + cDb s_k+1
//     V'' =       cE1 (f_k+1 - f_k) + cEa s_k + cEb s_k+1
struct MsZ { int kz; double cV1, cVa, cVb, cD1, cDa, cDb, cE1, cEa, cEb, cG1; };
template <bool GLOBAL>
GEOAC_HD void ms_zpos(MsZ& Z, const Grid3D& g, double z, int kz) {
    const Pair zh = ld_pair(g.axz + AX * kz);                            // (z[k], 1/h)
    const double z0 = zh.a, invh = zh.b;
    const double h = g.axz[AX * (kz + 1)] - z0;
    const double X = (z - z0) * invh, omX = 1.0 - X, XomX = X * omX, om2X = 1.0 - 2.0 * X;
    Z.kz = kz;
    Z.cV1 = X - XomX * om2X;            Z.cVa = XomX * omX * h;           Z.cVb = -(XomX * X * h);
    Z.cD1 = (1.0 - om2X * om2X + 2.0 * XomX) * invh;  Z.cDa = om2X * omX - XomX;  Z.cDb = -(om2X * X + XomX);
    const double inv2 = 2.0 * invh * invh;
    Z.cE1 = 3.0 * om2X * inv2;          Z.cEa = (3.0 * X - 2.0) * h * inv2;  Z.cEb = (3.0 * X - 1.0) * h * inv2;
    // vertical derivative of a finite-difference column: the Global file drops the leading (d1 - d0)/h term (App. A-9)
    Z.cG1 = GLOBAL ? Z.cD1 - invh : Z.cD1;
}
GEOAC_HD double ms_v(const MsZ& Z, double f0, double df, double s0, double s1)  { return fma(Z.cV1, df, fma(Z.cVa, s0, fma(Z.cVb, s1, f0))); }
GEOAC_HD double ms_vz(const MsZ& Z, double df, double s0, double s1)            { return fma(Z.cD1, df, fma(Z.cDa, s0, Z.cDb * s1)); }
GEOAC_HD double ms_vzz(const MsZ& Z, double df, double s0, double s1)           { return fma(Z.cE1, df, fma(Z.cEa, s0, Z.cEb * s1)); }
GEOAC_HD double ms_gz(const MsZ& Z, double dd, double s0, double s1)            { return fma(Z.cG1, dd, fma(Z.cDa, s0, Z.cDb * s1)); }

// the six data of one node and level for one field (48 aligned bytes): f, df/dz slope, the vertical slopes of the two
// node differences, and the node differences df/dax0, df/dax1 themselves
struct Node6 { double f, s, sa, sb, da, db; };
GEOAC_HD Node6 ms_ld6(const double* p) {
    const Pair a = ld_pair(p), b = ld_pair(p + 2), c = ld_pair(p + 4);
    Node6 n; n.f = a.a; n.s = a.b; n.sa = b.a; n.sb = b.b; n.da = c.a; n.db = c.b; return n;
}

// ---------------------------------------------------------------------------------------------------------------
// Row-wise accumulation with PINNED arithmetic.  A query sums the contributions of the four ax1 rows of the node block.
// The serial path adds them row after row; the cooperative path has four lanes evaluate one row each and passes the
// accumulator from lane to lane in the same order.  Every operation that combines rows is an explicit fma, so both paths
// produce the same bits whatever the compiler would otherwise contract -- a ray's record does not depend on how many
// lanes worked on it (tests: schedule neutrality, multi-context == single).
// ---------------------------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
GEOAC_HD double p_mul(double a, double b) { return __dmul_rn(a, b); }
GEOAC_HD double p_add(double a, double b) { return __dadd_rn(a, b); }
GEOAC_HD double p_sub(double a, double b) { return __dsub_rn(a, b); }
#else
GEOAC_HD double p_mul(double a, double b) { return a * b; }
GEOAC_HD double p_add(double a, double b) { return a + b; }
GEOAC_HD double p_sub(double a, double b) { return a - b; }
#endif

// ax1 weights of one row (slot jb): tensor weight and its derivative, slope weights, FD-of-values and FD-of-slopes weights
struct MsRowW { double ey, eyd, sy, syd, al, ald, be, bed; };
GEOAC_HD MsRowW ms_row_weights(const MsW& wb, int jb) {
    MsRowW r;
    r.ey  = (jb == 1) ? wb.h00 : ((jb == 2) ? wb.h01 : 0.0);
    r.eyd = (jb == 1) ? wb.e00 : ((jb == 2) ? wb.e01 : 0.0);
    r.sy  = (jb == 1) ? wb.S0 : ((jb == 2) ? wb.S1 : 0.0);
    r.syd = (jb == 1) ? wb.T0 : ((jb == 2) ? wb.T1 : 0.0);
    r.al  = (jb == 0) ? -wb.p  : ((jb == 1) ? -wb.q  : ((jb == 2) ? wb.p  : wb.q));
    r.ald = (jb == 0) ? -wb.pd : ((jb == 1) ? -wb.qd : ((jb == 2) ? wb.pd : wb.qd));
    r.be  = (jb == 0) ? -wb.P  : ((jb == 1) ? -wb.Q  : ((jb == 2) ? wb.P  : wb.Q));
    r.bed = (jb == 0) ? -wb.Pd : ((jb == 1) ? -wb.Qd : ((jb == 2) ? wb.Pd : wb.Qd));
    return r;
}
// a_0 Q1 + a_1 Q2 + b_0 (Q2 - Q0) + b_1 (Q3 - Q1), pinned
GEOAC_HD double p_row4(double a0, double a1, double b0, double b1, double Q0, double Q1, double Q2, double Q3) {
    return fma(b1, p_sub(Q3, Q1), fma(b0, p_sub(Q2, Q0), fma(a1, Q2, p_mul(a0, Q1))));
}
GEOAC_HD double p_row2(double a0, double a1, double Q1, double Q2) { return fma(a1, Q2, p_mul(a0, Q1)); }

// the row-level partial results of one field on one row of four nodes
struct MsRowVals { double Fv, FXv, FGb, EVz, BVz, GXZ, GYZ, FXd, EVzd, BVzd, GXZd, GYZd, EVzz, BVzz; };

template <bool GLOBAL, bool ORDER2>
GEOAC_HD void ms_row_vals(MsRowVals& R, const double* base, const unsigned (&aoff)[4], unsigned boff, const MsZ& Z, const MsW& wa) {
    double V[4], Vz[4], Vzz[4], Ga[4], Gb[4], Gaz[4], Gbz[4];
#pragma unroll
    for (int ia = 0; ia < 4; ia++) {
        const double* n0p = base + (aoff[ia] + boff);
        const Node6 lo = ms_ld6(n0p), hi = ms_ld6(n0p + MS_STRIDE);
        const double df = hi.f - lo.f, dda = hi.da - lo.da, ddb = hi.db - lo.db;
        V[ia] = ms_v(Z, lo.f, df, lo.s, hi.s);
        Vz[ia] = ms_vz(Z, df, lo.s, hi.s);
        if (ORDER2) Vzz[ia] = ms_vzz(Z, df, lo.s, hi.s); else Vzz[ia] = 0.0;
        Ga[ia] = ms_v(Z, lo.da, dda, lo.sa, hi.sa);          // column of the ax0 node difference (Eval_Vert_Spline_dfdx / ddfdxdz)
        Gaz[ia] = ms_gz(Z, dda, lo.sa, hi.sa);
        Gb[ia] = ms_v(Z, lo.db, ddb, lo.sb, hi.sb);          // column of the ax1 node difference
        Gbz[ia] = ms_gz(Z, ddb, lo.sb, hi.sb);
    }
    R.Fv  = p_row4(wa.h00, wa.h01, wa.P, wa.Q, V[0], V[1], V[2], V[3]);
    const double dV0 = p_sub(V[2], V[0]), dV1 = p_sub(V[3], V[1]), dG0 = p_sub(Ga[2], Ga[0]), dG1 = p_sub(Ga[3], Ga[1]);
    R.FXv = fma(wa.Q, dG1, fma(wa.P, dG0, fma(wa.q, dV1, p_mul(wa.p, dV0))));
    R.FGb = p_row4(wa.h00, wa.h01, wa.P, wa.Q, Gb[0], Gb[1], Gb[2], Gb[3]);
    R.EVz = p_row2(wa.h00, wa.h01, Vz[1], Vz[2]);
    R.BVz = fma(wa.Q, p_sub(Vz[3], Vz[1]), p_mul(wa.P, p_sub(Vz[2], Vz[0])));
    R.GXZ = p_row2(wa.S0, wa.S1, Gaz[1], Gaz[2]);            // used only on the corner rows (ey != 0)
    R.GYZ = p_row2(wa.h00, wa.h01, Gbz[1], Gbz[2]);
    if (ORDER2) {
        R.FXd  = fma(wa.Qd, dG1, fma(wa.Pd, dG0, fma(wa.qd, dV1, p_mul(wa.pd, dV0))));
        R.EVzd = p_row2(wa.e00, wa.e01, Vz[1], Vz[2]);
        R.BVzd = fma(wa.Qd, p_sub(Vz[3], Vz[1]), p_mul(wa.Pd, p_sub(Vz[2], Vz[0])));
        R.GXZd = p_row2(wa.T0, wa.T1, Gaz[1], Gaz[2]);
        R.GYZd = p_row2(wa.e00, wa.e01, Gbz[1], Gbz[2]);
        R.EVzz = p_row2(wa.h00, wa.h01, Vzz[1], Vzz[2]);
        R.BVzz = fma(wa.Q, p_sub(Vzz[3], Vzz[1]), p_mul(wa.P, p_sub(Vzz[2], Vzz[0])));
    }
}

// acc += contribution of one row (explicit fma chains on the accumulator: the order of the rows is the order of the calls)
template <bool ORDER2>
GEOAC_HD void ms_row_acc(double (&acc)[10], const MsRowVals& R, const MsRowW& w, double qs) {
    const double wy = p_add(w.ey, w.be), wyd = p_add(w.eyd, w.bed);
    const double EG = p_add(R.EVz, R.GXZ);
    acc[0] = fma(wy, R.Fv, acc[0]);
    acc[1] = fma(wy, R.FXv, acc[1]);
    acc[2] = fma(w.be, R.FGb, fma(w.al, R.Fv, acc[2]));
    acc[3] = fma(w.sy, R.GYZ, fma(w.be, R.BVz, fma(w.ey, EG, acc[3])));
    if (ORDER2) {
        acc[4] = fma(wy, R.FXd, acc[4]);
        acc[5] = fma(w.bed, R.FGb, fma(w.ald, R.Fv, acc[5]));
        // d2f/dz2 block: only its Py data carry the dx-for-dy slip, the Pxy data are scaled by dx*dy
        acc[6] = fma(w.be, R.BVzz, fma(p_mul(w.be, qs), R.EVzz, fma(w.ey, p_add(R.EVzz, R.BVzz), acc[6])));
        acc[7] = fma(wyd, R.FXv, acc[7]);
        acc[8] = fma(w.sy, R.GYZd, fma(w.be, R.BVzd, fma(w.ey, p_add(R.EVzd, R.GXZd), acc[8])));
        acc[9] = fma(w.syd, R.GYZ, fma(w.bed, R.BVz, fma(w.eyd, EG, acc[9])));
    }
}

// cooperative hand-over: every lane of the group takes the accumulator of lane `src` (glane0 + row)
template <int N>
GEOAC_HD void ms_group_take(double (&acc)[N], const Grid3D& g, int row) {
#if defined(__CUDA_ARCH__)
#pragma unroll
    for (int i = 0; i < N; i++) acc[i] = __shfl_sync(g.gmask, acc[i], g.glane0 + row);
#else
    (void)acc; (void)g; (void)row;
#endif
}

// ---------------------------------------------------------------------------------------------------------------
// Eval_Spline_AllOrder1 / AllOrder2 for T, u and v in one pass.  out[field][..] in GRID-axis order:
//   0 f, 1 d/da, 2 d/db, 3 d/dz, 4 d2/da2, 5 d2/db2, 6 d2/dz2, 7 d2/dadb, 8 d2/dadz, 9 d2/dbdz   (a = ax0, b = ax1, z = vertical)
// ---------------------------------------------------------------------------------------------------------------
template <bool GLOBAL, bool ORDER2>
GEOAC_HD void ms_sample_tuv(const Grid3D& g, double a_in, double b_in, double z_in, Cur3& cur, double (&out)[3][10]) {
    const double a = clampd(a_in, g.amin, g.amax), b = clampd(b_in, g.bmin, g.bmax), z = clampd(z_in, g.zmin, g.zmax);
    cur.ka = ms_find_warm(g.ax0, g.n0, a, cur.ka);
    cur.kb = ms_find_warm(g.ax1, g.n1, b, cur.kb);
    cur.kz = ms_find_warm(g.axz, g.nz, z, cur.kz);
    MsAxis A, B; MsZ Z;
    ms_axis(A, g.ax0, g.n0, cur.ka, a, (unsigned)(g.n1 * g.nz * MS_STRIDE));
    ms_axis(B, g.ax1, g.n1, cur.kb, b, (unsigned)(g.nz * MS_STRIDE));
    ms_zpos<GLOBAL>(Z, g, z, cur.kz);
    MsW wa, wb;
    ms_weights(wa, A, A.d);
    ms_weights(wb, B, B.d);
    // d2f/dz2 block: the Cartesian file scales the ax1 slope data by dx (App. A-8); Global uses dp
    const double qs = GLOBAL ? 1.0 : A.d * B.inv_d;
    const unsigned kofs = (unsigned)cur.kz * MS_STRIDE;

    const double ida = A.inv_d, idb = B.inv_d;
#pragma unroll 1
    for (int F = 0; F < 3; F++) {
        double acc[10];
#pragma unroll
        for (int i = 0; i < 10; i++) acc[i] = 0.0;
        const double* base = g.tuv + kofs + MS_FIELD * F;
        if (g.nrole == 1) {
#pragma unroll
            for (int jb = 0; jb < 4; jb++) {
                MsRowVals R;
                ms_row_vals<GLOBAL, ORDER2>(R, base, A.off, B.off[jb], Z, wa);
                ms_row_acc<ORDER2>(acc, R, ms_row_weights(wb, jb), qs);
            }
        } else {                                    // four lanes, one row each; the accumulator travels lane 0 -> 1 -> 2 -> 3 -> all
            const int jb = g.role;
            const unsigned boff = (jb == 0) ? B.off[0] : ((jb == 1) ? B.off[1] : ((jb == 2) ? B.off[2] : B.off[3]));
            MsRowVals R;
            ms_row_vals<GLOBAL, ORDER2>(R, base, A.off, boff, Z, wa);
            const MsRowW w = ms_row_weights(wb, jb);
#pragma unroll 1
            for (int r = 0; r < 4; r++) {
                if (r == jb) ms_row_acc<ORDER2>(acc, R, w, qs);
                ms_group_take<10>(acc, g, r);
            }
        }
        if (ORDER2 && !GLOBAL) {            // Global leaves the second derivatives in scaled units (App. A-9)
            acc[4] = p_mul(acc[4], ida); acc[5] = p_mul(acc[5], idb); acc[7] = p_mul(acc[7], idb); acc[8] = p_mul(acc[8], ida); acc[9] = p_mul(acc[9], idb);
        }
#pragma unroll
        for (int i = 0; i < 10; i++) out[F][i] = acc[i];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The scalar wrappers c(), u(), v(), rho() (Eval_Spline_f: Cartesian scales the ax1 slope data by dx, App. A-8) and the
// vertical derivative wrappers c_diff / u_diff / v_diff (Eval_Spline_df with the same scaling) -- used by travel time,
// absorption, amplitude, reflection and the per-launch invariants.  vals: T, u, v, rho;  dz: dT/dz, du/dz, dv/dz.
// ---------------------------------------------------------------------------------------------------------------
// GROUND (Global.RngDep absorption reference, sampled at the lowest levels every step): only T and rho are evaluated.
template <bool GLOBAL, bool WITH_RHO, bool WITH_DZ, bool GROUND = false>
GEOAC_HD void ms_wrappers(const Grid3D& g, double a_in, double b_in, double z_in, Cur3& cur, double (&vals)[4], double (&dz)[3]) {
    const double a = clampd(a_in, g.amin, g.amax), b = clampd(b_in, g.bmin, g.bmax), z = clampd(z_in, g.zmin, g.zmax);
    cur.ka = ms_find_warm(g.ax0, g.n0, a, cur.ka);
    cur.kb = ms_find_warm(g.ax1, g.n1, b, cur.kb);
    cur.kz = ms_find_warm(g.axz, g.nz, z, cur.kz);
    MsAxis A, B; MsZ Z;
    ms_axis(A, g.ax0, g.n0, cur.ka, a, (unsigned)(g.n1 * g.nz * MS_STRIDE));
    ms_axis(B, g.ax1, g.n1, cur.kb, b, (unsigned)(g.nz * MS_STRIDE));
    ms_zpos<GLOBAL>(Z, g, z, cur.kz);
    MsW wa, wb;
    ms_weights(wa, A, A.d);
    ms_weights(wb, B, GLOBAL ? B.d : A.d);              // the quirk: ax1 slope data times dx
    vals[1] = vals[2] = 0.0;
#pragma unroll 1
    for (int F = 0; F < (WITH_RHO ? 4 : 3); F += (GROUND ? 3 : 1)) {
        const bool is_rho = (F == 3);
        const double* base = is_rho ? g.rho : g.tuv + MS_FIELD * F;
        const int lvl = is_rho ? 2 : MS_STRIDE;          // doubles between vertical levels
        const unsigned ko = (unsigned)cur.kz * (is_rho ? 2u : (unsigned)MS_STRIDE);
        const unsigned shr = is_rho ? (unsigned)(MS_STRIDE / 2) : 1u;   // node offsets were built for the tuv layout: /9 for rho's 2 doubles
        double av[2] = { 0.0, 0.0 };               // value, d/dz
        const double bscale = GLOBAL ? 1.0 : B.d * A.inv_d;
        auto row = [&](int jb, unsigned boff) {
            double V[4], Vz[4], Gaz[4], Gbz[4];
#pragma unroll
            for (int ia = 0; ia < 4; ia++) {
                const unsigned o = (A.off[ia] + boff) / shr;
                const double* n0p = base + ko + o;
                const Pair lo = ld_pair(n0p), hi = ld_pair(n0p + lvl);            // (f, slope) at both levels
                const double df = hi.a - lo.a;
                V[ia] = ms_v(Z, lo.a, df, lo.b, hi.b);
                Vz[ia] = 0.0; Gaz[ia] = 0.0; Gbz[ia] = 0.0;
                if (WITH_DZ && !is_rho) {
                    Vz[ia] = ms_vz(Z, df, lo.b, hi.b);
                    const Pair slo = ld_pair(n0p + 2), shi = ld_pair(n0p + lvl + 2);  // (sa, sb) at both levels
                    const Pair dlo = ld_pair(n0p + 4), dhi = ld_pair(n0p + lvl + 4);  // (da, db) at both levels
                    Gaz[ia] = ms_gz(Z, dhi.a - dlo.a, slo.a, shi.a);
                    Gbz[ia] = ms_gz(Z, dhi.b - dlo.b, slo.b, shi.b);
                }
            }
            const MsRowW w = ms_row_weights(wb, jb);
            // the Pxy block of Eval_Spline_f / _df is scaled by dx*dy, only the Py block by the slipped scale: separate the two
            const double be_true = GLOBAL ? w.be : p_mul(w.be, bscale);
            const double EV = p_row2(wa.h00, wa.h01, V[1], V[2]);
            const double BV = fma(wa.Q, p_sub(V[3], V[1]), p_mul(wa.P, p_sub(V[2], V[0])));
            struct { double EV, BV, EVz, BVz, GXZ, GYZ, ey, be, bt, sy; } r = { EV, BV, 0, 0, 0, 0, w.ey, w.be, be_true, w.sy };
            if (WITH_DZ && !is_rho) {
                r.EVz = p_row2(wa.h00, wa.h01, Vz[1], Vz[2]);
                r.BVz = fma(wa.Q, p_sub(Vz[3], Vz[1]), p_mul(wa.P, p_sub(Vz[2], Vz[0])));
                r.GXZ = p_row2(wa.S0, wa.S1, Gaz[1], Gaz[2]);
                r.GYZ = p_row2(wa.h00, wa.h01, Gbz[1], Gbz[2]);
            }
            return r;
        };
        auto accumulate = [&](const auto& r) {
            av[0] = fma(r.bt, r.BV, fma(r.be, r.EV, fma(r.ey, p_add(r.EV, r.BV), av[0])));
            if (WITH_DZ && !is_rho) av[1] = fma(r.sy, r.GYZ, fma(r.bt, r.BVz, fma(r.ey, p_add(r.EVz, r.GXZ), av[1])));
        };
        if (g.nrole == 1) {
#pragma unroll
            for (int jb = 0; jb < 4; jb++) accumulate(row(jb, B.off[jb]));
        } else {
            const int jb = g.role;
            const unsigned boff = (jb == 0) ? B.off[0] : ((jb == 1) ? B.off[1] : ((jb == 2) ? B.off[2] : B.off[3]));
            const auto r = row(jb, boff);
#pragma unroll 1
            for (int k = 0; k < 4; k++) {
                if (k == jb) accumulate(r);
                ms_group_take<2>(av, g, k);
            }
        }
        const double accv = av[0], accz = av[1];
        vals[F] = accv;
        if (WITH_DZ && !is_rho) dz[F] = accz;
    }
}

}  // namespace geoac
