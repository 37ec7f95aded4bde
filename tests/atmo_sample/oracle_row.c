/* tests/atmo_sample/oracle_row.c -- TEST INFRASTRUCTURE: one row of geoac_sample_atmosphere (GEOAC_ATM_NF doubles,
 * include/geoac_b200.h) from the CPU oracle (oracle/liboracle.so, linked, not modified), as the reference's callers would
 * form it from a cold start: c, u, v, rho, c_diff / u_diff / v_diff along the vertical, SuthBass_Alpha, and f, d0, d1, d2,
 * d00, d11, d22, d01, d02, d12 of T, u, v (Eval_Spline_AllOrder2 on the grids; the vertical spline's f, f', f'' for
 * stratified atmospheres).  Built with the oracle's flags (-ffp-contract=off). */
#include <math.h>
#include "../../oracle/geoac_oracle.h"

/* exported by oracle/orc_mspline.c: outputs in the variant's coordinate order */
void orc_mspline_allorder2(orc_atmo* at, int field, double q0, double q1, double q2, double* f, double dout[3], double ddout[3][3]);

/* medium parameters orc_suthbass_alpha reads (the mains' z_grnd= and abs_coeff=) */
void orc_row_set_medium(orc_atmo* a, double z_grnd, double tweak_abs) { a->z_grnd = z_grnd; a->tweak_abs = tweak_abs; }

/* Every spline cursor back to 0.  The 1-D cursors are fields of the atmosphere.  A grid keeps one cursor per field and axis
 * inside the oracle; a look-up at the lowest corner (every coordinate clamps to the first knot) ends in interval 0 on every
 * axis from any cursor (Find_Segment: the cursor's interval, then its neighbours, then the scan, which hits interval 0
 * first), so one look-up per field resets them -- RHO's included. */
static void reset_cursors(orc_atmo* a) {
    if (a->kind < 2) { a->T.accel = 0; a->U.accel = 0; a->V.accel = 0; a->RHO.accel = 0; return; }
    const double lo = -1e300;
    (void)a->c(a, lo, lo, lo); (void)a->u(a, lo, lo, lo); (void)a->v(a, lo, lo, lo); (void)a->rho(a, lo, lo, lo);
}

void orc_row_sample(orc_atmo* a, double p0, double p1, double p2, double freq, double* out) {
    const int vi = a->vert_index;
    reset_cursors(a);
    out[GEOAC_ATM_C] = a->c(a, p0, p1, p2); out[GEOAC_ATM_U] = a->u(a, p0, p1, p2);
    out[GEOAC_ATM_V] = a->v(a, p0, p1, p2); out[GEOAC_ATM_RHO] = a->rho(a, p0, p1, p2);
    out[GEOAC_ATM_DC] = a->c_diff(a, p0, p1, p2, vi); out[GEOAC_ATM_DU] = a->u_diff(a, p0, p1, p2, vi);
    out[GEOAC_ATM_DV] = a->v_diff(a, p0, p1, p2, vi);
    for (int F = 0; F < 3; F++) {
        double* blk = out + GEOAC_ATM_T + 10 * F;
        for (int i = 0; i < 10; i++) blk[i] = 0.0;
        if (a->kind < 2) {
            orc_spline1d* s = F == 0 ? &a->T : (F == 1 ? &a->U : &a->V);
            double e = vi == 2 ? p2 : p0;                       /* clamp exactly as the oracle's 1-D wrappers do */
            e = fmax(fmin(e, a->vmax), a->vmin);
            blk[0] = orc_spline1d_f(e, s); blk[1 + vi] = orc_spline1d_df(e, s); blk[4 + vi] = orc_spline1d_ddf(e, s);
        } else {
            double f, d[3], dd[3][3];
            orc_mspline_allorder2(a, F, p0, p1, p2, &f, d, dd);
            blk[0] = f; blk[1] = d[0]; blk[2] = d[1]; blk[3] = d[2];
            blk[4] = dd[0][0]; blk[5] = dd[1][1]; blk[6] = dd[2][2]; blk[7] = dd[0][1]; blk[8] = dd[0][2]; blk[9] = dd[1][2];
        }
    }
    out[GEOAC_ATM_ALPHA] = orc_suthbass_alpha(a, p0, p1, p2, freq);     /* last: its reference-state look-ups move the cursors */
}
