// eigenray.cu -- batched eigenray search above the C ABI (host code only; every ray goes through geoac_trace_sources on the GPU).
//
// Replaces the body of GeoAc3D_RunEigSearch (Code/GeoAc3D_main.cpp:531-541, Code/GeoAc3D.RngDep_main.cpp likewise) and of
// GeoAcGlobal_RunEigSearch (Code/GeoAcGlobal_main.cpp:573-583, GeoAcGlobal.RngDep_main.cpp likewise; the Global routines
// are Code/GeoAc/GeoAc.Eigenray.Global.cpp:46-136 and :139-320 -- same algorithm on great-circle range and bearing):
//     for every bounce count:  theta_start = theta_min;
//         while theta_start < theta_max:  GeoAc_EstimateEigenray (Code/GeoAc/GeoAc.Eigenray.cpp:30-121)
//                                         on success GeoAc_3DEigenray_LM (:123-335);  theta_start = theta_next
// The reference traces one ray at a time (a 0.25-degree inclination fan per estimate, one ray per Levenberg-Marquardt
// iteration).  Here the two routines are restated literally over a RAY CACHE keyed by the source and the exact launch
// angles: a look-up that misses records a request -- for the fixed-step fans of the estimate, the whole remaining fan --
// and every chain (search, bounce count) not yet complete is replayed from its start once the requests of ALL searches,
// bounce counts and brackets have been traced in ONE geoac_trace_sources batch per calc_amp setting.  A replay only ever
// reads rays the sequential algorithm would have traced at exactly those angles from exactly that source, so the final
// replay of a chain IS the reference's sequence of decisions; batching changes only when rays are computed.  A complete
// chain read only cached rays, so its calls are final and it is not replayed again.
//   * the iteration-0 fan (one azimuth, theta_min..theta_max) is shared by every estimate call and every bounce count of a
//     search: a trace with `bounces = B` yields the arrivals of all bounce counts <= B;
//   * later estimate calls of a chain start from theta_next, which iteration 0 already fixes, so all brackets of a fan
//     refine their azimuth and run their LM iterations concurrently (speculatively: a call that ends on the reference's
//     theta_max_reached quirk cuts the chain, and the final replay honours that);
//   * LM iterations are one ray per live bracket per round (sequentially dependent inside a bracket, as in the reference).
// The one-source entry points (geoac_eigenray_search, geoac_eigenray_direct) are the n_src = 1 case of the same engine.
// `long double` is used exactly where the reference uses it (x87 extended on x86-64).
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <algorithm>
#include <string>
#include <tuple>
#include <unordered_map>
#include <vector>
#include "../../include/geoac_b200.h"

// capi.cu: the context's last error message, and the timing of its last eigenray search (geoac_last_eigenray_ms)
int geoac_fail_msg(geoac_ctx* ctx, int code, const std::string& msg);
void geoac_set_eigenray_ms(geoac_ctx* ctx, const double* ms3);

namespace {

constexpr double Pi = 3.141592653589793238462643;      // Code/GeoAc/GeoAc.Parameters.cpp:28

struct RayKey {
    uint64_t tb, pb; int32_t src, amp;
    bool operator==(const RayKey& o) const { return tb == o.tb && pb == o.pb && src == o.src && amp == o.amp; }
    bool operator<(const RayKey& o) const { return std::tie(amp, src, tb, pb) < std::tie(o.amp, o.src, o.tb, o.pb); }
};
struct RayKeyHash {
    size_t operator()(const RayKey& k) const {
        uint64_t h = k.tb * 0x9E3779B97F4A7C15ull;
        h ^= k.pb + 0x632BE59BD9B4E019ull + (h << 6) + (h >> 2);
        h ^= ((uint64_t)(uint32_t)k.src << 1 | (uint64_t)k.amp) + 0x94D049BB133111EBull + (h << 6) + (h >> 2);
        return (size_t)h;
    }
};
// What the search reads of a traced ray, in the pools of Search: the status of records 0..nb from st_off on and, per record,
// kCols[amp] state columns from x_off on -- the position (0..2) for the calc_amp = 0 fans of the estimate, the 18 state
// columns for the LM rays.
constexpr int kCols[2] = { 3, 18 };
struct RayVal { int nb; int64_t st_off, x_off; };
static uint64_t bits(double x) { uint64_t u; std::memcpy(&u, &x, 8); return u; }

struct Request { double theta, phi; int nb; };

// One source of a search
struct Src {
    double loc[3];                            // Source_Loc: (x, y, z) [km], or (lat, lon) [deg] and z for the Global variants; z clamped
    double trace[3];                          // as geoac_trace_sources takes it (the convention of geoac_params.src)
    double Mx = 0, My = 0;                    // u/c, v/c at the source (stratified LM, Eigenray.cpp:131-135; w = 0)
};

struct Search {
    geoac_ctx* ctx;
    int variant;
    bool strat, glob = false;
    geoac_eig_opts o;
    double z_grnd = 0.0;
    std::vector<Src> srcs;
    std::unordered_map<RayKey, RayVal, RayKeyHash> cache;
    std::vector<int32_t> st_pool;             // the cache's statuses and state columns; only appended to between replays, so
    std::vector<double> x_pool;               // a pointer from lookup() stays valid while the chains are replayed
    std::unordered_map<RayKey, Request, RayKeyHash> want;   // this round's misses (a set: their order changes no result)
    int64_t rays_traced = 0; int rounds = 0;
    double replay_ms = 0.0, kernel_ms = 0.0;

    // state of the ray launched from source si at (GeoAc_theta, GeoAc_phi) [radians, exactly the values the reference
    // assigns] after n_bnc reflections, or nullptr + a recorded request.  *brk receives the reference's BreakCheck (any
    // segment left the region; a step-limit end counts as one, see include/geoac_b200.h).
    const double* lookup(int si, double theta, double phi, int amp, int n_bnc, bool* brk, bool record = true) {
        RayKey k{ bits(theta), bits(phi), si, amp };
        auto it = cache.find(k);
        if (it != cache.end()) {
            const RayVal& v = it->second;
            const int32_t* st = st_pool.data() + v.st_off;
            const double* x = x_pool.data() + v.x_off;
            bool ended = false;
            for (int b = 0; b <= std::min(n_bnc, v.nb); b++) if (st[b] != GEOAC_ST_ARRIVAL) { ended = true; break; }
            if (ended) { *brk = true; return x; }
            if (v.nb >= n_bnc) { *brk = false; return x + (size_t)n_bnc * kCols[amp]; }
        }
        if (record) {
            auto w = want.find(k);
            if (w == want.end()) want.emplace(k, Request{ theta, phi, n_bnc });
            else w->second.nb = std::max(w->second.nb, n_bnc);
        }
        return nullptr;
    }

    // ---- GeoAc_EstimateEigenray, Eigenray.cpp:30-121 ----
    struct Est { bool complete = false, ok = false, next_known = false; double theta_est = 0, phi_est = 0, theta_next = 0; };
    static double modify_d_theta(double dr, double dr_dtheta, double big, double small_, double wf) {   // :23-27; Global :39-43 (width factor 1/2)
        const double width = wf * std::pow(dr_dtheta, 2);
        return big - (big - small_) * std::exp(-dr * dr / width);
    }
    static double bearing(double lat1, double long1, double lat2, double long2) {                 // Calc_Bearing, Eigenray.Global.cpp:25-30
        const double term1 = std::sin((long2 - long1) * Pi / 180.0);
        const double term2 = std::cos(lat1 * Pi / 180.0) * std::tan(lat2 * Pi / 180.0) - std::sin(lat1 * Pi / 180.0) * std::cos((long2 - long1) * Pi / 180.0);
        return std::atan2(term1, term2) * 180.0 / Pi;
    }
    static double gc_distance(double lat1, double long1, double lat2, double long2) {             // Calc_GC_Distance, :32-37
        const double term1 = std::pow(std::sin((lat2 - lat1) * Pi / 180.0 / 2.0), 2);
        const double term2 = std::cos(lat1 * Pi / 180.0) * std::cos(lat2 * Pi / 180.0) * std::pow(std::sin((long2 - long1) * Pi / 180.0 / 2.0), 2);
        return 2.0 * 6370.0 * std::asin(std::sqrt(term1 + term2));
    }
    Est estimate(int si, const double rcv[2], double theta_min, double theta_max, int bounces) {
        Est e;
        const double* src = srcs[si].loc;
        const double r_rcvr = glob ? gc_distance(src[0], src[1], rcv[0], rcv[1])
                                   : std::sqrt(std::pow(rcv[0] - src[0], 2) + std::pow(rcv[1] - src[1], 2));
        double phi = glob ? bearing(src[0], src[1], rcv[0], rcv[1])                       // Global: an azimuth; Cartesian: from the x axis
                          : 180.0 / 3.14159 * std::atan2(rcv[1] - src[1], rcv[0] - src[0]);
        int iterations = 0;
        e.theta_est = theta_max;
        double r, r_prev, d_theta = o.d_theta_big, d_phi = 10.0;
        bool theta_max_reached = false;
        while (std::fabs(d_phi) > o.azimuth_err_lim && iterations < 5) {
            r = r_rcvr; r_prev = r_rcvr;
            const double phi_rad = glob ? (90.0 - phi) * Pi / 180.0 : phi * Pi / 180.0;      // GeoAc_phi
            // Cartesian: theta <= theta_max (Eigenray.cpp:58); Global: theta < theta_max (Eigenray.Global.cpp:74)
            for (double theta = theta_min; glob ? theta < theta_max : theta <= theta_max; theta += d_theta) {
                if (theta + d_theta >= theta_max) theta_max_reached = true;
                bool brk;
                const double* s = lookup(si, theta * Pi / 180.0, phi_rad, 0, bounces, &brk);
                if (!s) {
                    if (iterations < 3) {          // fixed step: the rest of this fan is known now
                        int guard = 0;
                        for (double t = theta + d_theta; (glob ? t < theta_max : t <= theta_max) && guard < 100000; t += d_theta, guard++) { bool b2; lookup(si, t * Pi / 180.0, phi_rad, 0, bounces, &b2); }
                    }
                    return e;                      // incomplete
                }
                if (brk) { r = r_rcvr; r_prev = r_rcvr; }
                else if (glob) r = gc_distance(src[0], src[1], s[1] * 180.0 / Pi, s[2] * 180.0 / Pi);
                else r = std::sqrt(std::pow(s[0] - src[0], 2) + std::pow(s[1] - src[1], 2));
                if ((r - r_rcvr) * (r_prev - r_rcvr) < 0.0) {
                    if (iterations == 0) { e.theta_next = theta; e.next_known = true; }
                    if (glob) {
                        d_phi = bearing(src[0], src[1], rcv[0], rcv[1]);
                        d_phi -= bearing(src[0], src[1], s[1] * 180.0 / Pi, s[2] * 180.0 / Pi);
                    } else d_phi = (std::atan2(rcv[1] - src[1], rcv[0] - src[0]) - std::atan2(s[1] - src[1], s[0] - src[0])) * 180.0 / Pi;
                    while (d_phi > 180.0) d_phi -= 360.0;
                    while (d_phi < -180.0) d_phi += 360.0;
                    if (std::fabs(d_phi) < o.azimuth_err_lim) {
                        e.theta_est = theta - d_theta; e.phi_est = glob ? 90.0 - phi : phi; e.ok = true; e.complete = true;
                        return e;
                    }
                    phi += d_phi * 0.9;
                    theta_min = std::max(theta - 7.5, theta_min);
                    break;
                }
                if (iterations >= 3) d_theta = modify_d_theta(r - r_rcvr, (r - r_prev) / (2.0 * d_theta), o.d_theta_big, o.d_theta_small, glob ? 0.5 : 2.0);
                r_prev = r;
            }
            if (theta_max_reached) { e.theta_next = theta_max; e.next_known = true; break; }
            iterations++;
            if (iterations >= 1 && iterations < 3) d_theta = o.d_theta_big / 2.0;
        }
        e.complete = true;
        return e;
    }

    // ---- GeoAc_3DEigenray_LM, Eigenray.cpp:123-335 (search part; the attributes of a found eigenray come from one more trace) ----
    struct Lm { bool complete = false, found = false; double theta = 0, phi = 0; int iters = 0; };
    Lm lm(int si, const double rcv[2], double theta, double phi, int bnc_cnt) {
        Lm out; out.theta = theta; out.phi = phi;
        const double Mx = srcs[si].Mx, My = srcs[si].My;
        double dr, dr_prev = 10000.0;
        const double tolerance = o.tolerance, theta_lim_step = 0.2, phi_lim_step = 0.2;
        double step_scalar = 1.0;
        long double x, y, dx, dy, dx_dt, dy_dt, dx_dp, dy_dp, det, dt = 0, dp = 0;
        double nu0_xy[2] = { 0, 0 };
        for (int n = 0; n <= o.iterations; n++) {
            out.iters = n;
            if (n == o.iterations) break;
            const double th = theta * Pi / 180.0, ph = phi * Pi / 180.0;
            if (strat && !glob) {
                const double nu0[3] = { std::cos(th) * std::cos(ph), std::cos(th) * std::sin(ph), std::sin(th) };
                const double M = 1.0 + (nu0[0] * Mx + nu0[1] * My + nu0[2] * 0.0);
                nu0_xy[0] = nu0[0] / M; nu0_xy[1] = nu0[1] / M;
            }
            bool brk;
            const double* s = lookup(si, th, ph, 1, bnc_cnt, &brk);
            if (!s) { out.theta = theta; out.phi = phi; return out; }          // incomplete
            if (brk) break;
            if (glob) {                                                        // Eigenray.Global.cpp:183-184 (x = lat, y = lon)
                x = s[1]; y = s[2];
                dr = gc_distance((double)(x * 180.0 / Pi), (double)(y * 180.0 / Pi), rcv[0], rcv[1]);
            } else {
                x = s[0]; dx = rcv[0] - x;
                y = s[1]; dy = rcv[1] - y;
                dr = (double)std::sqrt(dx * dx + dy * dy);
            }
            if (dr < tolerance) { out.found = true; break; }
            else if (n > 0 && dr > dr_prev) {
                theta -= dt * step_scalar;
                phi -= dp * step_scalar;
                step_scalar /= 2.0;
                if (std::sqrt(dt * dt + dp * dp) * step_scalar < 1.0e-12) break;
            } else {
                step_scalar = std::min(1.0, step_scalar * 1.25);
                if (glob) {                                                    // Eigenray.Global.cpp:283-294; dx, dy = d_lat, d_lon
                    const double rg = 6370.0 + z_grnd;
                    dx = rcv[0] * Pi / 180.0 - x;
                    dy = rcv[1] * Pi / 180.0 - y;
                    dx_dt = s[7] - 1.0 / rg * s[4] / s[3] * s[6];
                    dx_dp = s[13] - 1.0 / rg * s[4] / s[3] * s[12];
                    dy_dt = s[8] - 1.0 / (rg * std::cos(x)) * s[5] / s[3] * s[6];
                    dy_dp = s[14] - 1.0 / (rg * std::cos(x)) * s[5] / s[3] * s[12];
                    det = dx_dt * dy_dp - dx_dp * dy_dt;
                    dt = (dy_dp * dx - dx_dp * dy) / det * 180.0 / Pi;
                    dp = (-dy_dt * dx + dx_dt * dy) / det * 180.0 / Pi;
                } else if (strat) {
                    dx_dt = s[4] - nu0_xy[0] / s[3] * s[6];
                    dy_dt = s[5] - nu0_xy[1] / s[3] * s[6];
                    dx_dp = s[8] - nu0_xy[0] / s[3] * s[10];
                    dy_dp = s[9] - nu0_xy[1] / s[3] * s[10];
                } else {
                    dx_dt = s[6] - s[3] / s[5] * s[8];
                    dy_dt = s[7] - s[4] / s[5] * s[8];
                    dx_dp = s[12] - s[3] / s[5] * s[14];
                    dy_dp = s[13] - s[4] / s[5] * s[14];
                }
                if (!glob) {
                    det = dx_dt * dy_dp - dx_dp * dy_dt;
                    dt = 1.0 / det * (dy_dp * dx - dx_dp * dy) * 180.0 / Pi;
                    dp = 1.0 / det * (dx_dt * dy - dy_dt * dx) * 180.0 / Pi;
                }
                if (dt > theta_lim_step) dt = theta_lim_step;
                if (dp > phi_lim_step) dp = phi_lim_step;
                if (dt < -theta_lim_step) dt = -theta_lim_step;
                if (dp < -phi_lim_step) dp = -phi_lim_step;
                theta += dt * step_scalar;
                phi += dp * step_scalar;
                dr_prev = dr;
            }
        }
        out.complete = true; out.theta = theta; out.phi = phi;
        return out;
    }

    // one GeoAc_EstimateEigenray call (+ its LM) of the chain of (search, bounce count)
    struct Call { int rcvr, n_bnc; Est e; Lm l; };
    // the calls of one search and bounce count, in the reference's order; done: every call complete (only cached rays read)
    struct Chain { int search, n_bnc; bool done = false; std::vector<Call> calls; };

    // Replays the chain against the cache from its start.  Returns true when nothing is missing.
    // direct != nullptr: -eig_direct (GeoAc3D_RunEigDirect, GeoAc3D_main.cpp:546-601): no estimate, one LM search from the
    // caller's { theta_est, phi_est [deg from the x axis], bounces } of the search.
    bool replay(Chain& ch, int si, const double rcv[2], const double* direct) {
        ch.calls.clear();
        bool all = true;
        if (direct) {
            Call c; c.rcvr = ch.search; c.n_bnc = ch.n_bnc;
            c.e.complete = c.e.ok = c.e.next_known = true; c.e.theta_est = direct[3 * ch.search]; c.e.phi_est = direct[3 * ch.search + 1]; c.e.theta_next = 0.0;
            c.l = lm(si, rcv, c.e.theta_est, c.e.phi_est, c.n_bnc);
            all = c.l.complete;
            ch.calls.push_back(c);
        } else {
            double theta_start = o.theta_min;
            int guard = 0;
            while (theta_start < o.theta_max && guard++ < 100000) {
                Call c; c.rcvr = ch.search; c.n_bnc = ch.n_bnc;
                c.e = estimate(si, rcv, theta_start, o.theta_max, ch.n_bnc);
                if (c.e.complete && c.e.ok) c.l = lm(si, rcv, c.e.theta_est, c.e.phi_est, ch.n_bnc);
                const bool done = c.e.complete && (!c.e.ok || c.l.complete);
                all = all && done;
                ch.calls.push_back(c);
                if (!c.e.next_known) break;                   // cannot place the next call yet (or theta_next was never set, as in the reference)
                theta_start = c.e.theta_next;
            }
        }
        ch.done = all;
        return all;
    }

    // The trace of n rays from the search's sources (sid: index into srcs) with the context's parameters but these bounces,
    // calc_amp and accum_per_segment.  Adds the kernel time to kernel_ms.
    int trace(int64_t n, const int32_t* sid, const double* th, const double* ph, int bounces, int amp, int accum,
              double* rec, int32_t* st, std::string& err) {
        geoac_params p; int rc = geoac_get_params(ctx, &p); if (rc) return rc;
        p.bounces = bounces; p.calc_amp = amp; p.accum_per_segment = accum;
        rc = geoac_set_params(ctx, &p); if (rc) return rc;
        std::vector<double> tsrc(3 * srcs.size());
        for (size_t i = 0; i < srcs.size(); i++) for (int k = 0; k < 3; k++) tsrc[3 * i + k] = srcs[i].trace[k];
        std::vector<int32_t> ns((size_t)n * (bounces + 1));
        rc = geoac_trace_sources(ctx, (int)srcs.size(), tsrc.data(), n, sid, th, ph, rec, st, ns.data());
        if (rc) { err = geoac_last_error(ctx); return rc; }
        int64_t steps = 0; double ms = 0.0;
        if (geoac_last_trace_stats(ctx, &steps, &ms) == GEOAC_OK) kernel_ms += ms;
        rays_traced += n;
        return GEOAC_OK;
    }

    // this round's requests, one batch per calc_amp setting, ordered by (source, theta, phi) so that warps hold rays of
    // one source; the results go into the cache
    int trace_requests(std::string& err) {
        std::vector<std::pair<RayKey, Request>> reqs(want.begin(), want.end());
        std::sort(reqs.begin(), reqs.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
        for (int amp = 0; amp < 2; amp++) {
            std::vector<double> th, ph; std::vector<int32_t> sid; std::vector<RayKey> keys; int nb = 0;
            for (const auto& kv : reqs) if (kv.first.amp == amp) {
                th.push_back(kv.second.theta); ph.push_back(kv.second.phi); sid.push_back(kv.first.src);
                keys.push_back(kv.first); nb = std::max(nb, kv.second.nb);
            }
            if (th.empty()) continue;
            const int64_t n = (int64_t)th.size(), n_rec = nb + 1, slots = n * n_rec;
            std::vector<double> rec((size_t)GEOAC_NFIELDS * slots);
            std::vector<int32_t> st((size_t)slots);
            if (int rc = trace(n, sid.data(), th.data(), ph.data(), nb, amp, 0, rec.data(), st.data(), err)) return rc;
            const int nc = kCols[amp];
            for (int64_t i = 0; i < n; i++) {
                const RayVal v{ nb, (int64_t)st_pool.size(), (int64_t)x_pool.size() };
                st_pool.insert(st_pool.end(), st.begin() + i * n_rec, st.begin() + (i + 1) * n_rec);
                for (int b = 0; b < n_rec; b++) for (int f = 0; f < nc; f++) x_pool.push_back(rec[(size_t)f * slots + i * n_rec + b]);
                cache[keys[i]] = v;
            }
        }
        want.clear();
        return GEOAC_OK;
    }
};

// Puts the caller's parameters back when the search ends, on every path.
struct RestoreParams {
    geoac_ctx* ctx; geoac_params p;
    ~RestoreParams() { geoac_set_params(ctx, &p); }
};

double ms_since(std::chrono::steady_clock::time_point t0) {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

}  // namespace

extern "C" int geoac_default_eig_opts(geoac_eig_opts* o) {
    if (!o) return GEOAC_ERR_BAD_ARG;
    std::memset(o, 0, sizeof *o);
    o->theta_min = 0.5; o->theta_max = 45.0; o->bnc_min = 0; o->bnc_max = 0; o->iterations = 25;      // GeoAc3D_main.cpp:461-464
    o->azimuth_err_lim = 2.0; o->d_theta_big = 0.25; o->d_theta_small = 0.002; o->tolerance = 0.1;   // Eigenray.cpp:20-21,139
    o->max_rounds = 4096; o->src_lat_deg = 30.0; o->src_lon_deg = 0.0;                              // GeoAcGlobal_main.cpp:497
    return GEOAC_OK;
}

// The search engine of every entry point.  n_src sources in the convention of geoac_eigenray_search_sources (Cartesian
// (x, y, z) [km]; Global (altitude [km], lat [deg], lon [deg])); search i runs from src[src_id[i]] to rcvr_xy[2i..2i+1].
// The pointers are checked by the caller, the sources too where they come from outside the context.
static int run_search(geoac_ctx* ctx, const geoac_eig_opts* opts, int n_src, const double* src, int n_rcvr, const int32_t* src_id,
                      const double* rcvr_xy, const double* direct, int64_t cap_rows, double* rows, int64_t* n_rows, int64_t* stats) {
    const auto t0 = std::chrono::steady_clock::now();
    const int variant = geoac_get_variant(ctx);
    if (variant == GEOAC_2D) return geoac_fail_msg(ctx, GEOAC_ERR_BAD_ARG, "the eigenray search needs a 3-D variant (GeoAc2D has none)");
    if (opts->bnc_min < 0 || opts->bnc_max < opts->bnc_min || opts->iterations < 0 || !(opts->d_theta_big > 0.0))
        return geoac_fail_msg(ctx, GEOAC_ERR_BAD_ARG, "eigenray options: need 0 <= bnc_min <= bnc_max, iterations >= 0 and d_theta_big > 0");
    if (int rc = geoac_sample_atmosphere(ctx, 0, nullptr, nullptr, nullptr, nullptr)) return rc;      // GEOAC_ERR_NO_ATMO, no device work
    geoac_params user; int rc = geoac_get_params(ctx, &user); if (rc) return rc;
    RestoreParams restore{ ctx, user };
    Search S; S.ctx = ctx; S.variant = variant; S.strat = variant == GEOAC_3D; S.o = *opts;
    S.glob = variant == GEOAC_GLOBAL || variant == GEOAC_GLOBAL_RNGDEP; S.z_grnd = user.z_grnd;
    S.srcs.resize(n_rcvr > 0 ? (size_t)n_src : 0);
    for (size_t i = 0; i < S.srcs.size(); i++) {
        const double* s = src + 3 * i;
        Src& q = S.srcs[i];
        if (S.glob) {
            // Source_Loc = (lat, lon) in degrees as the Global mains hold it (GeoAcGlobal_main.cpp:497); the rays start from
            // lat*Pi/180, lon*Pi/180 (Eigenray.Global.cpp:78)
            q.loc[0] = s[1]; q.loc[1] = s[2]; q.loc[2] = std::max(user.z_grnd, s[0]);
            q.trace[0] = q.loc[2]; q.trace[1] = q.loc[0] * Pi / 180.0; q.trace[2] = q.loc[1] * Pi / 180.0;
        } else {
            q.loc[0] = s[0]; q.loc[1] = s[1]; q.loc[2] = std::max(user.z_grnd, s[2]);
            for (int k = 0; k < 3; k++) q.trace[k] = s[k];
        }
    }
    if (S.strat && !S.srcs.empty()) {
        // c, u, v at the (clamped) source points: the kernels' source state (geoac_source_state), one device pass for all
        const size_t n = S.srcs.size();
        std::vector<double> p0(n), p1(n), p2(n), a((size_t)GEOAC_ATM_NF * n);
        for (size_t i = 0; i < n; i++) { p0[i] = S.srcs[i].loc[0]; p1[i] = S.srcs[i].loc[1]; p2[i] = S.srcs[i].loc[2]; }
        rc = geoac_sample_atmosphere(ctx, (int64_t)n, p0.data(), p1.data(), p2.data(), a.data()); if (rc) return rc;
        for (size_t i = 0; i < n; i++) {
            S.srcs[i].Mx = a[GEOAC_ATM_U * n + i] / a[GEOAC_ATM_C * n + i];
            S.srcs[i].My = a[GEOAC_ATM_V * n + i] / a[GEOAC_ATM_C * n + i];
        }
    }
    std::vector<Search::Chain> chains;
    for (int ir = 0; ir < n_rcvr; ir++) {
        if (direct) chains.push_back({ ir, (int)direct[3 * ir + 2] });
        else for (int n_bnc = opts->bnc_min; n_bnc <= opts->bnc_max; n_bnc++) chains.push_back({ ir, n_bnc });
    }
    std::string err;
    const int max_rounds = opts->max_rounds > 0 ? opts->max_rounds : 4096;
    bool done = false;
    for (S.rounds = 0; S.rounds < max_rounds; S.rounds++) {
        const auto r0 = std::chrono::steady_clock::now();
        done = true;
        for (Search::Chain& ch : chains)
            if (!ch.done) done = S.replay(ch, src_id[ch.search], rcvr_xy + 2 * ch.search, direct) && done;
        S.replay_ms += ms_since(r0);
        if (done) break;
        rc = S.trace_requests(err);
        if (rc) return rc;
    }
    if (!done) return geoac_fail_msg(ctx, GEOAC_ERR_TOO_LARGE, "eigenray search: not complete after max_rounds = " + std::to_string(max_rounds) + " trace batches");
    std::vector<const Search::Call*> calls;
    for (const Search::Chain& ch : chains) for (const Search::Call& c : ch.calls) calls.push_back(&c);
    // attributes of the eigenrays found: the per-segment sums of the reference's final pass (Eigenray.cpp:203-244), one batch
    std::vector<int> found;
    for (size_t i = 0; i < calls.size(); i++) if (calls[i]->e.ok && calls[i]->l.found) found.push_back((int)i);
    std::vector<double> rec; std::vector<int32_t> st; int nbmax = 0; int64_t slots = 0;
    if (!found.empty()) {
        std::vector<double> th, ph; std::vector<int32_t> sid;
        for (int i : found) {
            th.push_back(calls[i]->l.theta * Pi / 180.0); ph.push_back(calls[i]->l.phi * Pi / 180.0); sid.push_back(src_id[calls[i]->rcvr]);
            nbmax = std::max(nbmax, calls[i]->n_bnc);
        }
        slots = (int64_t)found.size() * (nbmax + 1);
        rec.resize((size_t)GEOAC_NFIELDS * slots); st.resize((size_t)slots);
        rc = S.trace((int64_t)found.size(), sid.data(), th.data(), ph.data(), nbmax, 1, 1, rec.data(), st.data(), err);
        if (rc) return rc;
    }
    *n_rows = (int64_t)calls.size();
    int64_t fi = 0;
    for (size_t i = 0; i < calls.size(); i++) {
        const Search::Call& c = *calls[i];
        const double* src = S.srcs[src_id[c.rcvr]].loc;
        const bool is_found = c.e.ok && c.l.found;
        if ((int64_t)i < cap_rows) {
            double* r = rows + i * GEOAC_EIG_NF;
            for (int k = 0; k < GEOAC_EIG_NF; k++) r[k] = 0.0;
            r[0] = c.rcvr; r[1] = c.n_bnc; r[2] = c.e.ok ? 1.0 : 0.0; r[3] = c.e.theta_est; r[4] = c.e.ok ? c.e.phi_est : 0.0; r[5] = c.e.theta_next;
            r[6] = is_found ? 1.0 : 0.0;
            if (c.e.ok) { r[7] = c.l.theta; r[8] = c.l.phi; r[16] = c.l.iters; }
            if (is_found) {
                const int64_t slot = fi * (nbmax + 1) + c.n_bnc;
                auto F = [&](int f) { return rec[(size_t)f * slots + slot]; };
                const double rx = rcvr_xy[2 * c.rcvr], ry = rcvr_xy[2 * c.rcvr + 1];
                const double tt = F(GEOAC_F_TRAVELTIME);
                r[9] = tt;
                r[11] = F(GEOAC_F_AMPLITUDE); r[12] = F(GEOAC_F_ATTEN); r[13] = F(GEOAC_F_INCLINATION);
                double back_az, dev;
                if (S.glob) {                                                                                      // Eigenray.Global.cpp:238-241,266-273
                    r[10] = Search::gc_distance(src[0], src[1], rx, ry) / tt;
                    if (variant == GEOAC_GLOBAL_RNGDEP) r[13] = -r[13];          // the record follows that main's +asin (App. A-16); the search prints -asin
                    back_az = 90.0 - std::atan2(-F(4), -F(5)) * 180.0 / Pi;
                    dev = back_az - Search::bearing(rx, ry, src[0], src[1]);
                    if (dev > 180.0) dev -= 360.0;
                    if (dev < -180.0) dev += 360.0;
                } else {
                    r[10] = std::sqrt(std::pow(F(0) - src[0], 2) + std::pow(F(1) - src[1], 2)) / tt;               // celerity, Eigenray.cpp:260
                    back_az = S.strat ? (90.0 - (c.l.phi * Pi / 180.0) * 180.0 / Pi) + 180.0                        // :239-244
                                      : 90.0 - std::atan2(-F(4), -F(3)) * 180.0 / Pi;
                    dev = back_az - (90.0 - std::atan2(src[1] - ry, src[0] - rx) * 180.0 / Pi);
                    while (back_az > 180.0) back_az -= 360.0;
                    while (back_az < -180.0) back_az += 360.0;
                    while (dev > 180.0) dev -= 360.0;
                    while (dev < -180.0) dev += 360.0;
                }
                r[14] = back_az; r[15] = dev;
                r[17] = st[(size_t)slot];
            }
        }
        if (is_found) fi++;
    }
    if (stats) { stats[0] = S.rounds; stats[1] = S.rays_traced; stats[2] = (int64_t)found.size(); }
    const double ms3[3] = { S.replay_ms, S.kernel_ms, ms_since(t0) };
    geoac_set_eigenray_ms(ctx, ms3);
    return (int64_t)calls.size() <= cap_rows ? GEOAC_OK
                                             : geoac_fail_msg(ctx, GEOAC_ERR_TOO_LARGE, std::to_string(calls.size()) + " rows produced, rows holds "
                                                              + std::to_string(cap_rows) + " (n_rows is set)");
}

// The one-source entry points: every search from params.src (Global: params.src[0] and opts' source in degrees)
static int run_one_source(geoac_ctx* ctx, const geoac_eig_opts* opts, int n_rcvr, const double* rcvr_xy, const double* direct,
                          int64_t cap_rows, double* rows, int64_t* n_rows, int64_t* stats) {
    if (!ctx || !opts || !rcvr_xy || !n_rows || n_rcvr < 0 || (cap_rows > 0 && !rows)) return GEOAC_ERR_BAD_ARG;
    geoac_params user; int rc = geoac_get_params(ctx, &user); if (rc) return rc;
    const int variant = geoac_get_variant(ctx);
    const bool glob = variant == GEOAC_GLOBAL || variant == GEOAC_GLOBAL_RNGDEP;
    const double src[3] = { user.src[0], glob ? opts->src_lat_deg : user.src[1], glob ? opts->src_lon_deg : user.src[2] };
    const std::vector<int32_t> src_id((size_t)n_rcvr, 0);
    return run_search(ctx, opts, 1, src, n_rcvr, src_id.data(), rcvr_xy, direct, cap_rows, rows, n_rows, stats);
}

extern "C" int geoac_eigenray_search(geoac_ctx* ctx, const geoac_eig_opts* opts, int n_rcvr, const double* rcvr_xy,
                                     int64_t cap_rows, double* rows, int64_t* n_rows, int64_t* stats) {
    return run_one_source(ctx, opts, n_rcvr, rcvr_xy, nullptr, cap_rows, rows, n_rows, stats);
}

extern "C" int geoac_eigenray_direct(geoac_ctx* ctx, const geoac_eig_opts* opts, int n, const double* rcvr_xy, const double* estimates,
                                     double* rows, int64_t* stats) {
    if (!estimates) return GEOAC_ERR_BAD_ARG;
    for (int i = 0; i < n; i++) if (!(estimates[3 * i + 2] >= 0.0) || estimates[3 * i + 2] > 1000.0) return GEOAC_ERR_BAD_ARG;
    int64_t n_rows = 0;
    return run_one_source(ctx, opts, n, rcvr_xy, estimates, n, rows, &n_rows, stats);
}

extern "C" int geoac_eigenray_search_sources(geoac_ctx* ctx, const geoac_eig_opts* opts, int n_src, const double* src,
                                             int n_rcvr, const int32_t* src_id, const double* rcvr_xy,
                                             int64_t cap_rows, double* rows, int64_t* n_rows, int64_t* stats) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    if (n_rcvr < 0) return geoac_fail_msg(ctx, GEOAC_ERR_BAD_ARG, "geoac_eigenray_search_sources: n_rcvr < 0");
    if (!opts || !n_rows || (n_rcvr > 0 && (!src || !src_id || !rcvr_xy)) || (cap_rows > 0 && !rows))
        return geoac_fail_msg(ctx, GEOAC_ERR_BAD_ARG, "geoac_eigenray_search_sources: need non-null opts, n_rows and buffers");
    if (n_rcvr > 0) {
        if (n_src < 1) return geoac_fail_msg(ctx, GEOAC_ERR_BAD_ARG, "geoac_eigenray_search_sources: need n_src >= 1");
        for (int s = 0; s < n_src; s++)
            if (!std::isfinite(src[3 * (size_t)s]) || !std::isfinite(src[3 * (size_t)s + 1]) || !std::isfinite(src[3 * (size_t)s + 2]))
                return geoac_fail_msg(ctx, GEOAC_ERR_BAD_ARG, "geoac_eigenray_search_sources: coordinates of source " + std::to_string(s) + " are not finite");
        for (int i = 0; i < n_rcvr; i++)
            if (src_id[i] < 0 || src_id[i] >= n_src)
                return geoac_fail_msg(ctx, GEOAC_ERR_BAD_ARG, "geoac_eigenray_search_sources: src_id of search " + std::to_string(i) + " is "
                                                              + std::to_string(src_id[i]) + ", outside [0, " + std::to_string(n_src) + ")");
    }
    return run_search(ctx, opts, n_src, src, n_rcvr, src_id, rcvr_xy, nullptr, cap_rows, rows, n_rows, stats);
}
