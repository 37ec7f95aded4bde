// capi.cu -- the extern "C" boundary of libgeoac_b200.so (declared in include/geoac_b200.h).
//
// Host side only: context management, table construction (the reference's Thomas recurrences,
// Code/Atmo/G2S_Spline1D.cpp:161-196, so the slope tables are bit-identical), kernel launches, H2D/D2H staging.
// There is deliberately NO CPU implementation of the trace here: without an sm_100 device every entry point fails.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cmath>
#include <string>
#include <vector>
#include <algorithm>
#include <type_traits>
#include <thread>
#include <atomic>
#include <limits>
#include <utility>

#include "core.cuh"
#include "eq_cartesian.cuh"
#include "eq_global.cuh"
#include "eq_rngdep.cuh"
#include "trace_kernel.cuh"
#include "atmo_sample.cuh"
#include "host_tables.hpp"

using namespace geoac;

static thread_local std::string g_create_error;

// Experiment / test knobs (DESIGN.md section 6).  Defaults come from the GEOAC_B200_* environment variables, read ONCE in
// geoac_create; afterwards only geoac_set_knob changes them -- nothing on the launch path touches the environment.
struct Knobs {
    int lpt = 1;            // claim order: 0 natural, 1 automatic, 2 always
    int scout_coarse = 0;   // step-size multiple of the cost scout (0 = default per variant)
    int cost_shift = 2;     // log2 coarsening of the cost key
    int coop = 1;           // cooperative (several lanes per ray) modes of the range-dependent sets
    int sbpoly = 1;         // absorption through per-interval polynomials
    int host_tables = 0;    // build the node tables on the host
    int long_alpha = 100;   // a packet is LONG if its cost exceeds long_alpha % of the average work of a lane
    int long_sm_pct = 90;   // at most this share of the SMs is given to the long-region launch (its CTAs help with the main region once theirs is drained)
    int exclusive = 1;      // long-region launch keeps its SMs to itself (0: one launch, which claims the main region first)
    int dilate = 400;       // range-dependent sets: the ordering cost of a ray is the maximum over its inclination neighbours within this many
                            // millidegrees (0 = off): the edge of a long ray family is scheduled as long
    int quarter = 1;        // the longest long-region packets are claimed as quarter packets while the exclusive SMs have warps to spare
    int quarter_alpha = 210;// ... those whose cost exceeds this % of the average lane work (lone-warp speed is ~2.1x the loaded one)
};
// name for geoac_set_knob, suffix of the environment variable, field, and the range a value is clamped to
struct KnobDef { const char* name; const char* env; int Knobs::* field; int lo, hi; };
constexpr int kLo = std::numeric_limits<int>::min(), kHi = std::numeric_limits<int>::max();   // no clamp
static const KnobDef kKnobs[] = {
    { "lpt", "LPT", &Knobs::lpt, kLo, kHi },
    { "scout_coarse", "SCOUT_COARSE", &Knobs::scout_coarse, 0, kHi },
    { "cost_shift", "COSTSHIFT", &Knobs::cost_shift, 0, 7 },
    { "coop", "COOP", &Knobs::coop, kLo, kHi },
    { "sbpoly", "SBPOLY", &Knobs::sbpoly, kLo, kHi },
    { "host_tables", "HOST_TABLES", &Knobs::host_tables, kLo, kHi },
    { "long_alpha", "LONG_ALPHA", &Knobs::long_alpha, 1, kHi },
    { "long_sm_pct", "LONG_SM_PCT", &Knobs::long_sm_pct, 1, 90 },
    { "exclusive", "EXCLUSIVE", &Knobs::exclusive, kLo, kHi },
    { "dilate", "DILATE", &Knobs::dilate, 0, kHi },
    { "quarter", "QUARTER", &Knobs::quarter, kLo, kHi },
    { "quarter_alpha", "QUARTER_ALPHA", &Knobs::quarter_alpha, 1, kHi },
};
static Knobs knobs_from_env() {
    Knobs k;
    for (const KnobDef& d : kKnobs)
        if (const char* e = std::getenv((std::string("GEOAC_B200_") + d.env).c_str())) k.*d.field = std::clamp(std::atoi(e), d.lo, d.hi);
    return k;
}

// One device allocation (PINNED: page-locked host memory) and its capacity in bytes, freed with its owner.  grow() keeps the
// allocation when it holds `need` bytes and otherwise frees it and allocates anew: the contents are not kept.
template <class T, bool PINNED = false>
struct Buf {
    T* p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf&& o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    Buf& operator=(Buf&& o) noexcept { if (this != &o) { release(); p = std::exchange(o.p, nullptr); cap = std::exchange(o.cap, 0); } return *this; }
    ~Buf() { release(); }
    void release() {
        if (PINNED) cudaFreeHost(p); else cudaFree(p);
        p = nullptr; cap = 0;
    }
    cudaError_t grow(size_t need) {
        if (need <= cap) return cudaSuccess;
        release();
        void* q = nullptr;
        const cudaError_t e = PINNED ? cudaHostAlloc(&q, need, cudaHostAllocDefault) : cudaMalloc(&q, need);
        if (e == cudaSuccess) { p = static_cast<T*>(q); cap = need; }
        return e;
    }
};

struct geoac_ctx {
    int variant = 0, device = 0, sm_count = 0;
    Knobs knobs;
    geoac_params prm{};
    std::string err;
    // 1-D table
    bool have_atmo = false;
    int n = 0;
    double xmin = 0, xmax = 0;
    std::vector<double> h_table;
    Buf<double> d_table;
    Buf<double> d_sbpoly;            // per-interval absorption polynomials of the 1-D table (core.cuh), rebuilt with the invariants
    // range-dependent grid
    bool is_grid = false;
    Grid3D grid{};
    Buf<double> d_tuv, d_rho, d_ax;
    Buf<LaunchConsts> d_consts;
    Buf<unsigned long long> d_counters;           // [0] ray counter, [1] total steps
    Buf<double> d_prev;                           // y_{k-1} scratch of the trace kernel
    Buf<double> d_path; Buf<int32_t> d_path_rows; // raypath capture staging
    Buf<double> d_caus; Buf<int32_t> d_caus_rows; // caustic event staging
    // longest-ray-first scheduling: predicted costs, the costs the order uses (dilated), claim order, sort scratch
    Buf<uint32_t> d_cost, d_cost_dilated, d_order, d_order2, d_hist, d_blockhist;
    Buf<uint8_t> d_keys;
    int last_launches = 0;
    // staging for the host-buffer entry point
    Buf<double> d_theta, d_phi, d_rec;
    Buf<int32_t> d_status, d_nsteps;
    cudaStream_t stream = nullptr, stream_long = nullptr;      // stream_long: the concurrent long-region launch of the range-dependent sets
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_fork = nullptr, ev_join = nullptr, ev_m0 = nullptr, ev_m1 = nullptr, ev_l0 = nullptr, ev_l1 = nullptr;
    cudaEvent_t ev_d0 = nullptr, ev_d1 = nullptr;                // the work of the last geoac_trace_device on the caller's stream
    bool timed_launches = false;
    int last_long_packets = 0, last_long_ctas = 0, last_quarter_packets = 0;
    int64_t last_steps = 0; double last_ms = 0.0;
    bool ms_pending = false;                                    // last_ms is still to be read from ev_d0 / ev_d1
    bool consts_dirty = true;
    bool src_set = false;
    // pinned host staging of geoac_trace_multi (this context's share of the batch: angles in, records out)
    Buf<double, true> pin_theta, pin_phi, pin_rec;
    Buf<int32_t, true> pin_status, pin_nsteps;
    // staging of geoac_sample_atmosphere: the three coordinates in, GEOAC_ATM_NF rows out, one pass of points at a time
    Buf<double> d_smp_in, d_smp_out;
};

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
    ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_); return GEOAC_ERR_CUDA; } } while (0)

static int fail(geoac_ctx* ctx, int code, const std::string& msg) { if (ctx) ctx->err = msg; return code; }

extern "C" int geoac_eq_count(int variant, int calc_amp) {          // Code/GeoAc/GeoAc.Interface.cpp:21-41
    switch (variant) {
        case GEOAC_2D: return calc_amp ? 6 : 3;
        case GEOAC_3D: return calc_amp ? 12 : 4;
        case GEOAC_GLOBAL: case GEOAC_3D_RNGDEP: case GEOAC_GLOBAL_RNGDEP: return calc_amp ? 18 : 6;
    }
    return -1;
}

extern "C" int geoac_default_params(int variant, geoac_params* p) {
    if (!p || variant < 0 || variant > GEOAC_GLOBAL_RNGDEP) return GEOAC_ERR_BAD_ARG;
    std::memset(p, 0, sizeof *p);
    const bool glob = (variant == GEOAC_GLOBAL || variant == GEOAC_GLOBAL_RNGDEP);
    p->ds_min = 0.001; p->ds_max = 0.5;                   // GeoAc.Parameters.cpp:20-21
    p->ray_limit = glob ? 10000.0 : 5000.0;              // GeoAc.Parameters.cpp:24 / .Global.cpp
    p->vert_limit = 200.0; p->range_limit = 2000.0;
    p->z_grnd = 0.0; p->tweak_abs = 0.3; p->freq = 0.1;
    p->bounces = 2; p->calc_amp = 1;
    p->accum_per_segment = (variant == GEOAC_2D) ? 1 : 0;
    if (variant == GEOAC_GLOBAL) { p->src[1] = 30.0 * kPi / 180.0; p->src[2] = 0.0; }   // GeoAcGlobal_main.cpp:120
    return GEOAC_OK;
}

extern "C" geoac_ctx* geoac_create(int variant, int device, int* status) {
    auto bail = [&](int code, const std::string& m) -> geoac_ctx* { g_create_error = m; if (status) *status = code; return nullptr; };
    if (variant < 0 || variant > GEOAC_GLOBAL_RNGDEP) return bail(GEOAC_ERR_BAD_ARG, "unknown variant");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return bail(GEOAC_ERR_NO_DEVICE, "no CUDA device (this library has no CPU path)");
    if (device < 0 || device >= ndev) return bail(GEOAC_ERR_BAD_ARG, "device ordinal out of range");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(GEOAC_ERR_CUDA, "cudaGetDeviceProperties failed");
    if (prop.major != 10) return bail(GEOAC_ERR_NO_DEVICE, std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) + ", kernels are built for sm_100a only");
    geoac_ctx* ctx = new geoac_ctx();
    ctx->variant = variant; ctx->device = device; ctx->sm_count = prop.multiProcessorCount;
    ctx->knobs = knobs_from_env();
    geoac_default_params(variant, &ctx->prm);
    cudaSetDevice(device);
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess
           && cudaStreamCreateWithPriority(&ctx->stream_long, cudaStreamNonBlocking, prio_hi) == cudaSuccess
           && cudaEventCreate(&ctx->ev0) == cudaSuccess && cudaEventCreate(&ctx->ev1) == cudaSuccess
           && cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) == cudaSuccess
           && cudaEventCreate(&ctx->ev_m0) == cudaSuccess && cudaEventCreate(&ctx->ev_m1) == cudaSuccess && cudaEventCreate(&ctx->ev_l0) == cudaSuccess && cudaEventCreate(&ctx->ev_l1) == cudaSuccess
           && cudaEventCreate(&ctx->ev_d0) == cudaSuccess && cudaEventCreate(&ctx->ev_d1) == cudaSuccess
           && ctx->d_consts.grow(sizeof(LaunchConsts)) == cudaSuccess
           && ctx->d_counters.grow(8 * sizeof(unsigned long long)) == cudaSuccess;
    if (!ok) { std::string m = cudaGetErrorString(cudaGetLastError()); delete ctx; return bail(GEOAC_ERR_CUDA, "context allocation failed: " + m); }
    if (status) *status = GEOAC_OK;
    return ctx;
}

extern "C" void geoac_destroy(geoac_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);                       // the buffers are freed with the context, on its device
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_m0) cudaEventDestroy(ctx->ev_m0);
    if (ctx->ev_m1) cudaEventDestroy(ctx->ev_m1);
    if (ctx->ev_l0) cudaEventDestroy(ctx->ev_l0);
    if (ctx->ev_l1) cudaEventDestroy(ctx->ev_l1);
    if (ctx->ev_d0) cudaEventDestroy(ctx->ev_d0);
    if (ctx->ev_d1) cudaEventDestroy(ctx->ev_d1);
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->stream_long) cudaStreamDestroy(ctx->stream_long);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* geoac_last_error(const geoac_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int geoac_get_params(const geoac_ctx* ctx, geoac_params* p) { if (!ctx || !p) return GEOAC_ERR_BAD_ARG; *p = ctx->prm; return GEOAC_OK; }
extern "C" int geoac_set_params(geoac_ctx* ctx, const geoac_params* p) {
    if (!ctx || !p) return GEOAC_ERR_BAD_ARG;
    if (p->bounces < 0 || p->ds_min <= 0.0 || p->ray_limit <= 0.0) return fail(ctx, GEOAC_ERR_BAD_ARG, "bad params");
    ctx->prm = *p; ctx->consts_dirty = true; ctx->src_set = true; return GEOAC_OK;
}

extern "C" int geoac_set_knob(geoac_ctx* ctx, const char* name, int value) {
    if (!ctx || !name) return GEOAC_ERR_BAD_ARG;
    for (const KnobDef& d : kKnobs)
        if (!std::strcmp(name, d.name)) { ctx->knobs.*d.field = std::clamp(value, d.lo, d.hi); return GEOAC_OK; }
    return fail(ctx, GEOAC_ERR_BAD_ARG, std::string("unknown knob ") + name);
}

// ---- knot slopes of the natural spline: same tridiagonal recurrences as G2S_Spline1D.cpp:161-196 ----
static void natural_slopes(const std::vector<double>& x, const double* f, double* s) {
    const int n = (int)x.size();
    std::vector<double> cp(n), dp(n);
    double lo, di, up, rh;
    di = 2.0 / (x[1] - x[0]); up = 1.0 / (x[1] - x[0]);
    rh = 3.0 * (f[1] - f[0]) / std::pow(x[1] - x[0], 2);
    cp[0] = up / di; dp[0] = rh / di;
    for (int i = 1; i < n - 1; i++) {
        lo = 1.0 / (x[i] - x[i - 1]);
        di = 2.0 * (1.0 / (x[i] - x[i - 1]) + 1.0 / (x[i + 1] - x[i]));
        up = 1.0 / (x[i + 1] - x[i]);
        rh = 3.0 * ((f[i] - f[i - 1]) / std::pow(x[i] - x[i - 1], 2) + (f[i + 1] - f[i]) / std::pow(x[i + 1] - x[i], 2));
        cp[i] = up / (di - cp[i - 1] * lo);
        dp[i] = (rh - dp[i - 1] * lo) / (di - cp[i - 1] * lo);
    }
    lo = 1.0 / (x[n - 1] - x[n - 2]); di = 2.0 / (x[n - 1] - x[n - 2]);
    rh = 3.0 * (f[n - 1] - f[n - 2]) / std::pow(x[n - 1] - x[n - 2], 2);
    dp[n - 1] = (rh - dp[n - 2] * lo) / (di - cp[n - 2] * lo);
    s[n - 1] = dp[n - 1];
    for (int i = n - 2; i > -1; i--) s[i] = dp[i] - cp[i] * s[i + 1];
}

extern "C" int geoac_set_atmosphere_1d(geoac_ctx* ctx, int n, const double* z, const double* T,
                                       const double* u, const double* v, const double* rho) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    if (ctx->variant != GEOAC_2D && ctx->variant != GEOAC_3D && ctx->variant != GEOAC_GLOBAL)
        return fail(ctx, GEOAC_ERR_BAD_ARG, "variant needs geoac_set_atmosphere_3d");
    if (n < 3 || !z || !T || !u || !v || !rho) return fail(ctx, GEOAC_ERR_BAD_ARG, "need >= 3 levels and non-null arrays");
    for (int i = 1; i < n; i++) if (!(z[i] > z[i - 1])) return fail(ctx, GEOAC_ERR_BAD_ARG, "altitudes must be strictly increasing");
    cudaSetDevice(ctx->device);
    const bool glob = ctx->variant == GEOAC_GLOBAL;
    std::vector<double> x(n), col(n), slo(n);
    for (int i = 0; i < n; i++) { x[i] = z[i]; if (glob) x[i] += kREarth; }   // r_vals[nr] += r_earth
    ctx->h_table.assign((size_t)TAB_NARR * n, 0.0);                           // one record per level (core.cuh)
    double* tb = ctx->h_table.data();
    for (int i = 0; i < n; i++) {
        tb[(size_t)i * TAB_NARR + TAB_X] = x[i];
        tb[(size_t)i * TAB_NARR + TAB_INVH] = (i + 1 < n) ? 1.0 / (x[i + 1] - x[i]) : 0.0;
    }
    const double* fields[4] = { T, u, v, rho };
    const int slots[4] = { TAB_T, TAB_U, TAB_V, TAB_RHO };
    for (int f = 0; f < 4; f++) {
        for (int i = 0; i < n; i++) col[i] = fields[f][i];
        natural_slopes(x, col.data(), slo.data());
        for (int i = 0; i < n; i++) { tb[(size_t)i * TAB_NARR + slots[f]] = col[i]; tb[(size_t)i * TAB_NARR + slots[f] + 1] = slo[i]; }
    }
    // build into fresh buffers and swap them in only after every step succeeded: a failed call leaves the previous
    // atmosphere (or "none") fully intact instead of dangling pointers
    Buf<double> nt, ns;
    if (ns.grow((size_t)(n - 1) * SBP_STRIDE * sizeof(double)) != cudaSuccess
        || nt.grow(ctx->h_table.size() * sizeof(double)) != cudaSuccess
        || cudaMemcpy(nt.p, tb, ctx->h_table.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess)
        return fail(ctx, GEOAC_ERR_CUDA, std::string("geoac_set_atmosphere_1d: ") + cudaGetErrorString(cudaGetLastError()));
    cudaStreamSynchronize(ctx->stream);                                          // no launch may still read the old tables
    ctx->d_table = std::move(nt); ctx->d_sbpoly = std::move(ns);
    ctx->n = n; ctx->xmin = x[0]; ctx->xmax = x[n - 1];
    // GeoAc_SetPropRegion: G2S_Spline1D.cpp:22-28 / G2S_GlobalSpline1D.cpp:22-30
    ctx->prm.vert_limit = ctx->xmax;
    ctx->prm.range_limit = glob ? 1500.0 : 10000.0;
    if (glob) { ctx->prm.box_min[0] = -kPi / 2.0; ctx->prm.box_max[0] = kPi / 2.0; ctx->prm.box_min[1] = -kPi; ctx->prm.box_max[1] = kPi; }
    ctx->have_atmo = true; ctx->consts_dirty = true;
    return GEOAC_OK;
}

// ---- device-side Set_Slopes_Multi (G2S_MultiDimSpline3D.cpp:306-425, G2S_GlobalMultiDimSpline3D.cpp:313-431) ----
// One thread per (horizontal node, quantity): the ten Thomas solves of a column (f and its two node differences for T, u,
// v; f for rho) are independent, and everything that depends on the vertical axis only (sub-diagonal, pivots, squared
// spacings, the c' sweep) is precomputed once on the host.  Explicit round-to-nearest intrinsics keep every operation
// separate (no FMA contraction), so the tables are bit-identical to host_tables.hpp::build_grid_tables, which follows the
// reference's recurrences operation by operation (checked bitwise by tests/test_gpu_scale.py).
struct ZAux { const double *A, *DEN, *NC, *P2LO, *P2HI; };      // each nz doubles

__global__ void grid_tables_kernel(int glob, int n0, int n1, int nz, const double* ax0, const double* ax1, ZAux za,
                                   const double* T, const double* u, const double* v, const double* rho, double* tuv, double* rh) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long ncol = (long long)n0 * n1;
    if (tid >= ncol * 10) return;
    const long long col = tid / 10; const int q = (int)(tid % 10);
    const int i = (int)(col / n1), j = (int)(col % n1);
    const int F = (q < 9) ? q / 3 : 3, kind = (q < 9) ? q % 3 : 0;
    const double* f = (F == 0) ? T : ((F == 1) ? u : ((F == 2) ? v : rho));
    const int iu = min(i + 1, n0 - 1), id = max(i - 1, 0), ju = min(j + 1, n1 - 1), jd = max(j - 1, 0);
    const double* fc = f + col * nz;
    const double* fu = (kind == 1) ? f + ((long long)iu * n1 + j) * nz : f + ((long long)i * n1 + ju) * nz;
    const double* fd = (kind == 1) ? f + ((long long)id * n1 + j) * nz : f + ((long long)i * n1 + jd) * nz;
    const double span = (kind == 1) ? __dsub_rn(ax0[iu], ax0[id]) : __dsub_rn(ax1[ju], ax1[jd]);
    auto val = [&](int k) { return (kind == 0) ? fc[k] : __ddiv_rn(__dsub_rn(fu[k], fd[k]), span); };
    const bool shifted = glob && kind != 0;                       // the Global file's dfdt[i] - dfdt[i+1] slip (App. A-9)
    double* o; int os, slope_at, value_at;
    if (F < 3) { o = tuv + col * nz * MS_STRIDE + MS_FIELD * F; os = MS_STRIDE; slope_at = 1 + kind; value_at = (kind == 0) ? 0 : 3 + kind; }
    else       { o = rh + col * nz * 2; os = 2; slope_at = 1; value_at = 0; }
    // forward sweep: d' parked in the slope slot
    double vm = val(0), vc = val(1), vp;
    o[value_at] = vm;
    double nd = __ddiv_rn(__ddiv_rn(__dmul_rn(3.0, __dsub_rn(vc, vm)), za.P2HI[0]), za.DEN[0]);       // di / bi
    o[slope_at] = nd;
    for (int k = 1; k < nz - 1; k++) {
        vp = val(k + 1);
        o[(size_t)k * os + value_at] = vc;
        const double lo = shifted ? __dsub_rn(vc, vp) : __dsub_rn(vc, vm);
        const double di = __dmul_rn(3.0, __dadd_rn(__ddiv_rn(lo, za.P2LO[k]), __ddiv_rn(__dsub_rn(vp, vc), za.P2HI[k])));
        nd = __ddiv_rn(__dsub_rn(di, __dmul_rn(nd, za.A[k])), za.DEN[k]);
        o[(size_t)k * os + slope_at] = nd;
        vm = vc; vc = vp;
    }
    {
        const int k = nz - 1;
        o[(size_t)k * os + value_at] = vc;
        const double di = __ddiv_rn(__dmul_rn(3.0, __dsub_rn(vc, vm)), za.P2LO[k]);
        nd = __ddiv_rn(__dsub_rn(di, __dmul_rn(nd, za.A[k])), za.DEN[k]);
        o[(size_t)k * os + slope_at] = nd;
    }
    // back substitution in place
    double sn = nd;
    for (int k = nz - 2; k >= 0; k--) {
        sn = __dsub_rn(o[(size_t)k * os + slope_at], __dmul_rn(za.NC[k], sn));
        o[(size_t)k * os + slope_at] = sn;
    }
}

static void build_zaux(const std::vector<double>& z, std::vector<double>& aux) {     // [A | DEN | NC | P2LO | P2HI], nz each
    const int n = (int)z.size();
    aux.assign((size_t)5 * n, 0.0);
    double *A = aux.data(), *DEN = A + n, *NC = DEN + n, *P2LO = NC + n, *P2HI = P2LO + n;
    double ai, bi, ci;
    bi = 2.0 / (z[1] - z[0]); ci = 1.0 / (z[1] - z[0]);
    DEN[0] = bi; NC[0] = ci / bi; P2HI[0] = std::pow(z[1] - z[0], 2);
    for (int i = 1; i < n - 1; i++) {
        ai = 1.0 / (z[i] - z[i - 1]);
        bi = 2.0 * (1.0 / (z[i] - z[i - 1]) + 1.0 / (z[i + 1] - z[i]));
        ci = 1.0 / (z[i + 1] - z[i]);
        A[i] = ai; DEN[i] = bi - NC[i - 1] * ai; NC[i] = ci / DEN[i];
        P2LO[i] = std::pow(z[i] - z[i - 1], 2); P2HI[i] = std::pow(z[i + 1] - z[i], 2);
    }
    ai = 1.0 / (z[n - 1] - z[n - 2]); bi = 2.0 / (z[n - 1] - z[n - 2]);
    A[n - 1] = ai; DEN[n - 1] = bi - NC[n - 2] * ai; P2LO[n - 1] = std::pow(z[n - 1] - z[n - 2], 2);
}

extern "C" int geoac_set_atmosphere_3d(geoac_ctx* ctx, int n0, int n1, int nz, const double* ax0, const double* ax1, const double* axz,
                                       const double* T, const double* u, const double* v, const double* rho) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    if (ctx->variant != GEOAC_3D_RNGDEP && ctx->variant != GEOAC_GLOBAL_RNGDEP)
        return fail(ctx, GEOAC_ERR_BAD_ARG, "variant needs geoac_set_atmosphere_1d");
    if (n0 < 2 || n1 < 2 || nz < 3 || !ax0 || !ax1 || !axz || !T || !u || !v || !rho)
        return fail(ctx, GEOAC_ERR_BAD_ARG, "need >= 2 x 2 x 3 nodes and non-null arrays");
    for (int i = 1; i < n0; i++) if (!(ax0[i] > ax0[i - 1])) return fail(ctx, GEOAC_ERR_BAD_ARG, "axis 0 must be strictly increasing");
    for (int i = 1; i < n1; i++) if (!(ax1[i] > ax1[i - 1])) return fail(ctx, GEOAC_ERR_BAD_ARG, "axis 1 must be strictly increasing");
    for (int i = 1; i < nz; i++) if (!(axz[i] > axz[i - 1])) return fail(ctx, GEOAC_ERR_BAD_ARG, "altitudes must be strictly increasing");
    const size_t nodes = (size_t)n0 * n1 * nz;
    if (nodes * MS_STRIDE >= (size_t)1 << 32) return fail(ctx, GEOAC_ERR_TOO_LARGE, "grid exceeds 2^32/18 nodes (32-bit element offsets in the kernel)");
    cudaSetDevice(ctx->device);
    const bool glob = ctx->variant == GEOAC_GLOBAL_RNGDEP;
    std::vector<double> z(nz);
    for (int k = 0; k < nz; k++) z[k] = axz[k] + (glob ? kREarth : 0.0);                     // r_vals[nr] += r_earth
    // build into fresh buffers and swap them in only after every step succeeded (a failed call -- e.g. out of memory on a
    // config-5-size grid -- leaves the previous atmosphere, or "none", fully intact)
    Buf<double> n_tuv, n_rho, n_ax;
    auto bail = [&](const std::string& what) {
        return fail(ctx, GEOAC_ERR_CUDA, "geoac_set_atmosphere_3d: " + what + ": " + cudaGetErrorString(cudaGetLastError()));
    };
    if (n_tuv.grow(nodes * MS_STRIDE * sizeof(double)) != cudaSuccess) return bail("node tables");
    if (n_rho.grow(nodes * 2 * sizeof(double)) != cudaSuccess) return bail("density table");
    std::vector<double> r0, r1, rz;
    build_axis_records(ax0, n0, r0); build_axis_records(ax1, n1, r1); build_axis_records(z.data(), nz, rz);
    if (n_ax.grow((size_t)(n0 + n1 + nz) * AX * sizeof(double)) != cudaSuccess) return bail("axis records");
    if (ctx->knobs.host_tables) {                                          // tests: build the tables on the host instead
        std::vector<double> zz, tuv, rh;
        build_grid_tables(glob, n0, n1, nz, ax0, ax1, axz, T, u, v, rho, zz, tuv, rh);
        if (cudaMemcpy(n_tuv.p, tuv.data(), tuv.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess
            || cudaMemcpy(n_rho.p, rh.data(), rh.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) return bail("table upload");
    } else {
        // raw fields + axis-only coefficients up, slopes and node differences built in HBM
        std::vector<double> aux; build_zaux(z, aux);
        Buf<double> f_buf, aux_buf;                                        // freed once the tables are built
        if (f_buf.grow(nodes * 4 * sizeof(double)) != cudaSuccess) return bail("raw fields");
        if (aux_buf.grow((aux.size() + n0 + n1) * sizeof(double)) != cudaSuccess) return bail("axis coefficients");
        double *d_f = f_buf.p, *d_aux = aux_buf.p;
        const double* src[4] = { T, u, v, rho };
        cudaError_t e = cudaSuccess;
        for (int F = 0; F < 4 && e == cudaSuccess; F++) e = cudaMemcpy(d_f + (size_t)F * nodes, src[F], nodes * sizeof(double), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(d_aux, aux.data(), aux.size() * sizeof(double), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(d_aux + aux.size(), ax0, n0 * sizeof(double), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMemcpy(d_aux + aux.size() + n0, ax1, n1 * sizeof(double), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) {
            ZAux za; za.A = d_aux; za.DEN = d_aux + nz; za.NC = d_aux + 2 * (size_t)nz; za.P2LO = d_aux + 3 * (size_t)nz; za.P2HI = d_aux + 4 * (size_t)nz;
            const long long nthreads = (long long)n0 * n1 * 10;
            grid_tables_kernel<<<(unsigned)((nthreads + 127) / 128), 128, 0, ctx->stream>>>(glob ? 1 : 0, n0, n1, nz, d_aux + aux.size(), d_aux + aux.size() + n0, za,
                                                                                           d_f, d_f + nodes, d_f + 2 * nodes, d_f + 3 * nodes, n_tuv.p, n_rho.p);
            e = cudaGetLastError();
            if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        }
        if (e != cudaSuccess) return bail("table build");
    }
    if (cudaMemcpy(n_ax.p, r0.data(), r0.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess
        || cudaMemcpy(n_ax.p + (size_t)n0 * AX, r1.data(), r1.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess
        || cudaMemcpy(n_ax.p + (size_t)(n0 + n1) * AX, rz.data(), rz.size() * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) return bail("axis upload");
    cudaStreamSynchronize(ctx->stream);                                          // no launch may still read the old tables
    ctx->d_tuv = std::move(n_tuv); ctx->d_rho = std::move(n_rho); ctx->d_ax = std::move(n_ax);
    Grid3D& g = ctx->grid;
    g.tuv = ctx->d_tuv.p; g.rho = ctx->d_rho.p; g.ax0 = ctx->d_ax.p; g.ax1 = ctx->d_ax.p + (size_t)n0 * AX; g.axz = ctx->d_ax.p + (size_t)(n0 + n1) * AX;
    g.n0 = n0; g.n1 = n1; g.nz = nz; g.scratch = nullptr; g.role = 0; g.nrole = 1; g.glane0 = 0; g.gmask = 0;
    g.amin = ax0[0]; g.amax = ax0[n0 - 1]; g.bmin = ax1[0]; g.bmax = ax1[n1 - 1]; g.zmin = z[0]; g.zmax = z[nz - 1];
    // GeoAc_SetPropRegion: G2S_MultiDimSpline3D.cpp:22-33 / G2S_GlobalMultiDimSpline3D.cpp:22-33
    ctx->prm.vert_limit = g.zmax;
    ctx->prm.box_min[0] = g.amin; ctx->prm.box_max[0] = g.amax; ctx->prm.box_min[1] = g.bmin; ctx->prm.box_max[1] = g.bmax;
    if (glob && !ctx->src_set) {      // GeoAcGlobal.RngDep_main.cpp:135-137: default source = grid midpoint
        ctx->prm.src[1] = (g.amin + g.amax) / 2.0; ctx->prm.src[2] = (g.bmin + g.bmax) / 2.0;
    }
    ctx->is_grid = true; ctx->have_atmo = true; ctx->consts_dirty = true;
    return GEOAC_OK;
}

// Test hook: the node tables as the kernels read them (tuv[n0][n1][nz][18], rho[n0][n1][nz][2]; mspline.cuh).
extern "C" int geoac_get_grid_tables(geoac_ctx* ctx, int64_t cap_tuv, double* tuv, int64_t cap_rho, double* rho) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    if (!ctx->is_grid || !ctx->d_tuv.p) return fail(ctx, GEOAC_ERR_NO_ATMO, "no range-dependent atmosphere set");
    const size_t nodes = (size_t)ctx->grid.n0 * ctx->grid.n1 * ctx->grid.nz;
    if (!tuv || !rho || (size_t)cap_tuv < nodes * MS_STRIDE || (size_t)cap_rho < nodes * 2) return fail(ctx, GEOAC_ERR_BAD_ARG, "get_grid_tables: buffers too small");
    cudaSetDevice(ctx->device);
    CK(cudaMemcpy(tuv, ctx->d_tuv.p, nodes * MS_STRIDE * sizeof(double), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(rho, ctx->d_rho.p, nodes * 2 * sizeof(double), cudaMemcpyDeviceToHost));
    return GEOAC_OK;
}

// ---- per-launch invariants, computed on the device with the same spline routines the kernel uses ----
__global__ void setup_consts_kernel(LaunchConsts* out, const LaunchConsts in, const double* table, int n,
                                    double xmin, double xmax, int variant) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    Table1D T; T.base = table; T.n = n; T.xmin = xmin; T.xmax = xmax; T.jump_scale = 0.0;
    LaunchConsts L = in;
    fill_launch_consts_1d(L, T, variant);
    *out = L;
}

// per-interval absorption polynomials (core.cuh: sbpoly_build_interval), one thread per interval, after the invariants
__global__ void build_sbpoly_kernel(const LaunchConsts* Lc, const double* table, int n, double xmin, double xmax, int glob, double* out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n - 1) return;
    Table1D T; T.base = table; T.n = n; T.xmin = xmin; T.xmax = xmax; T.jump_scale = 0.0; T.sbpoly = nullptr;
    double o[SBP_STRIDE];
    sbpoly_build_interval(*Lc, T, glob != 0, k, o);
    for (int i = 0; i < SBP_STRIDE; i++) out[(size_t)k * SBP_STRIDE + i] = o[i];
}

__global__ void setup_consts_grid_kernel(LaunchConsts* out, const LaunchConsts in, const Grid3D g, int variant) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    LaunchConsts L = in;
    fill_launch_consts_3d(L, g, variant);
    *out = L;
}

static int refresh_consts(geoac_ctx* ctx) {
    if (!ctx->have_atmo) return fail(ctx, GEOAC_ERR_NO_ATMO, "set an atmosphere first");      // the set-up kernel samples the tables
    if (!ctx->consts_dirty) return GEOAC_OK;
    const geoac_params& p = ctx->prm;
    LaunchConsts L; std::memset(&L, 0, sizeof L);
    L.ds_min = p.ds_min; L.ds_max = p.ds_max; L.vert_limit = p.vert_limit; L.range_limit = p.range_limit;
    L.z_grnd = p.z_grnd; L.tweak_abs = p.tweak_abs; L.freq = p.freq;
    for (int i = 0; i < 2; i++) { L.box_min[i] = p.box_min[i]; L.box_max[i] = p.box_max[i]; }
    for (int i = 0; i < 3; i++) L.src[i] = p.src[i];
    if (ctx->variant == GEOAC_2D || ctx->variant == GEOAC_3D || ctx->variant == GEOAC_3D_RNGDEP) L.src[2] = std::max(p.z_grnd, p.src[2]);   // z_src = max(z_grnd, z_src)
    else L.src[0] = std::max(p.z_grnd, p.src[0]);
    L.bounces = p.bounces; L.calc_amp = p.calc_amp;
    L.seg_mode = (ctx->variant == GEOAC_2D) ? 1 : (p.accum_per_segment ? 1 : 0);                          // App. A-2
    L.step_limit = (int)(p.ray_limit * (int)(1.0 / (p.ds_min * 10)));                                     // Solver.cpp:14
    L.per_bounce_zmax = (ctx->variant == GEOAC_3D_RNGDEP || ctx->variant == GEOAC_GLOBAL_RNGDEP);         // App. A-3
    if (ctx->is_grid) setup_consts_grid_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_consts.p, L, ctx->grid, ctx->variant);
    else {
        setup_consts_kernel<<<1, 32, 0, ctx->stream>>>(ctx->d_consts.p, L, ctx->d_table.p, ctx->n, ctx->xmin, ctx->xmax, ctx->variant);
        build_sbpoly_kernel<<<(ctx->n - 1 + 63) / 64, 64, 0, ctx->stream>>>(ctx->d_consts.p, ctx->d_table.p, ctx->n, ctx->xmin, ctx->xmax,
                                                                            ctx->variant == GEOAC_GLOBAL, ctx->d_sbpoly.p);
    }
    CK(cudaGetLastError());
    ctx->consts_dirty = false;
    return GEOAC_OK;
}

// ---- kernel launch ----
// cost scout: predicted RK4 step counts of the rays into ctx->d_cost, their maximum and sum.  Persistent, the table in shared
// memory when it fits.
template <class SEQ>
static int launch_cost_scout(geoac_ctx* ctx, const TraceArgs& a, int max_optin, cudaStream_t st, uint32_t* cmax, unsigned long long* cost_sum) {
    constexpr bool kGrid = PacketMode<SEQ>::value;
    constexpr int kScoutBlock = ScoutBlock<SEQ>::value;
    const size_t s_tab = kGrid ? 0 : 16 + (size_t)TAB_NARR * ctx->n * sizeof(double);
    const bool s_in = !kGrid && s_tab <= (size_t)max_optin;
    const void* sfn;
    if constexpr (kGrid) sfn = (const void*)scout_kernel<SEQ, false>;
    else sfn = s_in ? (const void*)scout_kernel<SEQ, true> : (const void*)scout_kernel<SEQ, false>;
    const size_t s_smem = s_in ? s_tab : 16;
    CK(cudaFuncSetAttribute(sfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s_smem));
    int s_per_sm = 1;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&s_per_sm, sfn, kScoutBlock, s_smem));
    const int sblocks = (int)std::min<int64_t>((int64_t)ctx->sm_count * std::max(1, s_per_sm), (a.n_rays + kScoutBlock - 1) / kScoutBlock);
    unsigned long long* scounter = ctx->d_counters.p + 3;
    int coarse = ctx->knobs.scout_coarse > 0 ? ctx->knobs.scout_coarse : (kGrid ? kScoutCoarse : 2 * kScoutCoarse);   // stratified: 32x measured best (404.8 vs 421.0 / 443.3 ms at 16x / 64x)
    void* sargs[] = { (void*)&a, (void*)&ctx->d_cost.p, (void*)&cmax, (void*)&cost_sum, (void*)&scounter, (void*)&coarse };
    CK(cudaLaunchKernel(sfn, dim3(sblocks), dim3(kScoutBlock), sargs, s_smem, st));
    ctx->last_launches += 1;
    return GEOAC_OK;
}

// Step 1: the longest-predicted-ray-first claim order (trace_kernel.cuh): cost scout, (range-dependent sets) cost dilation, sort.
// Sets a.order, a.n_claims, a.packet_refill and a.n_long_packets; n_quarter = long packets long enough for quarter claims.
// `lanes` = lanes of the main launch (the average work of a lane is the scout's cost sum over them).
template <class EQ>
static int build_claim_order(geoac_ctx* ctx, TraceArgs& a, long long lanes, int max_optin, cudaStream_t st, int64_t& n_quarter) {
    constexpr bool kGrid = PacketMode<EQ>::value;
    constexpr int group = kGrid ? 32 : 1;                     // range-dependent sets: packets of 32 consecutive rays
    const int64_t n = a.n_rays, n_entries = ((n + group - 1) / group) * group;
    const size_t ids = sizeof(uint32_t) * n_entries;
    // d_hist: [0..255] buckets, [256] largest cost, [257] long packets, [258] quarter packets, [260..261] cost sum (64 bit)
    const size_t hist_bytes = sizeof(uint32_t) * (kCostBuckets + 8);
    CK(ctx->d_cost.grow(ids)); CK(ctx->d_order.grow(ids)); CK(ctx->d_hist.grow(hist_bytes));
    CK(cudaMemsetAsync(ctx->d_hist.p, 0, hist_bytes, st));
    uint32_t* cmax = ctx->d_hist.p + kCostBuckets;
    uint32_t* n_long = cmax + 1;                              // n_long[1]: quarter packets
    unsigned long long* cost_sum = reinterpret_cast<unsigned long long*>(cmax + 4);
    if (int rc = launch_cost_scout<typename EQ::Scout>(ctx, a, max_optin, st, cmax, cost_sum)) return rc;
    if (kGrid) {
        const uint32_t* cost = ctx->d_cost.p;
        if (ctx->knobs.dilate > 0) {
            // the estimate used for the claim order: maximum over the inclination neighbours (trace_kernel.cuh: cost_dilate_kernel)
            CK(ctx->d_cost_dilated.grow(ids));
            cost_dilate_kernel<<<ctx->sm_count * 2, 256, 0, st>>>(ctx->d_cost.p, a.theta, n, ctx->knobs.dilate * 1e-3 * kPi / 180.0, 16, ctx->d_cost_dilated.p);
            cost = ctx->d_cost_dilated.p;
            ctx->last_launches += 1;
        }
        // packets by cost bucket, longest first; also counts the long and the quarter packets
        order_hist_kernel<<<ctx->sm_count, 256, 0, st>>>(cost, n, group, cmax, ctx->d_hist.p, cost_sum, lanes, n_long, ctx->knobs.long_alpha, n_long + 1, ctx->knobs.quarter_alpha);
        order_scan_kernel<<<1, kCostBuckets, 0, st>>>(ctx->d_hist.p);
        order_scatter_kernel<<<ctx->sm_count, 256, 0, st>>>(cost, n, group, cmax, ctx->d_hist.p, ctx->d_order.p);
        ctx->last_launches += 3;
    } else {
        // order by (cost bucket, inclination, batch index) + whole-warp refill: a warp's lanes then read the same few table
        // records (trace_kernel.cuh).  Two stable counting-sort passes, inclination first.
        const int nblk = ctx->sm_count;
        const int64_t chunk = (n + nblk - 1) / nblk;
        CK(ctx->d_blockhist.grow(sizeof(uint32_t) * (size_t)nblk * kCostBuckets + 2 * sizeof(double)));
        CK(ctx->d_keys.grow((size_t)2 * n)); CK(ctx->d_order2.grow(ids));
        double* trange = reinterpret_cast<double*>(ctx->d_blockhist.p + (size_t)nblk * kCostBuckets);
        uint8_t *key_t = ctx->d_keys.p, *key_c = ctx->d_keys.p + n;
        order_theta_range_kernel<<<1, 1024, 0, st>>>(a.theta, n, trange);
        order_keys_kernel<<<ctx->sm_count, 256, 0, st>>>(ctx->d_cost.p, a.theta, n, cmax, trange, key_t, key_c, ctx->knobs.cost_shift);
        auto pass = [&](const uint8_t* key, const uint32_t* src, uint32_t* dst) {
            stable_hist_kernel<<<nblk, 256, 0, st>>>(key, src, n, chunk, ctx->d_blockhist.p);
            stable_scan_kernel<<<1, kCostBuckets, 0, st>>>(ctx->d_blockhist.p, nblk);
            stable_scatter_kernel<<<nblk, 32, 0, st>>>(key, src, n, chunk, ctx->d_blockhist.p, dst);
        };
        pass(key_t, nullptr, ctx->d_order2.p);
        pass(key_c, ctx->d_order2.p, ctx->d_order.p);
        ctx->last_launches += 8;
        a.packet_refill = 1;
    }
    CK(cudaGetLastError());
    a.n_claims = n_entries;
    a.order = ctx->d_order.p;
    n_quarter = 0;
    if (kGrid && ctx->knobs.coop) {
        // the long region: packets that would outlast the pass on a fully loaded SM.  Their count sizes the second launch.
        uint32_t h[2] = { 0, 0 };
        CK(cudaMemcpyAsync(h, n_long, sizeof h, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        a.n_long_packets = std::min<int64_t>(h[0], n_entries / 32);
        n_quarter = h[1];
    }
    return GEOAC_OK;
}

// Step 2: CTAs of the exclusive long-region launch (0 = none: one launch, whose warps claim the main region first, then the
// long region, then the quarter packets -- trace_kernel.cuh).  Sets a.n_quarter_packets.  The capture kernels always run as
// one launch.
static int size_long_region(const geoac_ctx* ctx, TraceArgs& a, int64_t n_quarter, int block, bool paths) {
    if (a.n_long_packets == 0 || !ctx->knobs.exclusive || paths) return 0;
    const int64_t max_ctas = std::max<int64_t>(1, (int64_t)ctx->sm_count * ctx->knobs.long_sm_pct / 100);
    if (!ctx->knobs.quarter) return (int)std::max<int64_t>(1, std::min<int64_t>((a.n_long_packets * 32 + block - 1) / block, max_ctas));
    // The very longest packets set the length of the pass: even alone on its scheduler a warp needs ~60 us per step of its
    // 32 rays.  Packets whose cost exceeds quarter_alpha % of the average lane work (they would outlast the pass even at
    // lone-warp speed) are split over four warps -- quarter claims, four lanes per ray, ~40 us per step -- as far as the
    // exclusive SMs have warps to spare.  Measured on one GPU's share of the 8-way config-5 split: 31.4 s -> 22.2 s.
    const int64_t warps = max_ctas * (block / 32);
    a.n_quarter_packets = std::min<int64_t>(std::min<int64_t>(a.n_long_packets, n_quarter), std::max<int64_t>(0, (warps - a.n_long_packets) / 3));
    return (int)std::min<int64_t>(max_ctas, (a.n_long_packets + 3 * a.n_quarter_packets + (block / 32) - 1) / (block / 32));
}

// Step 3: the trace launch(es).  With a long region of its own, two concurrent launches of the same kernel: the long region
// -- packets that would outlast the pass on a loaded SM -- goes to CTAs that keep their SM to themselves (their
// shared-memory request leaves no room for a main CTA), launched first on a high-priority stream; the main launch fills the
// other SMs, and its surplus CTAs start as SMs free up.  Each side drains its own region first and then helps with the other.
template <class EQ, int BLOCK>
static int enqueue_launches(geoac_ctx* ctx, const void* fn, size_t smem, int max_optin, int grid, int grid_long, TraceArgs a, cudaStream_t st) {
    if (grid_long > 0) {
        const size_t smem_long = std::min((size_t)max_optin, std::max(smem, (size_t)max_optin - smem + 4096));
        CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_long));
        TraceArgs al = a;
        al.prefer_long = 1;
        if (NeedsPrev<EQ>::value) {                          // y_{k-1} scratch of both launches, the long one's after the main one's
            const size_t main_doubles = (size_t)EQ::NEQ * grid * BLOCK;
            const size_t need = (main_doubles + (size_t)EQ::NEQ * grid_long * BLOCK) * sizeof(double);
            if (need > ctx->d_prev.cap) {
                CK(cudaStreamSynchronize(st));                // a trace still running may use the old scratch
                CK(ctx->d_prev.grow(need));
            }
            a.prev = ctx->d_prev.p;
            al.prev = ctx->d_prev.p + main_doubles;
        }
        CK(cudaEventRecord(ctx->ev_fork, st));
        CK(cudaStreamWaitEvent(ctx->stream_long, ctx->ev_fork, 0));
        void* largs[] = { (void*)&al };
        CK(cudaEventRecord(ctx->ev_l0, ctx->stream_long));
        CK(cudaLaunchKernel(fn, dim3(grid_long), dim3(BLOCK), largs, smem_long, ctx->stream_long));
        CK(cudaEventRecord(ctx->ev_l1, ctx->stream_long));
        CK(cudaEventRecord(ctx->ev_join, ctx->stream_long));
        ctx->last_launches += 1; ctx->last_long_ctas = grid_long;
    }
    void* args[] = { (void*)&a };
    CK(cudaEventRecord(ctx->ev_m0, st));
    CK(cudaLaunchKernel(fn, dim3(grid), dim3(BLOCK), args, smem, st));
    CK(cudaEventRecord(ctx->ev_m1, st));
    ctx->timed_launches = true;
    if (grid_long > 0) CK(cudaStreamWaitEvent(st, ctx->ev_join, 0));
    ctx->last_launches += 1;
    return GEOAC_OK;
}

template <class EQ, int BLOCK, bool PATHS>
static int launch_trace(geoac_ctx* ctx, TraceArgs a, cudaStream_t st) {
    constexpr bool kGrid = PacketMode<EQ>::value;
    const size_t lane_doubles = ((size_t)LaneLayout<EQ>::STRIDE * BLOCK + 1) & ~(size_t)1;
    const size_t fixed = ((sizeof(LaunchConsts) + 15) / 16) * 16 + 16 + lane_doubles * sizeof(double);
    const size_t tab_bytes = kGrid ? 0 : (size_t)TAB_NARR * ctx->n * sizeof(double);
    int max_optin = 0;
    CK(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, ctx->device));
    if (fixed > (size_t)max_optin) return fail(ctx, GEOAC_ERR_CUDA, "lane records do not fit in shared memory");
    const bool in_smem = !kGrid && fixed + tab_bytes <= (size_t)max_optin;
    const size_t smem = in_smem ? fixed + tab_bytes : fixed;
    // the range-dependent node tables, and a profile too large for shared memory, are read through L1 / L2
    const void* fn;
    if constexpr (kGrid) fn = (const void*)trace_kernel<EQ, BLOCK, false, PATHS>;
    else fn = in_smem ? (const void*)trace_kernel<EQ, BLOCK, true, PATHS> : (const void*)trace_kernel<EQ, BLOCK, false, PATHS>;
    CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, BLOCK, smem));
    if (per_sm < 1) return fail(ctx, GEOAC_ERR_CUDA, "trace kernel does not fit on an SM");
    // persistent grid: every resident CTA slot of every SM, but never more lanes than rays
    const int64_t warps_needed = (a.n_rays + 31) / 32;
    const int64_t ctas_needed = std::max<int64_t>(1, (warps_needed + (BLOCK / 32) - 1) / (BLOCK / 32));
    const int grid = (int)std::min<int64_t>((int64_t)ctx->sm_count * per_sm, ctas_needed);
    if (NeedsPrev<EQ>::value) CK(ctx->d_prev.grow((size_t)EQ::NEQ * grid * BLOCK * sizeof(double)));
    a.prev = ctx->d_prev.p;
    a.order = nullptr; a.n_claims = a.n_rays; a.n_long_packets = 0; a.n_quarter_packets = 0; a.counter_long = ctx->d_counters.p + 4; a.counter_quarter = ctx->d_counters.p + 5;
    a.prefer_long = 0; a.packet_refill = 0;
    ctx->last_launches = 0; ctx->last_long_packets = 0; ctx->last_long_ctas = 0; ctx->last_quarter_packets = 0;
    int grid_long = 0;
    // longest-predicted-ray-first claim order, when a lane will process more than one ray (see trace_kernel.cuh)
    // knob lpt: 0 = natural order, 1 = automatic (default), 2 = always (used by the tests on small batches)
    const int lpt_mode = ctx->knobs.lpt;
    if ((lpt_mode == 2 || (lpt_mode == 1 && a.n_rays > (int64_t)grid * BLOCK)) && a.n_rays < ((int64_t)1 << 32)) {
        int64_t n_quarter = 0;
        if (int rc = build_claim_order<EQ>(ctx, a, (long long)grid * BLOCK, max_optin, st, n_quarter)) return rc;
        grid_long = size_long_region(ctx, a, n_quarter, BLOCK, PATHS);
    }
    ctx->last_long_packets = (int)a.n_long_packets;
    ctx->last_quarter_packets = (int)a.n_quarter_packets;
    return enqueue_launches<EQ, BLOCK>(ctx, fn, smem, max_optin, grid, grid_long, a, st);
}

// variant -> (equation set, lanes per CTA); PATHS: the raypath / caustic capture kernels (same lanes per SM as the plain ones)
template <bool PATHS>
static int dispatch_trace(geoac_ctx* ctx, const TraceArgs& a, cudaStream_t st) {
    const bool amp = ctx->prm.calc_amp != 0;
    switch (ctx->variant) {
        case GEOAC_2D:     return amp ? launch_trace<Eq2D<true>, 512, PATHS>(ctx, a, st) : launch_trace<Eq2D<false>, 512, PATHS>(ctx, a, st);
        // Eq3D<true>: 384 lanes = 3 warps per scheduler at <= 168 registers, no spills (420 ms per config-2 pass vs 491 (256) /
        // 494 (512) in round 1).  Nothing in between exists: the register file is four 16 K-register banks, one per scheduler, so
        // 13 or 14 warps put 4 on some scheduler and cap every lane at 128 registers -- the 512-lane case, which spills (measured
        // on B200: 416 / 448 lanes at 152 / 144 registers compile without spills but do not fit on an SM).
        case GEOAC_3D:     return amp ? launch_trace<Eq3D<true>, 384, PATHS>(ctx, a, st) : launch_trace<Eq3D<false>, 512, PATHS>(ctx, a, st);
        case GEOAC_GLOBAL: return amp ? launch_trace<EqGlobal<true>, 384, PATHS>(ctx, a, st) : launch_trace<EqGlobal<false>, 512, PATHS>(ctx, a, st);
        case GEOAC_3D_RNGDEP:     return amp ? launch_trace<Eq3DRD<true>, 128, PATHS>(ctx, a, st)     : launch_trace<Eq3DRD<false>, 128, PATHS>(ctx, a, st);
        case GEOAC_GLOBAL_RNGDEP: return amp ? launch_trace<EqGlobalRD<true>, 128, PATHS>(ctx, a, st) : launch_trace<EqGlobalRD<false>, 128, PATHS>(ctx, a, st);
    }
    return fail(ctx, GEOAC_ERR_BAD_ARG, "variant not implemented");
}

// One trace on `st`: zeroes the records and counters, fills in the context's part of `a` and launches.  The caller sets the
// rays (theta, phi, n_rays) and their outputs (rec, status, n_steps), and the capture fields (zero: no capture).  The launch
// invariants must be current (refresh_consts) and ordered before `st`.
static int enqueue_trace(geoac_ctx* ctx, TraceArgs a, cudaStream_t st) {
    const int n_rec = ctx->prm.bounces + 1;
    const int64_t n_slots = a.n_rays * n_rec;
    CK(cudaMemsetAsync(ctx->d_counters.p, 0, 8 * sizeof(unsigned long long), st));
    CK(cudaMemsetAsync(a.rec, 0, sizeof(double) * GEOAC_NFIELDS * n_slots, st));
    CK(cudaMemsetAsync(a.status, 0, sizeof(int32_t) * n_slots, st));
    CK(cudaMemsetAsync(a.n_steps, 0, sizeof(int32_t) * n_slots, st));
    a.grid = ctx->grid;
    a.table = ctx->d_table.p; a.table_n = ctx->n; a.table_xmin = ctx->xmin; a.table_xmax = ctx->xmax;
    a.sbpoly = (ctx->is_grid || !ctx->knobs.sbpoly) ? nullptr : ctx->d_sbpoly.p;   // knob sbpoly = 0: the full absorption model at every step (A/B measurements, tests)
    a.consts = ctx->d_consts.p; a.n_rec = n_rec;
    a.counter = ctx->d_counters.p; a.total_steps = ctx->d_counters.p + 1; a.warp_trips = ctx->d_counters.p + 2;
    return (a.path_stride > 0 || a.caus_cap > 0) ? dispatch_trace<true>(ctx, a, st) : dispatch_trace<false>(ctx, a, st);
}

extern "C" int geoac_trace_device(geoac_ctx* ctx, int64_t n_rays, const double* d_theta, const double* d_phi,
                                  double* d_rec, int32_t* d_status, int32_t* d_n_steps, void* cuda_stream) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    if (n_rays < 0) return fail(ctx, GEOAC_ERR_BAD_ARG, "geoac_trace_device: n_rays < 0");
    if (n_rays == 0) return GEOAC_OK;
    if (!d_theta || !d_phi || !d_rec || !d_status || !d_n_steps) return fail(ctx, GEOAC_ERR_BAD_ARG, "geoac_trace_device: null buffer");
    if (!ctx->have_atmo) return fail(ctx, GEOAC_ERR_NO_ATMO, "set an atmosphere first");
    cudaSetDevice(ctx->device);
    if (int rc = refresh_consts(ctx)) return rc;
    const cudaStream_t st = (cudaStream_t)cuda_stream;
    if (st != ctx->stream) {       // consts were written on ctx->stream: order the caller's stream after it
        CK(cudaEventRecord(ctx->ev0, ctx->stream));
        CK(cudaStreamWaitEvent(st, ctx->ev0, 0));
    }
    TraceArgs a{};
    a.theta = d_theta; a.phi = d_phi; a.n_rays = n_rays; a.rec = d_rec; a.status = d_status; a.n_steps = d_n_steps;
    ctx->last_ms = std::numeric_limits<double>::quiet_NaN(); ctx->ms_pending = false;
    CK(cudaEventRecord(ctx->ev_d0, st));
    if (int rc = enqueue_trace(ctx, a, st)) return rc;
    CK(cudaEventRecord(ctx->ev_d1, st));
    ctx->ms_pending = true;                                 // read by geoac_last_trace_stats once the stream has got there
    return GEOAC_OK;
}

// device staging of the host-buffer entry point (angles in, records out), grown on demand and kept across calls
static int reserve_staging(geoac_ctx* ctx, int64_t n_rays) {
    const size_t n_slots = (size_t)n_rays * (ctx->prm.bounces + 1);
    CK(ctx->d_theta.grow(sizeof(double) * n_rays)); CK(ctx->d_phi.grow(sizeof(double) * n_rays));
    CK(ctx->d_rec.grow(sizeof(double) * GEOAC_NFIELDS * n_slots));
    CK(ctx->d_status.grow(sizeof(int32_t) * n_slots)); CK(ctx->d_nsteps.grow(sizeof(int32_t) * n_slots));
    return GEOAC_OK;
}

extern "C" void* geoac_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (bytes == 0 || cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void geoac_host_free(void* p) { if (p) { cudaFreeHost(p); cudaGetLastError(); } }

extern "C" int geoac_reserve(geoac_ctx* ctx, int64_t n_rays) {
    if (!ctx || n_rays < 0) return GEOAC_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    return reserve_staging(ctx, n_rays);
}

// ---- compacted raypath / caustic rows: only the rows produced cross PCIe ----
__global__ void compact_rows_kernel(const double* dense, const int32_t* rows, const int64_t* offs, int64_t n, int64_t cap, int nf, double* out) {
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (int64_t r = warp; r < n; r += nwarps) {
        const int64_t m = (rows[r] < cap ? rows[r] : cap) * nf;
        const double* src = dense + r * cap * nf;
        double* dst = out + offs[r] * nf;
        for (int64_t i = lane; i < m; i += 32) dst[i] = src[i];
    }
}

// What a host trace captures besides the records (none for geoac_trace).  Dense: data[ray][cap][nf] and the rows produced per
// ray in `rows` (rows past cap are counted, not kept).  Compact: the kept rows ray after ray in `data`, which has room for
// total_cap of them; ray i's run from offs[i] to offs[i + 1].
enum class Capture { none, dense, compact };
struct CaptureOut { int64_t cap = 0; double* data = nullptr; int32_t* rows = nullptr; int64_t* offs = nullptr; int64_t total_cap = 0; };

// The host-buffer trace (geoac_trace, geoac_trace_paths, geoac_trace_paths_compact, each context of geoac_trace_multi):
// angles in, one trace on ctx->stream, records out, plus the raypath rows (every path_stride steps) and caustic events asked for.
static int trace_host(geoac_ctx* ctx, int64_t n_rays, const double* theta, const double* phi, double* rec, int32_t* status, int32_t* n_steps,
                      Capture mode = Capture::none, int path_stride = 0, CaptureOut path = {}, CaptureOut caus = {}) {
    if (!ctx || n_rays < 0 || (n_rays > 0 && (!theta || !phi || !rec || !status || !n_steps))) return GEOAC_ERR_BAD_ARG;
    const bool compact = mode == Capture::compact;
    auto has_rows = [&](const CaptureOut& c) { return compact ? c.offs != nullptr : c.rows != nullptr; };
    if (mode != Capture::none && (path_stride < 0 || caus.cap < 0 || (path_stride == 0 && caus.cap == 0)))
        return fail(ctx, GEOAC_ERR_BAD_ARG, "ask for raypath rows (path_stride > 0) and / or caustic events (caustic_cap > 0)");
    if (path_stride > 0 && (path.cap <= 0 || !path.data || !has_rows(path)))
        return fail(ctx, GEOAC_ERR_BAD_ARG, compact ? "raypath capture needs its buffers and a positive per-ray capacity"
                                                    : "raypath capture needs path buffers and a positive row capacity");
    if (caus.cap > 0 && (!caus.data || !has_rows(caus))) return fail(ctx, GEOAC_ERR_BAD_ARG, "caustic capture needs its buffers");
    if (caus.cap > 0 && !ctx->prm.calc_amp) return fail(ctx, GEOAC_ERR_BAD_ARG, "caustic capture needs calc_amp = 1 (the Jacobian uses the auxiliary equations)");
    if ((path_stride > 0 || caus.cap > 0) && ctx->variant != GEOAC_2D && !ctx->prm.accum_per_segment)
        return fail(ctx, GEOAC_ERR_BAD_ARG, "raypath / caustic rows need accum_per_segment = 1 (the mains' WriteRays accumulation, SURVEY App. A-2)");
    if (compact && path_stride > 0) path.offs[0] = 0;
    if (compact && caus.cap > 0) caus.offs[0] = 0;
    if (n_rays == 0) return GEOAC_OK;
    if (!ctx->have_atmo) return fail(ctx, GEOAC_ERR_NO_ATMO, "set an atmosphere first");
    cudaSetDevice(ctx->device);
    const int64_t n_slots = n_rays * (ctx->prm.bounces + 1);
    if (int rc = reserve_staging(ctx, n_rays)) return rc;
    const cudaStream_t st = ctx->stream;
    // the captures asked for, staged dense in the context: [ray][cap][nf] and the row count of each ray
    struct Staged { const CaptureOut& out; Buf<double>& data; Buf<int32_t>& rows; int nf; const char* what; };
    std::vector<Staged> staged;
    if (path_stride > 0) staged.push_back({ path, ctx->d_path, ctx->d_path_rows, GEOAC_PATH_NF, "raypath rows" });
    if (caus.cap > 0) staged.push_back({ caus, ctx->d_caus, ctx->d_caus_rows, GEOAC_CAUSTIC_NF, "caustic rows" });
    for (const Staged& s : staged) {
        const size_t bytes = (size_t)n_rays * s.out.cap * s.nf * sizeof(double);
        CK(s.data.grow(bytes)); CK(s.rows.grow(sizeof(int32_t) * n_rays));
        if (!compact) CK(cudaMemsetAsync(s.data.p, 0, bytes, st));       // the caller receives every slot; compaction copies only rows produced
        CK(cudaMemsetAsync(s.rows.p, 0, sizeof(int32_t) * n_rays, st));
    }
    TraceArgs a{};
    a.theta = ctx->d_theta.p; a.phi = ctx->d_phi.p; a.n_rays = n_rays; a.rec = ctx->d_rec.p; a.status = ctx->d_status.p; a.n_steps = ctx->d_nsteps.p;
    if (path_stride > 0) { a.path = ctx->d_path.p; a.path_rows = ctx->d_path_rows.p; a.path_stride = path_stride; a.path_cap = path.cap; }
    if (caus.cap > 0) { a.caus = ctx->d_caus.p; a.caus_rows = ctx->d_caus_rows.p; a.caus_cap = caus.cap; }
    CK(cudaMemcpyAsync(ctx->d_theta.p, theta, sizeof(double) * n_rays, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_phi.p, phi, sizeof(double) * n_rays, cudaMemcpyHostToDevice, st));
    if (int rc = refresh_consts(ctx)) return rc;                         // before ev0: the timed window holds the trace alone
    CK(cudaEventRecord(ctx->ev0, st));
    if (int rc = enqueue_trace(ctx, a, st)) return rc;
    CK(cudaEventRecord(ctx->ev1, st));
    CK(cudaMemcpyAsync(rec, ctx->d_rec.p, sizeof(double) * GEOAC_NFIELDS * n_slots, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(status, ctx->d_status.p, sizeof(int32_t) * n_slots, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(n_steps, ctx->d_nsteps.p, sizeof(int32_t) * n_slots, cudaMemcpyDeviceToHost, st));
    std::vector<int32_t> h_rows;
    for (const Staged& s : staged) {
        const int64_t cap = s.out.cap;
        if (!compact) {
            CK(cudaMemcpyAsync(s.out.data, s.data.p, (size_t)n_rays * cap * s.nf * sizeof(double), cudaMemcpyDeviceToHost, st));
            CK(cudaMemcpyAsync(s.out.rows, s.rows.p, sizeof(int32_t) * n_rays, cudaMemcpyDeviceToHost, st));
            continue;
        }
        // per-ray row counts -> offsets on the host (n_rays integers), rows gathered on the device, only those copied out
        h_rows.resize((size_t)n_rays);
        CK(cudaMemcpyAsync(h_rows.data(), s.rows.p, sizeof(int32_t) * n_rays, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        int64_t* offs = s.out.offs;
        for (int64_t i = 0; i < n_rays; i++) offs[i + 1] = offs[i] + std::min<int64_t>(h_rows[(size_t)i], cap);
        const int64_t total = offs[n_rays];
        if (total > s.out.total_cap) return fail(ctx, GEOAC_ERR_TOO_LARGE, std::string(s.what) + ": " + std::to_string(total) + " rows produced, buffer holds "
                                                 + std::to_string(s.out.total_cap) + " (the offsets are filled in: the last one is the size to allocate)");
        if (total == 0) continue;
        Buf<int64_t> d_offs; Buf<double> d_out;                        // scratch of this call: nothing of it stays allocated
        CK(d_offs.grow(sizeof(int64_t) * (n_rays + 1))); CK(d_out.grow(sizeof(double) * total * s.nf));
        CK(cudaMemcpyAsync(d_offs.p, offs, sizeof(int64_t) * (n_rays + 1), cudaMemcpyHostToDevice, st));
        compact_rows_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(s.data.p, s.rows.p, d_offs.p, n_rays, cap, s.nf, d_out.p);
        CK(cudaMemcpyAsync(s.out.data, d_out.p, sizeof(double) * total * s.nf, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
    }
    unsigned long long cnt[2] = { 0, 0 };
    CK(cudaMemcpyAsync(cnt, ctx->d_counters.p, sizeof cnt, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
    ctx->last_ms = ms; ctx->ms_pending = false; ctx->last_steps = (int64_t)cnt[1];
    return GEOAC_OK;
}

extern "C" int geoac_trace(geoac_ctx* ctx, int64_t n_rays, const double* theta, const double* phi,
                           double* rec, int32_t* status, int32_t* n_steps) {
    return trace_host(ctx, n_rays, theta, phi, rec, status, n_steps);
}

extern "C" int geoac_trace_paths(geoac_ctx* ctx, int64_t n_rays, const double* theta, const double* phi,
                                 double* rec, int32_t* status, int32_t* n_steps,
                                 int path_stride, int64_t path_cap, double* path, int32_t* path_rows,
                                 int64_t caustic_cap, double* caustic, int32_t* caustic_rows) {
    return trace_host(ctx, n_rays, theta, phi, rec, status, n_steps, Capture::dense, path_stride,
                      { path_cap, path, path_rows }, { caustic_cap, caustic, caustic_rows });
}

extern "C" int geoac_trace_paths_compact(geoac_ctx* ctx, int64_t n_rays, const double* theta, const double* phi,
                                         double* rec, int32_t* status, int32_t* n_steps,
                                         int path_stride, int64_t path_cap, int64_t path_total_cap, double* path, int64_t* path_offset,
                                         int64_t caustic_cap, int64_t caustic_total_cap, double* caustic, int64_t* caustic_offset) {
    return trace_host(ctx, n_rays, theta, phi, rec, status, n_steps, Capture::compact, path_stride,
                      { path_cap, path, nullptr, path_offset, path_total_cap }, { caustic_cap, caustic, nullptr, caustic_offset, caustic_total_cap });
}

// Scheduling facts of the last trace (range-dependent sets): out[0] reserved (0), out[1] packets in the long region, out[2] CTAs
// of the exclusive long-region launch, out[3] kernels enqueued, out[4] long packets claimed as quarter packets.
extern "C" int geoac_last_schedule(geoac_ctx* ctx, int64_t* out8) {
    if (!ctx || !out8) return GEOAC_ERR_BAD_ARG;
    for (int i = 0; i < 8; i++) out8[i] = 0;
    out8[1] = ctx->last_long_packets; out8[2] = ctx->last_long_ctas; out8[3] = ctx->last_launches;
    out8[4] = ctx->last_quarter_packets;
    return GEOAC_OK;
}
// Test / diagnosis hook: the cost scout's predicted RK4 step counts of the last trace's rays (n entries, batch order); zeros if no
// claim order was built.
extern "C" int geoac_get_costs(geoac_ctx* ctx, int64_t n, uint32_t* cost) {
    if (!ctx || !cost || n < 0) return GEOAC_ERR_BAD_ARG;
    if (!ctx->d_cost.p || (size_t)n * sizeof(uint32_t) > ctx->d_cost.cap) return fail(ctx, GEOAC_ERR_BAD_ARG, "geoac_get_costs: no claim order of that size was built");
    cudaSetDevice(ctx->device);
    CK(cudaMemcpy(cost, ctx->d_cost.p, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost));
    return GEOAC_OK;
}

// Durations [ms] of the trace kernel launch(es) of the last trace, valid once the trace has completed: ms2[0] the main launch,
// ms2[1] the concurrent long-region launch (0 if there was none).
extern "C" int geoac_last_launch_ms(geoac_ctx* ctx, double* ms2) {
    if (!ctx || !ms2) return GEOAC_ERR_BAD_ARG;
    ms2[0] = ms2[1] = 0.0;
    if (!ctx->timed_launches) return GEOAC_OK;
    cudaSetDevice(ctx->device);
    float a = 0.f, b = 0.f;
    if (cudaEventElapsedTime(&a, ctx->ev_m0, ctx->ev_m1) == cudaSuccess) ms2[0] = a;
    if (ctx->last_long_ctas > 0 && cudaEventElapsedTime(&b, ctx->ev_l0, ctx->ev_l1) == cudaSuccess) ms2[1] = b;
    cudaGetLastError();
    return GEOAC_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// Several devices behind one call (SURVEY 8b / 8e).  Rays are independent, so the flattened launch-angle list (the mains'
// phi-major, theta-minor order, Code/GeoAc3D_main.cpp:226-227) is dealt to the contexts in interleaved blocks of
// GEOAC_SHARD_BLOCK rays -- lifetimes vary smoothly with theta, so interleaving balances the load -- one host thread per
// context gathers its share into that context's PINNED staging, traces it (geoac_trace: H2D, kernels, D2H) and puts the
// records back at the rays' places in the caller's arrays.  No collective, no exchange between devices; the merged result
// is bitwise what one context yields (tests/test_gpu_parity.py).
// ---------------------------------------------------------------------------------------------------------------
extern "C" int geoac_create_multi(int variant, const int* device_ids, int n_devices, geoac_ctx** ctxs, int* status) {
    if (!device_ids || !ctxs || n_devices < 1) { if (status) *status = GEOAC_ERR_BAD_ARG; g_create_error = "geoac_create_multi: need device ordinals and room for the contexts"; return GEOAC_ERR_BAD_ARG; }
    for (int i = 0; i < n_devices; i++) {
        int st = GEOAC_OK;
        ctxs[i] = geoac_create(variant, device_ids[i], &st);
        if (!ctxs[i]) {
            for (int j = 0; j < i; j++) { geoac_destroy(ctxs[j]); ctxs[j] = nullptr; }
            if (status) *status = st;
            return st;
        }
    }
    if (status) *status = GEOAC_OK;
    return GEOAC_OK;
}

template <class F>
static int for_each_ctx(geoac_ctx* const* ctxs, int n_ctx, F f) {          // one host thread per context; first failure wins
    if (!ctxs || n_ctx < 1) return GEOAC_ERR_BAD_ARG;
    for (int i = 0; i < n_ctx; i++) if (!ctxs[i]) return GEOAC_ERR_BAD_ARG;
    std::vector<int> rc((size_t)n_ctx, GEOAC_OK);
    std::vector<std::thread> pool;
    for (int i = 1; i < n_ctx; i++) pool.emplace_back([&, i] { rc[(size_t)i] = f(ctxs[i], i); });
    rc[0] = f(ctxs[0], 0);
    for (auto& t : pool) t.join();
    for (int i = 0; i < n_ctx; i++) if (rc[(size_t)i] != GEOAC_OK) { if (i) ctxs[0]->err = "context " + std::to_string(i) + ": " + ctxs[i]->err; return rc[(size_t)i]; }
    return GEOAC_OK;
}

extern "C" int geoac_multi_set_atmosphere_1d(geoac_ctx* const* ctxs, int n_ctx, int n, const double* z, const double* T,
                                             const double* u, const double* v, const double* rho) {
    return for_each_ctx(ctxs, n_ctx, [&](geoac_ctx* c, int) { return geoac_set_atmosphere_1d(c, n, z, T, u, v, rho); });
}
extern "C" int geoac_multi_set_atmosphere_3d(geoac_ctx* const* ctxs, int n_ctx, int n0, int n1, int nz, const double* ax0, const double* ax1,
                                             const double* axz, const double* T, const double* u, const double* v, const double* rho) {
    return for_each_ctx(ctxs, n_ctx, [&](geoac_ctx* c, int) { return geoac_set_atmosphere_3d(c, n0, n1, nz, ax0, ax1, axz, T, u, v, rho); });
}
extern "C" int geoac_multi_set_params(geoac_ctx* const* ctxs, int n_ctx, const geoac_params* p) {
    return for_each_ctx(ctxs, n_ctx, [&](geoac_ctx* c, int) { return geoac_set_params(c, p); });
}

extern "C" int geoac_trace_multi(geoac_ctx* const* ctxs, int n_ctx, int64_t n_rays, const double* theta, const double* phi,
                                 double* rec, int32_t* status, int32_t* n_steps) {
    if (!ctxs || n_ctx < 1 || n_rays < 0) return GEOAC_ERR_BAD_ARG;
    for (int i = 0; i < n_ctx; i++) if (!ctxs[i]) return GEOAC_ERR_BAD_ARG;
    if (n_rays > 0 && (!theta || !phi || !rec || !status || !n_steps)) return fail(ctxs[0], GEOAC_ERR_BAD_ARG, "geoac_trace_multi: null buffer");
    for (int i = 1; i < n_ctx; i++)
        if (ctxs[i]->variant != ctxs[0]->variant || ctxs[i]->prm.bounces != ctxs[0]->prm.bounces || ctxs[i]->prm.calc_amp != ctxs[0]->prm.calc_amp)
            return fail(ctxs[0], GEOAC_ERR_BAD_ARG, "geoac_trace_multi: the contexts must share variant, bounces and calc_amp (set the same atmosphere and parameters on each)");
    if (n_rays == 0) return GEOAC_OK;
    const int n_rec = ctxs[0]->prm.bounces + 1;
    const int64_t B = GEOAC_SHARD_BLOCK, n_blocks = (n_rays + B - 1) / B, n_slots = n_rays * n_rec;
    return for_each_ctx(ctxs, n_ctx, [&](geoac_ctx* ctx, int r) -> int {
        cudaSetDevice(ctx->device);
        int64_t mine = 0;                                                       // rays of the blocks b = r, r + n_ctx, r + 2 n_ctx, ...
        for (int64_t b = r; b < n_blocks; b += n_ctx) mine += std::min(B, n_rays - b * B);
        if (mine == 0) return GEOAC_OK;
        const int64_t my_slots = mine * n_rec;
        CK(ctx->pin_theta.grow(sizeof(double) * mine)); CK(ctx->pin_phi.grow(sizeof(double) * mine));
        CK(ctx->pin_rec.grow(sizeof(double) * GEOAC_NFIELDS * my_slots));
        CK(ctx->pin_status.grow(sizeof(int32_t) * my_slots)); CK(ctx->pin_nsteps.grow(sizeof(int32_t) * my_slots));
        double *h_th = ctx->pin_theta.p, *h_ph = ctx->pin_phi.p, *h_rec = ctx->pin_rec.p;
        int32_t *h_st = ctx->pin_status.p, *h_ns = ctx->pin_nsteps.p;
        int64_t at = 0;
        for (int64_t b = r; b < n_blocks; b += n_ctx) {
            const int64_t s0 = b * B, len = std::min(B, n_rays - s0);
            std::memcpy(h_th + at, theta + s0, sizeof(double) * len); std::memcpy(h_ph + at, phi + s0, sizeof(double) * len);
            at += len;
        }
        const int rc = trace_host(ctx, mine, h_th, h_ph, h_rec, h_st, h_ns);
        if (rc != GEOAC_OK) return rc;
        at = 0;
        for (int64_t b = r; b < n_blocks; b += n_ctx) {                          // merge by ray index
            const int64_t s0 = b * B, len = std::min(B, n_rays - s0);
            for (int f = 0; f < GEOAC_NFIELDS; f++)
                std::memcpy(rec + (int64_t)f * n_slots + s0 * n_rec, h_rec + (int64_t)f * my_slots + at * n_rec, sizeof(double) * len * n_rec);
            std::memcpy(status + s0 * n_rec, h_st + at * n_rec, sizeof(int32_t) * len * n_rec);
            std::memcpy(n_steps + s0 * n_rec, h_ns + at * n_rec, sizeof(int32_t) * len * n_rec);
            at += len;
        }
        return GEOAC_OK;
    });
}

extern "C" int geoac_get_variant(const geoac_ctx* ctx) { return ctx ? ctx->variant : -1; }

// Atmosphere at the source point, sampled on the device by the same spline code the kernels use (the per-launch invariants).
extern "C" int geoac_source_state(geoac_ctx* ctx, double* out4) {
    if (!ctx || !out4) return GEOAC_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    int rc = refresh_consts(ctx); if (rc != GEOAC_OK) return rc;
    LaunchConsts L;
    CK(cudaMemcpyAsync(&L, ctx->d_consts.p, sizeof L, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    out4[0] = L.c_src; out4[1] = L.u_src; out4[2] = L.v_src; out4[3] = L.rho_src;
    return GEOAC_OK;
}

// ---- the atmosphere at arbitrary points (atmo_sample.cuh): one thread per point, coordinates and rows SoA ----
enum { SMP_1D = 0, SMP_1D_GLOBAL = 1, SMP_GRID = 2, SMP_GRID_GLOBAL = 3 };
template <int KIND>
__global__ void __launch_bounds__(128) sample_atmosphere_kernel(const LaunchConsts* __restrict__ Lc, const Table1D T, const Grid3D g, int64_t n,
                                                                const double* __restrict__ p, double* __restrict__ out) {
    const LaunchConsts& L = *Lc;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double p0 = p[i], p1 = p[n + i], p2 = p[2 * n + i];
        if constexpr (KIND == SMP_1D) sample_point_1d<false>(L, T, p0, p2, out + i, n);
        else if constexpr (KIND == SMP_1D_GLOBAL) sample_point_1d<true>(L, T, p0, p2, out + i, n);
        else if constexpr (KIND == SMP_GRID) sample_point_grid<false>(L, g, p0, p1, p2, out + i, n);
        else sample_point_grid<true>(L, g, p0, p1, p2, out + i, n);
    }
}

extern "C" int geoac_sample_atmosphere(geoac_ctx* ctx, int64_t n, const double* p0, const double* p1, const double* p2, double* out) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    if (n < 0) return fail(ctx, GEOAC_ERR_BAD_ARG, "geoac_sample_atmosphere: n < 0");
    if (n > 0 && (!p0 || !p1 || !p2 || !out)) return fail(ctx, GEOAC_ERR_BAD_ARG, "geoac_sample_atmosphere: null buffer");
    for (int64_t i = 0; i < n; i++)
        if (!std::isfinite(p0[i]) || !std::isfinite(p1[i]) || !std::isfinite(p2[i]))
            return fail(ctx, GEOAC_ERR_BAD_ARG, "geoac_sample_atmosphere: coordinates of point " + std::to_string(i) + " are not finite");
    if (!ctx->have_atmo) return fail(ctx, GEOAC_ERR_NO_ATMO, "set an atmosphere first");
    if (n == 0) return GEOAC_OK;
    cudaSetDevice(ctx->device);
    if (int rc = refresh_consts(ctx)) return rc;                       // L.sb and the absorption parameters; no trace state is touched
    const int64_t B = std::min<int64_t>(n, GEOAC_SAMPLE_BLOCK);
    CK(ctx->d_smp_in.grow(sizeof(double) * 3 * B));
    CK(ctx->d_smp_out.grow(sizeof(double) * GEOAC_ATM_NF * B));
    const cudaStream_t st = ctx->stream;
    Table1D T{}; T.base = ctx->d_table.p; T.n = ctx->n; T.xmin = ctx->xmin; T.xmax = ctx->xmax; T.jump_scale = 0.0; T.sbpoly = nullptr;
    const int kind = ctx->is_grid ? (ctx->variant == GEOAC_GLOBAL_RNGDEP ? SMP_GRID_GLOBAL : SMP_GRID)
                                  : (ctx->variant == GEOAC_GLOBAL ? SMP_1D_GLOBAL : SMP_1D);
    for (int64_t s0 = 0; s0 < n; s0 += B) {
        const int64_t m = std::min(B, n - s0);
        double *in = ctx->d_smp_in.p, *res = ctx->d_smp_out.p;
        CK(cudaMemcpyAsync(in, p0 + s0, sizeof(double) * m, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(in + m, p1 + s0, sizeof(double) * m, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(in + 2 * m, p2 + s0, sizeof(double) * m, cudaMemcpyHostToDevice, st));
        const int grid = (int)std::min<int64_t>((m + 127) / 128, (int64_t)ctx->sm_count * 16);
        switch (kind) {
            case SMP_1D:          sample_atmosphere_kernel<SMP_1D><<<grid, 128, 0, st>>>(ctx->d_consts.p, T, ctx->grid, m, in, res); break;
            case SMP_1D_GLOBAL:   sample_atmosphere_kernel<SMP_1D_GLOBAL><<<grid, 128, 0, st>>>(ctx->d_consts.p, T, ctx->grid, m, in, res); break;
            case SMP_GRID:        sample_atmosphere_kernel<SMP_GRID><<<grid, 128, 0, st>>>(ctx->d_consts.p, T, ctx->grid, m, in, res); break;
            default:              sample_atmosphere_kernel<SMP_GRID_GLOBAL><<<grid, 128, 0, st>>>(ctx->d_consts.p, T, ctx->grid, m, in, res); break;
        }
        CK(cudaGetLastError());
        for (int f = 0; f < GEOAC_ATM_NF; f++)
            CK(cudaMemcpyAsync(out + (int64_t)f * n + s0, res + (int64_t)f * m, sizeof(double) * m, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return GEOAC_OK;
}

extern "C" int geoac_last_trace_stats(geoac_ctx* ctx, int64_t* total_steps, double* kernel_ms) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    unsigned long long cnt[2] = { 0, 0 };
    CK(cudaMemcpy(cnt, ctx->d_counters.p, sizeof cnt, cudaMemcpyDeviceToHost));   // also valid after geoac_trace_device + sync
    ctx->last_steps = (int64_t)cnt[1];
    if (ctx->ms_pending) {                                  // geoac_trace_device: NaN until its work on the caller's stream has completed
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev_d0, ctx->ev_d1) == cudaSuccess) { ctx->last_ms = ms; ctx->ms_pending = false; }
        else cudaGetLastError();
    }
    if (total_steps) *total_steps = ctx->last_steps;
    if (kernel_ms) *kernel_ms = ctx->last_ms;
    return GEOAC_OK;
}

extern "C" int geoac_last_trace_counters(geoac_ctx* ctx, int64_t* warp_trips, int64_t* kernel_launches) {
    if (!ctx) return GEOAC_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    unsigned long long t = 0;
    CK(cudaMemcpy(&t, ctx->d_counters.p + 2, sizeof t, cudaMemcpyDeviceToHost));
    if (warp_trips) *warp_trips = (int64_t)t;
    if (kernel_launches) *kernel_launches = ctx->last_launches;
    return GEOAC_OK;
}

// ---- Load_G2S: Code/Atmo/G2S_Spline1D.cpp:109-142 (Cartesian), G2S_GlobalSpline1D.cpp:113-152 (Global taper arithmetic) ----
extern "C" int geoac_load_met_1d(const char* path, const char* format, double z_grnd_taper, int global_taper,
                                 int cap, int* n, double* z, double* T, double* u, double* v, double* rho) {
    if (!path || !format || !n || !z || !T || !u || !v || !rho) return GEOAC_ERR_BAD_ARG;
    int fmt = !std::strncmp(format, "zTuvdp", 6) ? 0 : (!std::strncmp(format, "zuvwTdp", 7) ? 1 : -1);
    if (fmt < 0) return GEOAC_ERR_BAD_ARG;
    FILE* f = std::fopen(path, "r");
    if (!f) return GEOAC_ERR_IO;
    // file_length(): number of newline-terminated rows (G2S_Spline1D.cpp:53-71)
    long rows = 0; for (int ch; (ch = std::fgetc(f)) != EOF;) if (ch == '\n') rows++;
    std::rewind(f);
    int cnt = 0; double tmp, tmp2;
    while (cnt < cap && cnt < rows) {
        int got = fmt == 0 ? std::fscanf(f, "%lf %lf %lf %lf %lf %lf", &z[cnt], &T[cnt], &u[cnt], &v[cnt], &rho[cnt], &tmp)
                           : std::fscanf(f, "%lf %lf %lf %lf %lf %lf %lf", &z[cnt], &u[cnt], &v[cnt], &tmp, &T[cnt], &rho[cnt], &tmp2);
        if (got != (fmt == 0 ? 6 : 7)) break;
        double arg;
        if (global_taper) { const double r = z[cnt] + kREarth; arg = -(r - kREarth - z_grnd_taper) / 0.2; }
        else arg = -(z[cnt] - z_grnd_taper) / 0.2;
        u[cnt] *= (2.0 / (1.0 + std::exp(arg)) - 1.0) / 1000.0;      // m/s -> km/s and ground taper (App. A-10)
        v[cnt] *= (2.0 / (1.0 + std::exp(arg)) - 1.0) / 1000.0;
        cnt++;
    }
    std::fclose(f);
    *n = cnt;
    return cnt >= 3 ? GEOAC_OK : GEOAC_ERR_IO;
}

// ---- Load_G2S_Multi: Code/Atmo/G2S_MultiDimSpline3D.cpp:139-189 (Cartesian), G2S_GlobalMultiDimSpline3D.cpp:142-199 (Global) ----
// The reference reads its 40 000 - 65 000 node files one after another with operator>>.  Node files are independent: the
// first one fixes the level count, the rest are read whole and parsed with strtod (the conversion operator>> / fscanf use,
// so every value has the same bits) by a pool of host threads, each writing its own columns of the dense arrays.
static int parse_met_column(const std::string& path, int fmt, int global, int max_rows, double* axz, double* T, double* u, double* v, double* rho) {
    FILE* f = std::fopen(path.c_str(), "rb"); if (!f) return -1;
    std::string buf;
    char chunk[1 << 16]; size_t got;
    while ((got = std::fread(chunk, 1, sizeof chunk, f)) > 0) buf.append(chunk, got);
    std::fclose(f);
    const char* p = buf.c_str();
    const int ncol = fmt == 0 ? 6 : 7;
    int k = 0;
    while (k < max_rows) {
        double c[7]; int got_cols = 0;
        for (; got_cols < ncol; got_cols++) { char* e; c[got_cols] = std::strtod(p, &e); if (e == p) break; p = e; }
        if (got_cols < ncol) break;
        const double zz = c[0];
        double tt, uu, vv, rr;
        if (fmt == 0) { tt = c[1]; uu = c[2]; vv = c[3]; rr = c[4]; } else { uu = c[1]; vv = c[2]; tt = c[4]; rr = c[5]; }
        double arg;                                                             // ground taper: width 0.05 Cartesian, 0.2 Global; z_grnd = 0 at load
        if (global) { const double r = zz + kREarth; arg = -(r - kREarth - 0.0) / 0.2; }
        else        arg = -(zz - 0.0) / 0.05;
        uu *= (2.0 / (1.0 + std::exp(arg)) - 1.0) / 1000.0;
        vv *= (2.0 / (1.0 + std::exp(arg)) - 1.0) / 1000.0;
        if (axz) axz[k] = zz;
        T[k] = tt; u[k] = uu; v[k] = vv; rho[k] = rr;
        k++;
    }
    return k;
}

extern "C" int geoac_load_met_grid(const char* prefix, const char* loc0, const char* loc1, const char* format, int global,
                                   int cap0, int cap1, int capz, int* n0, int* n1, int* nz,
                                   double* ax0, double* ax1, double* axz, double* T, double* u, double* v, double* rho) {
    if (!prefix || !loc0 || !loc1 || !format || !n0 || !n1 || !nz || !ax0 || !ax1 || !axz || !T || !u || !v || !rho) return GEOAC_ERR_BAD_ARG;
    int fmt = !std::strncmp(format, "zTuvdp", 6) ? 0 : (!std::strncmp(format, "zuvwTdp", 7) ? 1 : -1);
    if (fmt < 0) return GEOAC_ERR_BAD_ARG;
    auto read_axis = [&](const char* path, double* out, int cap) -> int {
        FILE* f = std::fopen(path, "r"); if (!f) return -1;
        int c = 0; while (c < cap && std::fscanf(f, "%lf", &out[c]) == 1) c++;
        std::fclose(f); return c;
    };
    const int c0 = read_axis(loc0, ax0, cap0), c1 = read_axis(loc1, ax1, cap1);
    if (c0 < 2 || c1 < 2) return GEOAC_ERR_IO;
    if (global) { for (int i = 0; i < c0; i++) ax0[i] *= kPi / 180.0; for (int i = 0; i < c1; i++) ax1[i] *= kPi / 180.0; }   // degrees -> radians
    auto node_path = [&](long long idx) { return std::string(prefix) + std::to_string(idx) + ".met"; };   // <prefix><i0*n1+i1>.met
    const int cz = parse_met_column(node_path(0), fmt, global, capz, axz, T, u, v, rho);   // the first profile fixes the level count
    if (cz < 3) return GEOAC_ERR_IO;
    const long long ncol = (long long)c0 * c1;
    unsigned nthr = std::thread::hardware_concurrency(); if (nthr == 0) nthr = 1;
    if (const char* e = std::getenv("GEOAC_B200_LOAD_THREADS")) nthr = (unsigned)std::max(1, std::atoi(e));
    nthr = (unsigned)std::min<long long>(std::min(nthr, 64u), std::max(1LL, ncol - 1));
    std::atomic<long long> next{1};
    std::atomic<int> bad{0};
    auto work = [&]() {
        std::vector<double> zcol((size_t)cz);
        for (;;) {
            const long long c = next.fetch_add(1);
            if (c >= ncol || bad.load()) return;
            const size_t o = (size_t)c * cz;
            const int k = parse_met_column(node_path(c), fmt, global, cz, zcol.data(), T + o, u + o, v + o, rho + o);
            if (k != cz) { bad.store(1); return; }
            if (c == ncol - 1) std::copy(zcol.begin(), zcol.end(), axz);   // the reference overwrites z with every file; the last one stays
        }
    };
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < nthr; t++) pool.emplace_back(work);
    work();
    for (auto& t : pool) t.join();
    if (bad.load()) return GEOAC_ERR_IO;
    *n0 = c0; *n1 = c1; *nz = cz;
    return GEOAC_OK;
}

// ---- accuracy self-test of the branch-free FP64 primitives (core.cuh) against libdevice, on the device ----
__global__ void selftest_math_kernel(int n, unsigned long long* worst) {        // worst[7]: rcp, rsqrt, sqrt, exp, exp10, sin, cos (bits of max err)
    unsigned long long s = 0x9E3779B97F4A7C15ull * (blockIdx.x * blockDim.x + threadIdx.x + 1);
    auto uni = [&]() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return (double)(s >> 11) * (1.0 / 9007199254740992.0); };
    double w[7] = { 0, 0, 0, 0, 0, 0, 0 };
    for (int i = 0; i < n; i++) {
        const double mant = 1.0 + uni(), ex = floor(uni() * 1800.0) - 900.0;
        const double x = ldexp(mant, (int)ex);                                  // 2^-900 .. 2^900
        const double xe = (uni() * 2.0 - 1.0) * 690.0, xt = (uni() * 2.0 - 1.0) * 290.0;
        const double a[1] = { xe }, b[1] = { xt }; double oa[1], ob[1];
        g_exp_n<false, 1>(a, oa); g_exp_n<true, 1>(b, ob);
        double rs; const double sq = g_sqrt_rs(x, rs);
        const double got[5] = { g_rcp(x), g_rsqrt(x), sq, oa[0], ob[0] };
        const double ref[5] = { 1.0 / x, rsqrt(x), sqrt(x), exp(xe), exp10(xt) };
        for (int k = 0; k < 5; k++) w[k] = fmax(w[k], fabs(got[k] - ref[k]) / fabs(ref[k]));
        const double xa = (uni() * 2.0 - 1.0) * 12.0;                            // a few turns; absolute error for sin / cos
        double gs, gc; g_sincos(xa, &gs, &gc);
        w[5] = fmax(w[5], fabs(gs - sin(xa))); w[6] = fmax(w[6], fabs(gc - cos(xa)));
    }
    for (int k = 0; k < 7; k++) atomicMax(worst + k, (unsigned long long)__double_as_longlong(w[k]));   // positive doubles order like integers
}

extern "C" int geoac_selftest_math(geoac_ctx* ctx, int n_per_thread, double* max_rel_err) {
    if (!ctx || !max_rel_err || n_per_thread <= 0) return GEOAC_ERR_BAD_ARG;
    cudaSetDevice(ctx->device);
    Buf<unsigned long long> d;
    CK(d.grow(7 * sizeof(unsigned long long)));
    CK(cudaMemset(d.p, 0, 7 * sizeof(unsigned long long)));
    selftest_math_kernel<<<ctx->sm_count, 256, 0, ctx->stream>>>(n_per_thread, d.p);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(max_rel_err, d.p, 7 * sizeof(double), cudaMemcpyDeviceToHost));
    return GEOAC_OK;
}

// ---- FP64 roofline denominator: dependent-chain-free DFMA loop, 8 independent accumulators per thread ----
__global__ void dfma_peak_kernel(double* out, int iters, double a, double b) {
    double x0 = threadIdx.x * 1e-9, x1 = x0 + 1.0, x2 = x0 + 2.0, x3 = x0 + 3.0, x4 = x0 + 4.0, x5 = x0 + 5.0, x6 = x0 + 6.0, x7 = x0 + 7.0;
#pragma unroll 1
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}

extern "C" double geoac_measure_fp64_peak(geoac_ctx* ctx, double* out_ms) {
    if (!ctx) return -1.0;
    cudaSetDevice(ctx->device);
    const int block = 512, grid = ctx->sm_count * 4, iters = 4096;
    Buf<double> d;
    if (d.grow(sizeof(double) * block * grid) != cudaSuccess) return -1.0;
    float best = 1e30f;
    for (int rep = 0; rep < 5; rep++) {
        cudaEventRecord(ctx->ev0, ctx->stream);
        dfma_peak_kernel<<<grid, block, 0, ctx->stream>>>(d.p, iters, 0.999999, 1e-7);
        cudaEventRecord(ctx->ev1, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        float ms = 0; cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1);
        if (rep > 0 && ms < best) best = ms;
    }
    if (out_ms) *out_ms = best;
    const double flops = 2.0 * 64.0 * (double)iters * (double)block * (double)grid;
    return flops / (best * 1e-3) / 1e12;
}
