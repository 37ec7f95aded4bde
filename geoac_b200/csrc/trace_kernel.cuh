// trace_kernel.cuh -- the persistent one-thread-per-ray RK4 kernel, generic over the equation set.
//
// Replaces, for a whole batch of launch angles, the body of the reference's `-prop` loops
// (Code/GeoAc3D_main.cpp:226-304 and siblings) including GeoAc_Propagate_RK4 (Code/GeoAc/GeoAc.Solver.cpp:12-72).
//
// Design (B200-first, not a translation):
//  * ONE resident CTA per SM; the spline table is pulled into shared memory by a single TMA bulk copy
//    (cp.async.bulk + mbarrier) and stays there for the life of the kernel.
//  * a lane owns one ray at a time and advances it by exactly ONE RK4 step (+ its travel-time / absorption
//    segment) per trip round a flat loop, so all lanes of a warp execute the same instruction stream no matter how
//    far along their rays are.  Bounces / arrivals / breaks are handled in a rare divergent tail of the trip.
//  * finished lanes are refilled at the top of the trip: a warp ballot counts the idle lanes, one lane claims that
//    many ray indices from a global counter with a single atomicAdd, the indices are handed out by lane rank.
//  * only three states are ever needed (k-2, k-1, k): y_k sits in the lane's shared-memory record, y_{k+1} is built in
//    registers, y_{k-1} is parked in an L2-resident global scratch (one coalesced store per equation per step; read back
//    only at a reflection).  The reference stores 500 000 x EqCnt.
//  * RK4 combination in the reference's association order  y + k1/6 + k2/3 + k3/3 + k4/6  (Solver.cpp:54), built
//    on the fly so no k_i is kept.
#pragma once
#include <type_traits>
#include "core.cuh"
#include "mspline.cuh"

namespace geoac {

struct TraceArgs {
    Grid3D grid;                // range-dependent variants: node tables in global memory (L1/L2 resident working set)
    const double* table;        // global copy of the table (n records of TAB_NARR doubles, 16-byte aligned)
    int table_n;
    double table_xmin, table_xmax;
    const double* sbpoly;       // per-interval absorption polynomials of the table (core.cuh) or nullptr = exact evaluation
    const LaunchConsts* consts; // device
    const double* theta;        // [n_rays]
    const double* phi;
    int64_t n_rays;
    int n_rec;                  // bounces + 1
    double* rec;                // [GEOAC_NFIELDS][n_rays*n_rec]
    int32_t* status;            // [n_rays*n_rec]
    int32_t* n_steps;
    unsigned long long* counter;      // next unclaimed ray
    unsigned long long* total_steps;  // RK4 steps taken (all rays)
    unsigned long long* warp_trips;   // trips round the step loop, summed over warps (lane occupancy = steps / (32 trips))
    const uint32_t* order;            // claim order (longest-predicted first) or nullptr = natural order; 0xffffffff = empty slot
    int64_t n_claims;                 // entries of `order` (a multiple of 32 in packet mode), or n_rays
    // packet mode (range-dependent sets): the first n_long_packets packets of `order` are the LONG region -- packets whose
    // predicted cost exceeds the average work of a lane, i.e. which would outlast the pass on a fully loaded SM.  They are
    // claimed by the CTAs of a second, concurrent launch that keeps its SMs to itself (one warp per scheduler: see capi.cu).
    int64_t n_long_packets;
    int64_t n_quarter_packets;        // the first of them -- the very longest -- are claimed eight rays at a time and traced four lanes per
                                      // ray from the start: a warp with 8 rays keeps their cells in L1 and needs ~0.6x the instructions per step
    unsigned long long* counter_quarter;
    unsigned long long* counter_long; // next unclaimed entry of the long region
    int prefer_long;                  // this launch claims the long region first (1) or the main region first (0)
    int packet_refill;                // stratified sets: refill a warp only when all of its lanes are idle (set with the sorted claim order;
                                      // the PacketMode sets always refill this way)
    double* path; int32_t* path_rows; int path_stride; int64_t path_cap;   // raypath capture (PATHS kernels), else unused
    double* caus; int32_t* caus_rows; int64_t caus_cap;                    // caustic events (PATHS kernels), else unused
    double* prev;                     // y_{k-1} scratch: [NEQ][grid * block] doubles (variants with a quadratic intercept)
};
// Arguments of the many-source kernels (MSRC): ray r is launched from source src_id[r], whose invariants are
// src_consts[src_id[r]].  A type of their own, so that the single-source kernels keep their parameters as they are.
struct TraceArgsMS : TraceArgs {
    const LaunchConsts* src_consts;
    const int32_t* src_id;
};
// Arguments of the ensemble kernels (stratified sets): ray r is traced through member atm_id[r] of an ensemble of 1-D
// profiles, with that member's invariants atm_consts[m] and table atm_tab[m] (base, n, xmin, xmax, sbpoly; jump_scale 0).
// The cost scout reads atm_tab_scout[m] instead (the same table with jump_scale = (n-1)/(xmax-xmin), no sbpoly).  All of
// them in global memory, read through L1.
struct TraceArgsEns : TraceArgs {
    const LaunchConsts* atm_consts;
    const Table1D* atm_tab;
    const Table1D* atm_tab_scout;
    const int32_t* atm_id;
};
template <class ARGS> struct IsMSrc { static constexpr bool value = std::is_same<ARGS, TraceArgsMS>::value; };
template <class ARGS> struct IsEns { static constexpr bool value = std::is_same<ARGS, TraceArgsEns>::value; };

// Per-launch invariants of the stratified variants (source / ground / reference-level atmosphere samples and the
// Sutherland-Bass reference state), evaluated once with the same spline routines the rays use.
GEOAC_HD void fill_launch_consts_1d(LaunchConsts& L, const Table1D& T, int variant) {
    const bool glob = (variant == GEOAC_GLOBAL);
    int cur = 0;
    double c, u, v, rho, dc, du, dv;
    auto sample = [&](double x) {
        const SegPos sp = seg_locate(T, x, cur);
        double Tv, dT, ddT, d2;
        spl_f2(T, TAB_T, sp, Tv, dT, ddT);
        spl_f2(T, TAB_U, sp, u, du, d2);
        spl_f2(T, TAB_V, sp, v, dv, d2);
        rho = spl_f(T, TAB_RHO, sp);
        c = sqrt(kGamR * Tv);
        dc = kGamR / (2.0 * c) * dT;
    };
    L.ground = glob ? kREarth + L.z_grnd : L.z_grnd;
    sample(glob ? L.src[0] + kREarth : L.src[2]);
    L.c_src = c; L.u_src = u; L.v_src = v; L.rho_src = rho;
    sample(0.0);
    L.c_000 = c;                                   // c(0,0,0) of the 3-D travel time (App. A-4)
    sample(L.ground);
    L.c_gnd = c; L.rho_gnd = rho; L.dc_gnd = dc; L.du_gnd = du; L.dv_gnd = dv;
    // Sutherland-Bass reference state: c, rho at (0,0,z_grnd) (Cartesian, Absorption.cpp:33-34) or at r = z_grnd, i.e.
    // clamped to the lowest level (Global, Absorption.Global.cpp:31-32; SURVEY App. A-14)
    sample(L.z_grnd);
    suthbass_setup(L, c, rho);
}

struct RecOut {
    double* rec; int32_t* status; int32_t* n_steps; int64_t n_slots; int n_rec;
    // raypath capture (PATHS kernels only): rows of GEOAC_PATH_NF doubles, `path_cap` rows reserved per ray
    double* path; int32_t* path_rows; int path_stride; int64_t path_cap;
    // caustic events (PATHS kernels only): rows of GEOAC_CAUSTIC_NF doubles where the Jacobian changes sign
    double* caus; int32_t* caus_rows; int64_t caus_cap;
};

// ---------------------------------------------------------------------------------------------------------------
// One lane = one ray in flight.  The FP64 part of its state (LaneD: y_k, the per-ray constants, the running sums) lives
// in SHARED memory on the device -- one contiguous record per thread with an odd stride in doubles, so the 64-bit
// accesses of a half-warp fall into 16 distinct bank pairs -- which is what lets 512 threads (16 warps) per SM fit
// the register file next to the 112 KB spline table.  The integer part (LaneI) stays in registers.
// lane_advance() performs exactly one RK4 step, the travel-time/absorption bookkeeping of that step's segment, and --
// rarely -- the end-of-bounce tail (arrival record, reflection, break).  It is the whole per-ray state machine of
// SURVEY 3.4; the kernel below only adds lane refill around it.
// ---------------------------------------------------------------------------------------------------------------
template <class EQ>
struct LaneD {
    double y[EQ::NEQ];
    typename EQ::RayC rc;
    double tt_total, att_total, tt_b, att_b, zmax;
    double D_prev;          // Jacobian at the previous step (caustic capture)
};
template <class EQ>
struct LaneI {
    typename EQ::Cursor cur;
    int bounce, ksteps;
    int path_n, caus_n;     // raypath rows / caustic events emitted so far (PATHS kernels)
    int caus_b;             // caustic events of the current bounce segment (GeoAc_CausticCnt)
    int64_t ray;
};

// packet scheduling (see the refill step of trace_kernel): the range-dependent sets, whose node tables are read through L1
template <class EQ> struct PacketMode { static constexpr bool value = std::is_same<typename EQ::Atmo, Grid3D>::value; };

// does the reflection need y_{k-2}?  (quadratic intercept: 2D, 3D, 3D.RngDep; the Global variants fit a line, App. A-7)
template <class EQ> struct NeedsPrev { static constexpr bool value = !(EQ::VARIANT == GEOAC_GLOBAL || EQ::VARIANT == GEOAC_GLOBAL_RNGDEP); };

template <class EQ>
GEOAC_HD void lane_start(LaneD<EQ>& d, LaneI<EQ>& n, const LaunchConsts& L, const typename EQ::Atmo& T, int64_t idx, double theta, double phi) {
    n.ray = idx; n.bounce = 0; n.ksteps = 0; n.path_n = 0; n.caus_n = 0; n.caus_b = 0; n.cur = typename EQ::Cursor{};
    d.tt_total = d.att_total = d.tt_b = d.att_b = d.zmax = 0.0; d.D_prev = 0.0;
    EQ::init(L, T, theta, phi, d.rc, d.y, n.cur);
}

// Range-dependent sets keep the RK4 accumulator and the stage input in the lane's shared-memory record as well (their
// right-hand side needs the registers for the 4x4-node sampler); the stratified sets keep them in registers.
// The four RK4 stages are unrolled for the Cartesian stratified sets (the tail of a stage overlaps the head of the next;
// config 2: 399.5 -> 387.5 ms per pass, config 1: 100 -> 88 ms) and kept as a loop for the spherical set (18 equations at
// the register ceiling: unrolled it spills more, config 3: 3.76 -> 4.19 s) and for the range-dependent ones.
#ifndef GEOAC_STAGE_UNROLL
#define GEOAC_STAGE_UNROLL 4
#endif
template <class EQ> struct WorkInMem { static constexpr bool value = std::is_same<typename EQ::Atmo, Grid3D>::value; };

// Cooperative mode (several lanes advance ONE ray on its shared-memory record, every lane executing the same read-modify-write
// of the record redundantly): the lanes of the group must not run ahead of each other between a read and the matching write.
// They are in lock step by construction, but the CUDA memory model does not promise it, so the group synchronises around the
// record updates.  No-op for one lane per ray.
GEOAC_HD void group_sync(const Table1D&) {}
GEOAC_HD void group_sync(const Grid3D& g) {
#if defined(__CUDA_ARCH__)
    if (g.nrole > 1) __syncwarp(g.gmask);
#else
    (void)g;
#endif
}

// prev[i * pstride] holds y_{k-1}[i] (only maintained when NeedsPrev); work = 2 NEQ doubles (WorkInMem) or nullptr;
// returns false when the ray has ended.  PATHS: also emit one raypath row every o.path_stride steps (WriteRays=True of the
// mains, Code/GeoAc3D_main.cpp:249-262: position, amplitude at that point, absorption and travel-time sums so far).
template <class EQ, bool PATHS = false>
GEOAC_HD bool lane_advance(LaneD<EQ>& d, LaneI<EQ>& n, const LaunchConsts& L, const typename EQ::Atmo& T, double* prev, int64_t pstride,
                           const RecOut& o, double* work) {
    constexpr int NEQ = EQ::NEQ;
    constexpr bool MEM = WorkInMem<EQ>::value;
    double* const y = d.y;
    d.zmax = fmax(d.zmax, EQ::altitude(y));                     // running turning height over m < k (App. A-3)
    const double ds = EQ::step_size(L, y);
    double acc_r[MEM ? 1 : NEQ], p_r[MEM ? 1 : NEQ], f[NEQ];
    double* const acc = MEM ? work : acc_r;
    double* const p = MEM ? work + NEQ : p_r;
#pragma unroll
    for (int i = 0; i < NEQ; i++) { acc[i] = y[i]; p[i] = acc[i]; }
    constexpr int kStageUnroll = (MEM || NEQ > 12) ? 1 : GEOAC_STAGE_UNROLL;
#pragma unroll(kStageUnroll)
    for (int s = 0; s < 4; s++) {
        const double sc = EQ::rhs(L, T, d.rc, p, f, n.cur);     // right-hand sides up to their common factor (1 / |c_prop|)
        const double dsa = (ds * ((s == 2) ? 1.0 : 0.5)) * sc;
        const double dsb = (ds * ((s == 0 || s == 3) ? (1.0 / 6.0) : (1.0 / 3.0))) * sc;
        if (MEM) {                                             // the record is shared by the lanes of a cooperative group
            double a_new[NEQ];
#pragma unroll
            for (int i = 0; i < NEQ; i++) a_new[i] = fma(f[i], dsb, acc[i]);
            group_sync(T);                                     // every lane has read acc / p (rhs) before any lane overwrites them
#pragma unroll
            for (int i = 0; i < NEQ; i++) { acc[i] = a_new[i]; p[i] = fma(f[i], dsa, y[i]); }
            group_sync(T);
        } else {
#pragma unroll
            for (int i = 0; i < NEQ; i++) {
                acc[i] = fma(f[i], dsb, acc[i]);               // y + k1/6 + k2/3 + k3/3 + k4/6, left to right (k_i = ds f_i)
                p[i] = fma(f[i], dsa, y[i]);                   // y + k_i/2 (stage 4: y + k_3)
            }
        }
    }
    n.ksteps++;
    double dtt, datt;
    EQ::segment(L, T, d.rc, y, acc, n.cur, dtt, datt);
    const bool brk = EQ::left_region(L, d.rc, acc);              // BreakCheck first (Solver.cpp:57-64)
    const bool gnd = !brk && EQ::below_ground(L, acc);
    const bool lim = !brk && !gnd && (n.ksteps >= L.step_limit - 1);
    {   // running sums: read, (cooperative group: everyone has read), write
        const double tt0 = d.tt_total, at0 = d.att_total, tb0 = d.tt_b, ab0 = d.att_b;
        if (MEM) group_sync(T);
        if (L.seg_mode) { if (!(brk || gnd || lim)) { d.tt_total = tt0 + dtt; d.att_total = at0 + datt; } }
        else            { d.tt_b = tb0 + dtt; d.att_b = ab0 + datt; }
    }

    if (!(brk || gnd || lim)) {
        if (PATHS) {
            if (o.caus_cap > 0) {
                // WriteCaustics=True (Code/GeoAc3D_main.cpp:241-268): D_prev starts as the Jacobian of step 1 of each bounce; a
                // row { position, travel time } wherever D * D_prev < 0
                const double D = EQ::jacobian(L, T, d.rc, acc, n.cur);
                const double Dp = d.D_prev;
                if (n.ksteps > 1 && D * Dp < 0.0) {
                    if (n.caus_n < o.caus_cap) {
                        double* row = o.caus + ((int64_t)n.ray * o.caus_cap + n.caus_n) * GEOAC_CAUSTIC_NF;
                        row[0] = acc[0]; row[1] = acc[1]; row[2] = acc[2]; row[3] = d.tt_total;
                        row[4] = (double)n.bounce; row[5] = (double)n.ksteps;
                    }
                    n.caus_n++; n.caus_b++;
                }
                if (MEM) group_sync(T);
                d.D_prev = D;
            }
            if (o.path_stride > 0 && n.ksteps % o.path_stride == 0) {   // row for state m = ksteps (m < k: never the sub-ground point)
                if (n.path_n < o.path_cap) {
                    double* row = o.path + ((int64_t)n.ray * o.path_cap + n.path_n) * GEOAC_PATH_NF;
                    row[0] = acc[0]; row[1] = acc[1]; row[2] = acc[2];
                    row[3] = EQ::amplitude(L, T, d.rc, acc, n.cur);
                    row[4] = d.att_total; row[5] = d.tt_total;
                    row[6] = (double)n.bounce; row[7] = (double)n.ksteps;
                }
                n.path_n++;
            }
        }
#pragma unroll
        for (int i = 0; i < NEQ; i++) { if (NeedsPrev<EQ>::value) prev[i * pstride] = y[i]; }
        if (MEM) group_sync(T);                                 // every lane of the group has parked y_k before it becomes y_{k+1}
#pragma unroll
        for (int i = 0; i < NEQ; i++) y[i] = acc[i];
        return true;
    }
    // ---------------- rare tail: end of a bounce segment ----------------
    const int64_t slot = n.ray * o.n_rec + n.bounce;
    if (!gnd) {
        o.status[slot] = brk ? GEOAC_ST_BREAK : GEOAC_ST_LIMIT;
        o.n_steps[slot] = brk ? n.ksteps : L.step_limit;
        if (brk) o.rec[(int64_t)GEOAC_F_MARGIN * o.n_slots + slot] = EQ::break_margin(L, d.rc, y, acc);   // how marginal the break was
        if (PATHS) { if (o.path_rows) o.path_rows[n.ray] = n.path_n; if (o.caus_rows) o.caus_rows[n.ray] = n.caus_n; }
        return false;
    }
    if (!L.seg_mode) {
        const double tt0 = d.tt_total + d.tt_b, at0 = d.att_total + d.att_b;
        if (MEM) group_sync(T);
        d.tt_total = tt0; d.att_total = at0; d.tt_b = 0.0; d.att_b = 0.0;
        if (MEM) group_sync(T);
    }
    double amp, incl, baz, aux, margin;
    EQ::arrival(L, T, d.rc, y, acc, d.tt_total, n.cur, amp, incl, baz, aux, margin);
#pragma unroll
    for (int i = 0; i < NEQ; i++) o.rec[(int64_t)i * o.n_slots + slot] = acc[i];
    o.rec[(int64_t)GEOAC_F_TRAVELTIME * o.n_slots + slot] = d.tt_total;
    o.rec[(int64_t)GEOAC_F_ATTEN * o.n_slots + slot] = d.att_total;
    o.rec[(int64_t)GEOAC_F_TURNHEIGHT * o.n_slots + slot] = d.zmax;
    o.rec[(int64_t)GEOAC_F_AMPLITUDE * o.n_slots + slot] = amp;
    o.rec[(int64_t)GEOAC_F_INCLINATION * o.n_slots + slot] = incl;
    o.rec[(int64_t)GEOAC_F_BACKAZ * o.n_slots + slot] = baz;
    o.rec[(int64_t)GEOAC_F_AUX * o.n_slots + slot] = aux;
    o.rec[(int64_t)GEOAC_F_MARGIN * o.n_slots + slot] = margin;
    o.rec[(int64_t)GEOAC_F_JACOBIAN * o.n_slots + slot] = EQ::jacobian(L, T, d.rc, acc, n.cur);
    o.rec[(int64_t)GEOAC_F_CAUSTICS * o.n_slots + slot] = (PATHS && o.caus_cap > 0) ? (double)n.caus_b : -1.0;
    o.status[slot] = GEOAC_ST_ARRIVAL;
    o.n_steps[slot] = n.ksteps;
    if (n.bounce >= L.bounces) {
        if (PATHS) { if (o.path_rows) o.path_rows[n.ray] = n.path_n; if (o.caus_rows) o.caus_rows[n.ray] = n.caus_n; }
        return false;
    }
    double ym2[NEQ], y0[NEQ];
#pragma unroll
    for (int i = 0; i < NEQ; i++) ym2[i] = NeedsPrev<EQ>::value ? prev[i * pstride] : 0.0;
    EQ::reflect(L, T, d.rc, ym2, y, acc, y0, n.cur);
    if (MEM) group_sync(T);                                     // the intercept read y_{k-1} (= y) and y_k on every lane of the group
#pragma unroll
    for (int i = 0; i < NEQ; i++) y[i] = y0[i];
    n.bounce++; n.ksteps = 0; n.caus_b = 0;
    if (L.per_bounce_zmax) d.zmax = 0.0;
    return true;
}

#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// stage `bytes` (multiple of 16) from global to shared with TMA bulk copies issued by thread 0
__device__ __forceinline__ void tma_stage_table(double* dst, const double* src, uint32_t bytes, uint64_t* bar) {
    const uint32_t bar_a = smem_u32(bar);
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
        uint32_t off = 0;
        while (off < bytes) {
            uint32_t chunk = min(bytes - off, 65536u);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(smem_u32((const char*)dst + off)), "l"((const char*)src + off), "r"(chunk), "r"(bar_a)
                         : "memory");
            off += chunk;
        }
    }
    uint32_t done = 0;                                   // everyone waits for phase 0 to complete
    while (!done) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar_a) : "memory");
    }
}

// odd number of doubles per lane record: conflict-free 64-bit shared-memory accesses with one record per thread
// layout of a record: [LaneD][WorkInMem: acc (NEQ), stage input (NEQ), sampler outputs (MS_SCRATCH)]
template <class EQ> struct LaneLayout {
    static constexpr int WORK = (int)(sizeof(LaneD<EQ>) / sizeof(double));
    static constexpr int EXTRA = WorkInMem<EQ>::value ? 2 * EQ::NEQ + MS_SCRATCH : 0;
    static constexpr int STRIDE = (WORK + EXTRA) | 1;
};

// The invariants a ray is traced with: the launch's (L) or, in the many-source kernels, those of the ray's own source s (in
// the ensemble kernels: of its member s), read from global memory through L1 (a warp whose rays share a source reads one
// address).  Rays keep the caller's order among equal claim keys, so a batch laid out source by source (member by member)
// gives warps of mostly one source (member).
template <class ARGS>
__device__ __forceinline__ const LaunchConsts& ray_consts(const LaunchConsts& L, const ARGS& a, int s) {
    if constexpr (IsMSrc<ARGS>::value) return a.src_consts[s];
    else if constexpr (IsEns<ARGS>::value) return a.atm_consts[s];
    else return L;
}
// The atmosphere a ray is traced through: the launch's (T) or, in the ensemble kernels, the table of its member s -- a
// reference into global memory, not a register copy.
template <class ARGS, class ATMO>
__device__ __forceinline__ const ATMO& ray_atmo(const ATMO& T, const ARGS& a, int s) {
    if constexpr (IsEns<ARGS>::value) return a.atm_tab[s];
    else return T;
}

// ARGS: TraceArgs, TraceArgsMS for the many-source kernels (MSRC) or TraceArgsEns for the ensemble kernels (ENS, stratified
// sets, TABLE_IN_SMEM = false)
template <class EQ, int BLOCK, bool TABLE_IN_SMEM, bool PATHS = false, class ARGS = TraceArgs>
__global__ void __launch_bounds__(BLOCK, 1) trace_kernel(const __grid_constant__ ARGS a) {
    constexpr bool MSRC = IsMSrc<ARGS>::value, ENS = IsEns<ARGS>::value;
    static_assert(!ENS || (!TABLE_IN_SMEM && !PacketMode<EQ>::value), "the ensemble kernels read 1-D tables from global memory");
    constexpr int NEQ = EQ::NEQ;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: [LaunchConsts][mbarrier][lane records: BLOCK x STRIDE doubles][table]
    LaunchConsts* Ls = reinterpret_cast<LaunchConsts*>(smem_raw);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw + ((sizeof(LaunchConsts) + 15) / 16) * 16);
    double* lanes = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(bar) + 16);
    double* tab_s = lanes + ((LaneLayout<EQ>::STRIDE * BLOCK + 1) & ~1);          // keep the table 16-byte aligned

    if constexpr (!MSRC && !ENS) {              // the many-source / ensemble kernels read each ray's invariants from global memory instead
        for (int i = threadIdx.x; i < (int)(sizeof(LaunchConsts) / 8); i += BLOCK)
            reinterpret_cast<double*>(Ls)[i] = reinterpret_cast<const double*>(a.consts)[i];
    }
    typename EQ::Atmo T;
    double* const work = lanes + (size_t)threadIdx.x * LaneLayout<EQ>::STRIDE + LaneLayout<EQ>::WORK;
    if constexpr (std::is_same<typename EQ::Atmo, Grid3D>::value) {
        T = a.grid;
        T.scratch = work + 2 * NEQ;
    } else {
        T.n = a.table_n; T.xmin = a.table_xmin; T.xmax = a.table_xmax; T.jump_scale = 0.0; T.sbpoly = a.sbpoly;
        if (TABLE_IN_SMEM) {
            tma_stage_table(tab_s, a.table, (uint32_t)(TAB_NARR * a.table_n * sizeof(double)), bar);
            T.base = tab_s;
        } else {
            T.base = a.table;
        }
    }
    __syncthreads();
    const LaunchConsts& L = *Ls;

    const unsigned lane = threadIdx.x & 31;
    RecOut o; o.rec = a.rec; o.status = a.status; o.n_steps = a.n_steps; o.n_rec = a.n_rec; o.n_slots = a.n_rays * a.n_rec;
    o.path = a.path; o.path_rows = a.path_rows; o.path_stride = a.path_stride; o.path_cap = a.path_cap;
    o.caus = a.caus; o.caus_rows = a.caus_rows; o.caus_cap = a.caus_cap;
    LaneD<EQ>& ld = *reinterpret_cast<LaneD<EQ>*>(lanes + (size_t)threadIdx.x * LaneLayout<EQ>::STRIDE);
    LaneI<EQ> li;
    int rsrc = 0;                      // MSRC: source of the lane's ray; ENS: its member
    // y_{k-1} history (quadratic intercept only): [eq][global thread] in an L2-resident global scratch, written once per step
    const int64_t pstride = (int64_t)gridDim.x * BLOCK;
    double* prev = a.prev + ((int64_t)blockIdx.x * BLOCK + threadIdx.x);
    bool have_ray = false, exhausted = false;
    unsigned region_done = 0;          // packet mode, lane 0: bit 0 = long region drained, bit 1 = main region drained
    unsigned long long my_steps = 0;
    unsigned my_trips = 0;

    while (true) {
        // ---------------- refill idle lanes (warp-aggregated claim) ----------------
        if constexpr (PacketMode<EQ>::value) {
            // PACKET sets (range dependent): a warp takes 32 rays of one packet at once -- neighbouring launch angles, chosen by
            // the host so that the lanes walk through the same few grid cells (capi.cu) -- and refills only when all of them have
            // ended.  Two regions of the claim order, two counters; which one a warp drains first depends on the launch it
            // belongs to (long-region CTAs run one warp per scheduler, so a long packet advances at lone-warp speed).
            if (!exhausted && !__any_sync(0xffffffffu, have_ray)) {
                unsigned long long base = 0; int width = 0;
                if (lane == 0) {
                    const unsigned long long nq = (unsigned long long)a.n_quarter_packets * 32ull;                 // [0, nq): quarter claims
                    const unsigned long long nl = (unsigned long long)a.n_long_packets * 32ull;                    // [nq, nl): whole long packets
                    const unsigned long long nm = (unsigned long long)a.n_claims - nl;                             // [nl, n_claims): main region
                    for (int attempt = 0; attempt < 3 && width == 0; attempt++) {
                        // long-region CTAs: quarter, long, main; main CTAs: main, long, quarter
                        const int region = a.prefer_long ? attempt : 2 - attempt;
                        if (region == 0) {
                            if (nq && !(region_done & 4u)) {
                                const unsigned long long q = atomicAdd(a.counter_quarter, 8ull);
                                if (q < nq) { base = q; width = 8; } else region_done |= 4u;
                            }
                        } else if (region == 1) {
                            if (nl > nq && !(region_done & 1u)) {
                                const unsigned long long q = atomicAdd(a.counter_long, 32ull);
                                if (nq + q < nl) { base = nq + q; width = 32; } else region_done |= 1u;
                            }
                        } else if (nm && !(region_done & 2u)) {
                            const unsigned long long q = atomicAdd(a.counter, 32ull);
                            if (q < nm) { base = nl + q; width = 32; } else region_done |= 2u;
                        }
                    }
                }
                base = __shfl_sync(0xffffffffu, base, 0);
                width = __shfl_sync(0xffffffffu, width, 0);
                if (width == 0) exhausted = true;
                else if ((int)lane < width) {
                    const int64_t idx = (int64_t)base + lane;
                    const int64_t r = a.order ? (int64_t)a.order[idx] : idx;
                    if (r < a.n_rays) {
                        if constexpr (MSRC) rsrc = a.src_id[r];
                        if constexpr (ENS) rsrc = a.atm_id[r];
                        lane_start<EQ>(ld, li, ray_consts(L, a, rsrc), ray_atmo(T, a, rsrc), r, a.theta[r], a.phi[r]); have_ray = true;
                    }
                }
            }
        } else {
            const bool busy = a.packet_refill && __any_sync(0xffffffffu, have_ray);
            const bool want = !have_ray && !exhausted && !busy;
            const unsigned wmask = __ballot_sync(0xffffffffu, want);
            if (wmask) {
                unsigned long long base = 0;
                const int leader = __ffs(wmask) - 1;
                if ((int)lane == leader) base = atomicAdd(a.counter, (unsigned long long)__popc(wmask));
                base = __shfl_sync(0xffffffffu, base, leader);
                const int rank = __popc(wmask & ((1u << lane) - 1u));
                if (want) {
                    const int64_t idx = (int64_t)base + rank;
                    if (idx < a.n_claims) {
                        const int64_t r = a.order ? (int64_t)a.order[idx] : idx;
                        if (r < a.n_rays) {
                            if constexpr (MSRC) rsrc = a.src_id[r];
                            if constexpr (ENS) rsrc = a.atm_id[r];
                            lane_start<EQ>(ld, li, ray_consts(L, a, rsrc), ray_atmo(T, a, rsrc), r, a.theta[r], a.phi[r]); have_ray = true;
                        }
                    }
                    else exhausted = true;
                }
            }
        }
        const unsigned act = __ballot_sync(0xffffffffu, have_ray);
        if (!act) break;
        my_trips++;
        if constexpr (PacketMode<EQ>::value) {
            // ---------------- four lanes per ray when <= 8 rays of the packet are live ----------------
            // The lane records live in shared memory, so any lane can work on any ray of its warp: group g (lanes 4g..4g+3)
            // advances the g-th live ray, each lane evaluating one row of the 4x4 node block per sample (mspline.cuh); every
            // other operation is executed redundantly and identically by the four lanes.  Same bits as the serial path.
            // One call site serves both modes (the step function is large; two inlined copies would double the kernel).
            const int nact = __popc(act);
            const bool coop = nact <= 8;
            const int grp = (int)lane >> 2;
            const int owner = (coop && grp < nact) ? (int)__fns(act, 0, grp + 1) : (int)lane;
            const bool run = coop ? (grp < nact) : have_ray;
            LaneI<EQ> gi;
            gi.cur.ka = __shfl_sync(0xffffffffu, li.cur.ka, owner); gi.cur.kb = __shfl_sync(0xffffffffu, li.cur.kb, owner);
            gi.cur.kz = __shfl_sync(0xffffffffu, li.cur.kz, owner);
            gi.bounce = __shfl_sync(0xffffffffu, li.bounce, owner); gi.ksteps = __shfl_sync(0xffffffffu, li.ksteps, owner);
            gi.ray = __shfl_sync(0xffffffffu, (long long)li.ray, owner);
            gi.path_n = __shfl_sync(0xffffffffu, li.path_n, owner); gi.caus_n = __shfl_sync(0xffffffffu, li.caus_n, owner);
            gi.caus_b = PATHS ? __shfl_sync(0xffffffffu, li.caus_b, owner) : 0;
            const int gsrc = (MSRC || ENS) ? __shfl_sync(0xffffffffu, rsrc, owner) : 0;     // a ray keeps its source: nothing to hand back
            const int othread = (int)(threadIdx.x & ~31u) + owner;
            double* const rec = lanes + (size_t)othread * LaneLayout<EQ>::STRIDE;
            double* const gwork = rec + LaneLayout<EQ>::WORK;
            typename EQ::Atmo Tg = T;
            Tg.scratch = gwork + 2 * NEQ;
            if (coop) { Tg.role = (int)lane & 3; Tg.nrole = 4; Tg.glane0 = (int)lane & ~3; Tg.gmask = 0xFu << ((int)lane & ~3); }
            bool alive = false;
            if (run) alive = lane_advance<EQ, PATHS>(*reinterpret_cast<LaneD<EQ>*>(rec), gi, ray_consts(L, a, gsrc), Tg,
                                                       a.prev + ((int64_t)blockIdx.x * BLOCK + othread), pstride, o, gwork);
            // hand the integer state back to the lane that owns the ray (itself in serial mode)
            const int src = (coop && have_ray) ? 4 * __popc(act & ((1u << lane) - 1u)) : (int)lane;
            const int bka = __shfl_sync(0xffffffffu, gi.cur.ka, src), bkb = __shfl_sync(0xffffffffu, gi.cur.kb, src);
            const int bkz = __shfl_sync(0xffffffffu, gi.cur.kz, src);
            const int bbo = __shfl_sync(0xffffffffu, gi.bounce, src), bks = __shfl_sync(0xffffffffu, gi.ksteps, src);
            const int bal = __shfl_sync(0xffffffffu, (int)alive, src);
            const int bpn = __shfl_sync(0xffffffffu, gi.path_n, src), bcn = __shfl_sync(0xffffffffu, gi.caus_n, src);
            const int bcb = PATHS ? __shfl_sync(0xffffffffu, gi.caus_b, src) : 0;
            if (have_ray) {
                li.cur.ka = bka; li.cur.kb = bkb; li.cur.kz = bkz; li.bounce = bbo; li.ksteps = bks; li.path_n = bpn; li.caus_n = bcn; li.caus_b = bcb;
                have_ray = bal != 0;
                my_steps++;
            }
        } else {
            if (have_ray) {
                have_ray = lane_advance<EQ, PATHS>(ld, li, ray_consts(L, a, rsrc), ray_atmo(T, a, rsrc), prev, pstride, o, work);
                my_steps++;
            }
        }
    }
    for (int off = 16; off > 0; off >>= 1) my_steps += __shfl_xor_sync(0xffffffffu, my_steps, off);
    if (lane == 0 && my_steps) { atomicAdd(a.total_steps, my_steps); atomicAdd(a.warp_trips, (unsigned long long)my_trips); }   // per warp
}

// ---------------------------------------------------------------------------------------------------------------
// Longest-ray-first scheduling.  Ray lifetimes differ by an order of magnitude and a lane processes only a few rays,
// so with the natural claim order ~30 % of the lane-steps of a 2e5-ray batch idle in the tail while the last long
// rays finish.  A SCOUT pass predicts each ray's RK4 step count by tracing it with the amplitude-free equation set
// (EQ<false>) at COARSE times the step size -- ~1/COARSE of the steps at ~1/4 of the cost per step, i.e. a few per cent
// of the real trace -- then a counting sort over 256 cost buckets yields the claim order, longest first.  The order
// only affects scheduling: every ray's arithmetic is independent of which lane runs it and when.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kScoutCoarse = 16;
constexpr int kCostBuckets = 256;

// lanes per CTA of the scout: 512 (<= 128 registers) for the stratified sets, 256 for the range-dependent sampler
template <class EQ> struct ScoutBlock { static constexpr int value = std::is_same<typename EQ::Atmo, Grid3D>::value ? 256 : 512; };

// The atmosphere the scout predicts a ray in: the launch's (T) or, in the ensemble scout, the table of its member s.
template <class ARGS, class ATMO>
__device__ __forceinline__ const ATMO& scout_atmo(const ATMO& T, const ARGS& a, int s) {
    if constexpr (IsEns<ARGS>::value) return a.atm_tab_scout[s];
    else return T;
}

// Persistent like the trace kernel: lanes are refilled from a counter as their rays end (a warp of rays with different
// lifetimes never idles), the 1-D table sits in shared memory; the ray state (<= 6 equations, no auxiliary set) fits
// in registers.
// ARGS = TraceArgsMS (MSRC): each ray is predicted with its own source's invariants (ray_consts).  ARGS = TraceArgsEns (ENS):
// with its own member's invariants and table (atm_tab_scout); a.consts is then any member's (only the parameters are read).
template <class EQ, bool TABLE_IN_SMEM, class ARGS = TraceArgs>
__global__ void __launch_bounds__(ScoutBlock<EQ>::value, 1) scout_kernel(const __grid_constant__ ARGS a, uint32_t* cost, uint32_t* cost_max,
                                                               unsigned long long* cost_sum, unsigned long long* counter, int coarse) {
    constexpr bool MSRC = IsMSrc<ARGS>::value, ENS = IsEns<ARGS>::value;
    static_assert(!ENS || !TABLE_IN_SMEM, "the ensemble scout reads 1-D tables from global memory");
    constexpr int NEQ = EQ::NEQ;
    constexpr bool kGrid = std::is_same<typename EQ::Atmo, Grid3D>::value;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
    double* tab_s = reinterpret_cast<double*>(smem_raw + 16);
    const LaunchConsts& L = *a.consts;
    typename EQ::Atmo T;
    double sbuf[kGrid ? MS_SCRATCH : 1];
    if constexpr (kGrid) { T = a.grid; T.scratch = sbuf; }
    else {
        T.n = a.table_n; T.xmin = a.table_xmin; T.xmax = a.table_xmax; T.base = a.table;
        T.jump_scale = (double)(a.table_n - 1) / (a.table_xmax - a.table_xmin);
        if (TABLE_IN_SMEM) { tma_stage_table(tab_s, a.table, (uint32_t)(TAB_NARR * a.table_n * sizeof(double)), bar); T.base = tab_s; }
    }
    __syncthreads();
    const unsigned lane = threadIdx.x & 31;
    const uint32_t cap = (uint32_t)L.step_limit;
    double y[NEQ], ym1[NEQ];
    typename EQ::RayC rc; typename EQ::Cursor cur = typename EQ::Cursor{};
    uint32_t est = 0, seg = 0, worst = 0; int bounce = 0; int64_t ray = 0;
    int rsrc = 0;
    unsigned long long total = 0;
    bool have_ray = false, exhausted = false;
    while (true) {
        const bool want = !have_ray && !exhausted;
        const unsigned wmask = __ballot_sync(0xffffffffu, want);
        if (wmask) {
            unsigned long long base = 0;
            const int leader = __ffs(wmask) - 1;
            if ((int)lane == leader) base = atomicAdd(counter, (unsigned long long)__popc(wmask));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (want) {
                ray = (int64_t)(base + __popc(wmask & ((1u << lane) - 1u)));
                if (ray < a.n_rays) {
                    cur = typename EQ::Cursor{};
                    if constexpr (MSRC) rsrc = a.src_id[ray];
                    if constexpr (ENS) rsrc = a.atm_id[ray];
                    EQ::init(ray_consts(L, a, rsrc), scout_atmo(T, a, rsrc), a.theta[ray], a.phi[ray], rc, y, cur);
#pragma unroll
                    for (int i = 0; i < NEQ; i++) ym1[i] = y[i];
                    est = 0; seg = 0; bounce = 0; have_ray = true;
                } else exhausted = true;
            }
        }
        if (!__any_sync(0xffffffffu, have_ray)) break;
        if (!have_ray) continue;
        const LaunchConsts& Lr = ray_consts(L, a, rsrc);
        const typename EQ::Atmo& Tr = scout_atmo(T, a, rsrc);
        double acc[NEQ], p[NEQ], f[NEQ];
        const double ds = (double)coarse * EQ::step_size(Lr, y);
#pragma unroll
        for (int i = 0; i < NEQ; i++) { acc[i] = y[i]; p[i] = y[i]; }
#pragma unroll 1
        for (int s = 0; s < 4; s++) {
            const double sc = EQ::rhs(Lr, Tr, rc, p, f, cur);
            const double dsa = ds * ((s == 2) ? 1.0 : 0.5) * sc, dsb = ds * ((s == 0 || s == 3) ? (1.0 / 6.0) : (1.0 / 3.0)) * sc;
#pragma unroll
            for (int i = 0; i < NEQ; i++) { acc[i] = fma(f[i], dsb, acc[i]); p[i] = fma(f[i], dsa, y[i]); }
        }
        est += (uint32_t)coarse; seg += (uint32_t)coarse;
        bool done = EQ::left_region(Lr, rc, acc) || seg >= cap;
        if (!done && EQ::below_ground(Lr, acc)) {
            if (bounce >= L.bounces) done = true;
            else {
                double y0[NEQ];
                EQ::reflect(Lr, Tr, rc, ym1, y, acc, y0, cur);
#pragma unroll
                for (int i = 0; i < NEQ; i++) { acc[i] = y0[i]; y[i] = y0[i]; }      // restart: y = ym1 = reflected state
                bounce++; seg = 0;
            }
        }
        if (done) {
            cost[ray] = est; total += est;
            worst = max(worst, est); have_ray = false;
        }
        else {
#pragma unroll
            for (int i = 0; i < NEQ; i++) { ym1[i] = y[i]; y[i] = acc[i]; }
        }
    }
    worst = __reduce_max_sync(0xffffffffu, worst);
    for (int off = 16; off > 0; off >>= 1) total += __shfl_xor_sync(0xffffffffu, total, off);
    if (lane == 0 && worst) { atomicMax(cost_max, worst); atomicAdd(cost_sum, total); }
}

#ifndef GEOAC_TRACE_KERNELS_ONLY          // the claim-order kernels below have one home: capi.cu
// The cost scout is accurate in bulk (config 5: correlation 0.988 with the true step counts, median ratio 0.999) but a ray at the edge
// of a ducted family can go either way: measured, a ray predicted at 21 k steps took 389 k, its packet sat at the back of the
// claim order and one rank in eight ran 27 s instead of 22.5 s.  Such rays are neighbours in inclination of rays that ARE predicted
// long, so the estimate used for ordering is the maximum over the neighbours within `dtheta` of the ray (same azimuth row): the
// edge of a long family is treated as long.  Scheduling only.
__global__ void cost_dilate_kernel(const uint32_t* cost, const double* theta, int64_t n, double dtheta, int radius, uint32_t* out) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        uint32_t c = cost[i];
        const double t = theta[i];
        for (int d = 1; d <= radius; d++) {
            if (i - d >= 0 && fabs(theta[i - d] - t) <= dtheta) c = max(c, cost[i - d]);
            if (i + d < n && fabs(theta[i + d] - t) <= dtheta) c = max(c, cost[i + d]);
        }
        out[i] = c;
    }
}

// counting sort by predicted cost, descending: hist[b] of bucket(cost) -> start offsets -> scatter.  The sorted items are
// GROUPS of `group` consecutive rays (1, or 32 in packet mode: a packet's cost is that of its longest ray); `order` gets
// n_groups * group entries, 0xffffffff where the last group runs past the batch.
__device__ __forceinline__ int cost_bucket(uint32_t c, uint32_t cmax) {
    return (kCostBuckets - 1) - (int)(((uint64_t)c * (kCostBuckets - 1)) / (cmax ? cmax : 1u));      // longest -> bucket 0
}
__device__ __forceinline__ uint32_t group_cost(const uint32_t* cost, int64_t n, int64_t g, int group) {
    uint32_t c = 0;
    for (int l = 0; l < group; l++) { const int64_t r = g * group + l; if (r < n) c = max(c, cost[r]); }
    return c;
}
// Also counts the LONG groups: those whose predicted cost exceeds the average work of a lane (cost_sum / lanes) -- traced
// serially such a packet alone would outlast the rest of the batch, so it is traced four lanes per ray instead.
__global__ void order_hist_kernel(const uint32_t* cost, int64_t n, int group, const uint32_t* cost_max, uint32_t* hist,
                                  const unsigned long long* cost_sum, long long lanes, uint32_t* n_long, int alpha_pct, uint32_t* n_quarter, int alpha2_pct) {
    __shared__ uint32_t h[kCostBuckets];
    __shared__ uint32_t nl, nq;
    for (int i = threadIdx.x; i < kCostBuckets; i += blockDim.x) h[i] = 0;
    if (threadIdx.x == 0) { nl = 0; nq = 0; }
    __syncthreads();
    const uint32_t cmax = *cost_max;
    const unsigned long long avg = *cost_sum / (unsigned long long)lanes;
    const unsigned long long thr = avg * (unsigned long long)alpha_pct / 100ull, thr2 = avg * (unsigned long long)alpha2_pct / 100ull;
    const int64_t ng = (n + group - 1) / group;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < ng; g += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t c = group_cost(cost, n, g, group);
        atomicAdd(&h[cost_bucket(c, cmax)], 1u);
        if (group == 32 && (unsigned long long)c > thr) atomicAdd(&nl, 1u);
        if (group == 32 && (unsigned long long)c > thr2) atomicAdd(&nq, 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kCostBuckets; i += blockDim.x) if (h[i]) atomicAdd(&hist[i], h[i]);
    if (threadIdx.x == 0 && nl) atomicAdd(n_long, nl);
    if (threadIdx.x == 0 && nq) atomicAdd(n_quarter, nq);
}
__global__ void order_scan_kernel(uint32_t* hist) {          // one block of kCostBuckets threads: exclusive prefix in place
    __shared__ uint32_t h[kCostBuckets];
    const int t = threadIdx.x;
    h[t] = hist[t];
    __syncthreads();
    for (int off = 1; off < kCostBuckets; off <<= 1) {
        const uint32_t v = (t >= off) ? h[t - off] : 0u;
        __syncthreads();
        h[t] += v;
        __syncthreads();
    }
    hist[t] = h[t] - hist[t];
}
__global__ void order_scatter_kernel(const uint32_t* cost, int64_t n, int group, const uint32_t* cost_max, uint32_t* offs, uint32_t* order) {
    const uint32_t cmax = *cost_max;
    const int64_t ng = (n + group - 1) / group;
    for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < ng; g += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t pos = atomicAdd(&offs[cost_bucket(group_cost(cost, n, g, group), cmax)], 1u);
        for (int l = 0; l < group; l++) {
            const int64_t r = g * group + l;
            order[(int64_t)pos * group + l] = (r < n) ? (uint32_t)r : 0xffffffffu;
        }
    }
}

// ---- claim order of the stratified sets: (cost bucket descending, inclination, batch index) ----
// A warp claims 32 consecutive entries and refills only when all of them have ended.  Sorted this way they are rays of
// near-equal predicted cost, EQUAL inclination and neighbouring azimuths (the mains enumerate the grid azimuth by azimuth),
// i.e. near-identical altitude histories: the lanes' table reads hit the same one or two records (a shared-memory broadcast
// instead of the 5-way bank conflict of unrelated altitudes) and the interval searches do not diverge.
// Two passes of a STABLE counting sort (LSD order): by inclination bucket, then by cost bucket.  Block b owns the contiguous
// slice [b*chunk, (b+1)*chunk) of the sequence: per-block histograms, one scan over (bucket, block), then every block (one
// warp) places its slice in order, ranks within a warp step from __match_any_sync.  The order only schedules: records do not
// depend on it (tests/test_gpu_parity.py::test_longest_ray_first_schedule_is_result_neutral).
__global__ void order_theta_range_kernel(const double* theta, int64_t n, double* range) {        // one block; range[0] = min, [1] = max
    __shared__ double lo[32], hi[32];
    double a = 1e300, b = -1e300;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) { const double t = theta[i]; a = fmin(a, t); b = fmax(b, t); }
    for (int off = 16; off > 0; off >>= 1) { a = fmin(a, __shfl_xor_sync(0xffffffffu, a, off)); b = fmax(b, __shfl_xor_sync(0xffffffffu, b, off)); }
    if ((threadIdx.x & 31) == 0) { lo[threadIdx.x >> 5] = a; hi[threadIdx.x >> 5] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); w++) { a = fmin(a, lo[w]); b = fmax(b, hi[w]); }
        range[0] = a; range[1] = b;
    }
}
// cost_shift coarsens the cost key (256 >> shift levels): a level must be wide enough to hold a whole run of neighbouring
// azimuths of one inclination, and narrow enough that the rays of a warp end within a few per cent of each other.
__global__ void order_keys_kernel(const uint32_t* cost, const double* theta, int64_t n, const uint32_t* cost_max, const double* range,
                                  uint8_t* key_theta, uint8_t* key_cost, int cost_shift) {
    const uint32_t cmax = *cost_max;
    const double t0 = range[0], span = range[1] - range[0];
    const double sc = span > 0.0 ? (kCostBuckets - 1) / span : 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        int kt = (int)((theta[i] - t0) * sc + 0.5);
        key_theta[i] = (uint8_t)(kt < 0 ? 0 : (kt > kCostBuckets - 1 ? kCostBuckets - 1 : kt));
        key_cost[i] = (uint8_t)(cost_bucket(cost[i], cmax) >> cost_shift);
    }
}
__global__ void stable_hist_kernel(const uint8_t* key, const uint32_t* src, int64_t n, int64_t chunk, uint32_t* blockhist) {
    __shared__ uint32_t h[kCostBuckets];
    for (int i = threadIdx.x; i < kCostBuckets; i += blockDim.x) h[i] = 0;
    __syncthreads();
    const int64_t g0 = (int64_t)blockIdx.x * chunk, g1 = min(n, g0 + chunk);
    for (int64_t g = g0 + threadIdx.x; g < g1; g += blockDim.x) atomicAdd(&h[key[src ? src[g] : (uint32_t)g]], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < kCostBuckets; i += blockDim.x) blockhist[(size_t)blockIdx.x * kCostBuckets + i] = h[i];
}
__global__ void stable_scan_kernel(uint32_t* blockhist, int nblk) {        // one block of kCostBuckets threads: counts -> start offsets
    __shared__ uint32_t h[kCostBuckets];
    const int t = threadIdx.x;
    uint32_t tot = 0;
    for (int b = 0; b < nblk; b++) tot += blockhist[(size_t)b * kCostBuckets + t];
    h[t] = tot;
    __syncthreads();
    for (int off = 1; off < kCostBuckets; off <<= 1) {
        const uint32_t v = (t >= off) ? h[t - off] : 0u;
        __syncthreads();
        h[t] += v;
        __syncthreads();
    }
    uint32_t run = h[t] - tot;
    for (int b = 0; b < nblk; b++) { const uint32_t v = blockhist[(size_t)b * kCostBuckets + t]; blockhist[(size_t)b * kCostBuckets + t] = run; run += v; }
}
__global__ void stable_scatter_kernel(const uint8_t* key, const uint32_t* src, int64_t n, int64_t chunk, const uint32_t* blockoffs, uint32_t* dst) {   // 32 threads
    __shared__ uint32_t base[kCostBuckets];
    for (int i = threadIdx.x; i < kCostBuckets; i += 32) base[i] = blockoffs[(size_t)blockIdx.x * kCostBuckets + i];
    __syncwarp();
    const int64_t g0 = (int64_t)blockIdx.x * chunk, g1 = min(n, g0 + chunk);
    const unsigned lane = threadIdx.x;
    for (int64_t gb = g0; gb < g1; gb += 32) {
        const int64_t g = gb + lane;
        const bool on = g < g1;
        const unsigned active = __ballot_sync(0xffffffffu, on);
        if (on) {
            const uint32_t r = src ? src[g] : (uint32_t)g;
            const int b = key[r];
            const unsigned m = __match_any_sync(active, b);
            const uint32_t pos = base[b] + (uint32_t)__popc(m & ((1u << lane) - 1u));
            __syncwarp(active);
            if ((int)lane == __ffs(m) - 1) base[b] += (uint32_t)__popc(m);
            dst[pos] = r;
        }
        __syncwarp();
    }
}

#endif  // GEOAC_TRACE_KERNELS_ONLY

// The many-source kernels (ARGS = TraceArgsMS) are instantiated in trace_sources.cu, a translation unit of their own: the out-of-line
// absorption path (core.cuh: suthbass_alpha_cold) is one function per unit, compiled for the shared-memory invariants of the
// single-source kernels; a caller passing global-memory invariants in the same unit would turn its shared loads generic.
template <class EQ, int BLOCK, bool TABLE_IN_SMEM> const void* msrc_trace_kernel();
template <class EQ, bool TABLE_IN_SMEM> const void* msrc_scout_kernel();
// Their raypath / caustic capture counterparts (PATHS = true) live in trace_sources_paths.cu, a unit of their own as well.
template <class EQ, int BLOCK, bool TABLE_IN_SMEM> const void* msrc_paths_trace_kernel();
// The ensemble kernels (ARGS = TraceArgsEns), and the set-up of the ensemble's invariants, live in trace_ensemble.cu for the
// same reason.  They have one table placement (global memory): TABLE_IN_SMEM is ignored.
template <class EQ, int BLOCK> const void* ens_trace_kernel();
template <class EQ> const void* ens_scout_kernel();
// On `st`: the invariants of every member, out[m] = `in` (the parameters, source clamped) filled in from table tab[m] (no
// sbpoly), then the absorption polynomials of every interval of every member into poly (member m's intervals from
// iv_off[m] on, n_iv in all).  One thread per member, then one per (member, interval).
cudaError_t ens_setup(LaunchConsts* out, const LaunchConsts& in, const Table1D* tab, int n_atm, const int64_t* iv_off, int64_t n_iv,
                      int variant, double* poly, cudaStream_t st);
template <class EQ, int BLOCK, bool TABLE_IN_SMEM, bool PATHS, class ARGS>
const void* trace_kernel_fn() {
    if constexpr (IsMSrc<ARGS>::value) {
        if constexpr (PATHS) return msrc_paths_trace_kernel<EQ, BLOCK, TABLE_IN_SMEM>();
        else return msrc_trace_kernel<EQ, BLOCK, TABLE_IN_SMEM>();
    }
    else if constexpr (IsEns<ARGS>::value) {
        static_assert(!PATHS, "the ensemble kernels have no raypath / caustic capture");
        return ens_trace_kernel<EQ, BLOCK>();
    }
    else return (const void*)trace_kernel<EQ, BLOCK, TABLE_IN_SMEM, PATHS>;
}
template <class EQ, bool TABLE_IN_SMEM, class ARGS>
const void* scout_kernel_fn() {
    if constexpr (IsMSrc<ARGS>::value) return msrc_scout_kernel<EQ, TABLE_IN_SMEM>();
    else if constexpr (IsEns<ARGS>::value) return ens_scout_kernel<EQ>();
    else return (const void*)scout_kernel<EQ, TABLE_IN_SMEM>;
}

#endif  // __CUDACC__
}  // namespace geoac
