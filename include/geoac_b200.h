/* geoac_b200.h -- C ABI of the B200-native batched ray-tracing engine (libgeoac_b200.so).
 *
 * The drop-in boundary sits between the launch-angle loops of the reference's `-prop` front ends and everything
 * inside them (reference: Code/GeoAc3D_main.cpp:226-304, Code/GeoAc2D_main.cpp:170-229,
 * Code/GeoAcGlobal_main.cpp:241-322, Code/GeoAc3D.RngDep_main.cpp:244-323, Code/GeoAcGlobal.RngDep_main.cpp:251-331).
 * One call to geoac_trace() replaces, for EVERY (theta, phi) launch angle of the batch:
 *   GeoAc_SetInitialConditions        (Code/GeoAc/GeoAc.EquationSets.h:8-10)
 *   GeoAc_Propagate_RK4               (Code/GeoAc/GeoAc.Solver.h:8)   incl. GeoAc_UpdateSources / GeoAc_EvalSrcEq /
 *                                      GeoAc_Set_ds / GeoAc_BreakCheck / GeoAc_GroundCheck (EquationSets.h:15-23)
 *   GeoAc_TravelTime[Segment], GeoAc_SB_Atten[Segment], GeoAc_Jacobian, GeoAc_Amplitude (EquationSets.h:25-30)
 *   GeoAc_SetReflectionConditions / GeoAc_ApproximateIntercept         (EquationSets.h:12-13)
 * and the atmosphere API they call (Code/Atmo/Atmo_State.h:11-36: rho,c,u,v,w + _diff/_ddiff, SuthBass_Alpha).
 *
 * Plain pointers and sizes only; the caller owns every host buffer; a context owns its device memory.
 * There is NO CPU fallback: without an sm_100 device geoac_create() fails with GEOAC_ERR_NO_DEVICE.
 */
#ifndef GEOAC_B200_H_
#define GEOAC_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- variants (one per reference executable, makefile:10-23) ---- */
enum {
    GEOAC_2D            = 0,   /* GeoAc2D            : effective sound speed, EqCnt 3/6            */
    GEOAC_3D            = 1,   /* GeoAc3D            : stratified moving medium, EqCnt 4/12        */
    GEOAC_GLOBAL        = 2,   /* GeoAcGlobal        : spherical stratified, EqCnt 6/18            */
    GEOAC_3D_RNGDEP     = 3,   /* GeoAc3D.RngDep     : Cartesian range dependent, EqCnt 6/18       */
    GEOAC_GLOBAL_RNGDEP = 4    /* GeoAcGlobal.RngDep : spherical range dependent, EqCnt 6/18       */
};

/* ---- status codes ---- */
enum {
    GEOAC_OK = 0,
    GEOAC_ERR_NO_DEVICE = 1,      /* no CUDA device / not sm_100                                   */
    GEOAC_ERR_BAD_ARG   = 2,
    GEOAC_ERR_NO_ATMO   = 3,      /* trace called before an atmosphere was set                     */
    GEOAC_ERR_CUDA      = 4,      /* CUDA runtime error, text in geoac_last_error()                */
    GEOAC_ERR_TOO_LARGE = 5,      /* table does not fit the kernel's staging (message says why)    */
    GEOAC_ERR_IO        = 6
};

/* ---- arrival record fields: rec[field * n_slots + ray * n_rec + bounce], n_slots = n_rays * n_rec ---- */
enum {
    GEOAC_F_STATE0     = 0,    /* 0..17: state vector at index k (first sub-ground point, SURVEY App. A-1),
                                  layout per variant as in the reference's solution[k][*]; unused entries 0 */
    GEOAC_F_TRAVELTIME = 18,   /* [s]   accumulated over bounces                                  */
    GEOAC_F_ATTEN      = 19,   /* [dB]  Sutherland-Bass, accumulated, positive (host prints -atten)*/
    GEOAC_F_TURNHEIGHT = 20,   /* [km]  running max altitude (accumulated or per bounce, App. A-3) */
    GEOAC_F_AMPLITUDE  = 21,   /* linear GeoAc_Amplitude(solution,k); host prints 20*log10; 0 if !calc_amp */
    GEOAC_F_INCLINATION= 22,   /* [deg] as printed by the variant's main (sign conventions App. A-16) */
    GEOAC_F_BACKAZ     = 23,   /* [deg] as printed by the variant's main; 0 for 2D                 */
    GEOAC_F_AUX        = 24,   /* Global variants: celerity [km/s]; otherwise 0                    */
    GEOAC_F_MARGIN     = 25,   /* ARRIVAL: (z_k - z_grnd)/|z_k - z_{k-1}| in (-1,0): how far into the last step the ground was
                                  crossed.  BREAK: fraction in (0,1] of the last step that lay beyond the violated limit
                                  (smallest over the limits violated).  Values within ~1e-6 of 0 / -1 / 1 flag rays whose step
                                  count or outcome is within rounding of a branch threshold (geoac_b200/nearthreshold.py) */
    GEOAC_F_JACOBIAN   = 26,   /* GeoAc_Jacobian(solution,k): the determinant D the amplitude divides by (0 if !calc_amp);
                                  |D| small against its own terms = near a caustic, amplitude ill-conditioned */
    GEOAC_F_CAUSTICS   = 27,   /* GeoAc_CausticCnt(solution,1,k): sign changes of D within this bounce segment, counted only by
                                  geoac_trace_paths with caustic_cap > 0 (the plain trace does not evaluate D per step): else -1 */
    GEOAC_NFIELDS      = 28,
    /* one raypath row (geoac_trace_paths): state[0..2], amplitude (linear), absorption sum, travel-time sum, bounce, step */
    GEOAC_PATH_NF      = 8,
    /* one caustic event: state[0..2] at the step where the Jacobian changed sign, travel-time sum, bounce, step */
    GEOAC_CAUSTIC_NF   = 6
};

/* ---- atmosphere sample fields (geoac_sample_atmosphere): out[field * n + i] ---- */
enum {
    GEOAC_ATM_C     = 0,       /* c() [km/s] = sqrt(gamR T)                                                               */
    GEOAC_ATM_U     = 1,       /* u() [km/s]                                                                              */
    GEOAC_ATM_V     = 2,       /* v() [km/s]                                                                              */
    GEOAC_ATM_RHO   = 3,       /* rho() [g/cm^3]                                                                          */
    GEOAC_ATM_DC    = 4,       /* c_diff / u_diff / v_diff along the vertical coordinate (z Cartesian, r Global)          */
    GEOAC_ATM_DU    = 5,
    GEOAC_ATM_DV    = 6,
    GEOAC_ATM_ALPHA = 7,       /* SuthBass_Alpha [dB/km] (x tweak_abs), full model                                       */
    GEOAC_ATM_T     = 8,       /* 8..17: T and its derivatives over (p0, p1, p2): f, d0, d1, d2, d00, d11, d22, d01, d02, d12,
                                  as the right-hand side sees them (Eval_Spline_AllOrder2 on the grids, slips of SURVEY
                                  App. A-8 / A-9 included; the vertical spline's f, f', f'' for stratified atmospheres)   */
    GEOAC_ATM_UF    = 18,      /* 18..27: u, the same 10 entries                                                         */
    GEOAC_ATM_VF    = 28,      /* 28..37: v, the same 10 entries                                                         */
    GEOAC_ATM_NF    = 38
};
/* points per device pass of geoac_sample_atmosphere (bounds its device memory at 41 doubles per point of a pass) */
enum { GEOAC_SAMPLE_BLOCK = 1 << 20 };

/* per-slot status */
enum {
    GEOAC_ST_NONE    = 0,      /* ray ended before this bounce                                     */
    GEOAC_ST_ARRIVAL = 1,      /* ground arrival; record fields valid                              */
    GEOAC_ST_BREAK   = 2,      /* left the propagation region (no results row, ray ends; App. A-19)*/
    GEOAC_ST_LIMIT   = 3       /* step limit reached                                               */
};

typedef struct geoac_params {
    /* solver (Code/GeoAc/GeoAc.Parameters*.cpp) */
    double ds_min;             /* 0.001                                                            */
    double ds_max;             /* 0.5                                                              */
    double ray_limit;          /* 5000 (Cartesian) / 10000 (Global); step_limit = ray_limit*int(1/(ds_min*10)) */
    /* propagation region; set from the atmosphere by geoac_set_atmosphere_* exactly like GeoAc_SetPropRegion,
       then overridable (alt_max= / rng_max= / x_min= ... of the mains) */
    double vert_limit;         /* z_max of the table (Cartesian) or absolute r_max (Global)        */
    double range_limit;        /* 10000 (2D/3D), 1500 (Global)                                     */
    double box_min[2];         /* RngDep: x_min,y_min  or lat_min,lon_min [rad]                    */
    double box_max[2];
    /* medium */
    double z_grnd;             /* ground elevation [km]                                            */
    double tweak_abs;          /* abs_coeff, 0.3                                                   */
    double freq;               /* Hz, 0.1                                                          */
    /* source: (x,y,z) Cartesian; 2D uses src[2] only; Global: (z_src [km above sea level], lat [rad], lon [rad]) */
    double src[3];
    int32_t bounces;           /* max ground reflections; n_rec = bounces + 1                      */
    int32_t calc_amp;          /* CalcAmp: integrate the auxiliary (Jacobian) equations            */
    int32_t accum_per_segment; /* 1: WriteRays/WriteCaustics convention (segments 0..k-2, App. A-2; always for 2D)
                                  0: GeoAc_TravelTime(solution,k) convention (segments 0..k-1)     */
    int32_t reserved;
} geoac_params;

typedef struct geoac_ctx geoac_ctx;

/* Create a context for `variant` on CUDA device `device` (ordinal). Fails (NULL, *status set) without sm_100.
 *
 * Concurrency contract: a context owns per-launch scratch (claim counters, claim order, per-launch invariants, the
 * y_{k-1} history) that every trace reuses, so AT MOST ONE trace may be in flight per context, on ONE stream at a time:
 * calls on one context are serialised by the caller (the reference itself is single-threaded and non-reentrant,
 * Code/GeoAc/GeoAc.Parameters.h globals), and after geoac_trace_device the caller must synchronise the stream it passed
 * before the next call on that context (any entry point, geoac_set_params included) other than another
 * geoac_trace_device on the same stream.  Different contexts are
 * independent and may be driven from different host threads -- one context per device is how a front end uses
 * several GPUs (geoac_trace_multi below does exactly that). */
geoac_ctx* geoac_create(int variant, int device, int* status);
void       geoac_destroy(geoac_ctx* ctx);
const char* geoac_last_error(const geoac_ctx* ctx);     /* ctx may be NULL: last create() error    */

/* Fill `p` with the variant's defaults (Code/GeoAc/GeoAc.Parameters*.cpp, mains' local defaults). */
int geoac_default_params(int variant, geoac_params* p);

/* Stratified atmosphere (replaces Spline_Single_G2S, Code/Atmo/G2S_Spline1D.cpp:293-312 / G2S_GlobalSpline1D.cpp:305-322).
 * Arrays are the loader's output: z [km, sea-level based, NOT offset by r_earth], T [K], u,v [km/s] AFTER the
 * unit conversion and ground taper (use geoac_load_met_1d), rho [g/cm^3].  The spline slopes are computed inside
 * with the reference's Thomas recurrences.  Resets ctx params' vert_limit/range_limit like GeoAc_SetPropRegion. */
int geoac_set_atmosphere_1d(geoac_ctx* ctx, int n, const double* z, const double* T,
                            const double* u, const double* v, const double* rho);

/* Range-dependent atmosphere (replaces Spline_Multi_G2S + GeoAc_SetPropRegion, Code/Atmo/G2S_MultiDimSpline3D.cpp).
 * ax0/ax1: horizontal node coordinates (x,y [km] or lat,lon [rad]); axz: altitude [km, sea-level based];
 * fields are dense [n0][n1][nz] (z fastest), winds already tapered and in km/s. */
int geoac_set_atmosphere_3d(geoac_ctx* ctx, int n0, int n1, int nz,
                            const double* ax0, const double* ax1, const double* axz,
                            const double* T, const double* u, const double* v, const double* rho);

int geoac_get_params(const geoac_ctx* ctx, geoac_params* p);
int geoac_set_params(geoac_ctx* ctx, const geoac_params* p);

/* Trace n_rays launch angles (radians; phi in the math convention pi/2 - azimuth, exactly the values the mains
 * store in GeoAc_theta / GeoAc_phi).  HOST buffers; copies angles H2D, runs the kernels, copies records D2H.
 *   rec     : GEOAC_NFIELDS * n_rays * (bounces+1) doubles (SoA, see field enum)
 *   status  : n_rays * (bounces+1) int32
 *   n_steps : n_rays * (bounces+1) int32  (k returned by GeoAc_Propagate_RK4 for that segment)            */
int geoac_trace(geoac_ctx* ctx, int64_t n_rays, const double* theta, const double* phi,
                double* rec, int32_t* status, int32_t* n_steps);

/* Same, but every pointer is a DEVICE pointer on ctx's device and the work is enqueued on `cuda_stream`
 * (a cudaStream_t passed as void*, NULL = default stream); returns without synchronising.  The call zeroes every record
 * slot before the trace, so the outputs need no initialisation.  Parameter and atmosphere changes made before the call are
 * ordered into `cuda_stream` by the call itself.  Calls that follow one another on the SAME stream need no synchronisation
 * between them (each one's work, the concurrent long-region launch of the range-dependent sets included, is complete
 * before the next one's starts); any other call on the context waits for a synchronisation of that stream (geoac_create).
 * Errors, returned before anything is enqueued: GEOAC_ERR_BAD_ARG (NULL context, n_rays < 0, a NULL pointer with
 * n_rays > 0), GEOAC_ERR_NO_ATMO; n_rays == 0 enqueues nothing and is GEOAC_OK whatever the pointers. */
int geoac_trace_device(geoac_ctx* ctx, int64_t n_rays, const double* d_theta, const double* d_phi,
                       double* d_rec, int32_t* d_status, int32_t* d_n_steps, void* cuda_stream);

/* geoac_trace() plus the raypath rows of the mains' WriteRays=True mode (Code/GeoAc3D_main.cpp:249-262 and siblings; the
 * same call serves `-interactive`, which plots one ray): every `path_stride` steps (the mains use 25) one row of
 * GEOAC_PATH_NF doubles { state[0], state[1], state[2], amplitude (linear, 0 with calc_amp = 0), absorption sum, travel-time
 * sum, bounce index, step index within the bounce } is stored for the ray, at most `path_cap` rows per ray:
 *   path      : n_rays * path_cap * GEOAC_PATH_NF doubles, row r of ray i at path[(i*path_cap + r)*GEOAC_PATH_NF]
 *   path_rows : n_rays int32, rows PRODUCED for the ray (if > path_cap the surplus was dropped)
 * The front end prints lat/lon in degrees, max(z, 0), 20 log10(amplitude) and -absorption exactly as it does today.
 * With caustic_cap > 0 the call also returns the WriteCaustics=True rows (:241-268): wherever the Jacobian determinant
 * (GeoAc_Jacobian) changes sign between consecutive steps, one row of GEOAC_CAUSTIC_NF doubles { state[0], state[1],
 * state[2], travel-time sum, bounce index, step index }, at most caustic_cap per ray (caustic / caustic_rows laid out like
 * path / path_rows; needs calc_amp = 1).  Either capture may be switched off (path_stride = 0 or caustic_cap = 0), not both.
 * Requires params.accum_per_segment = 1 (the accumulation convention of those modes, SURVEY App. A-2; always so for 2D). */
int geoac_trace_paths(geoac_ctx* ctx, int64_t n_rays, const double* theta, const double* phi,
                      double* rec, int32_t* status, int32_t* n_steps,
                      int path_stride, int64_t path_cap, double* path, int32_t* path_rows,
                      int64_t caustic_cap, double* caustic, int32_t* caustic_rows);

/* geoac_trace_paths with COMPACTED rows: ray i's raypath rows are path[path_offset[i] .. path_offset[i+1]) (rows of
 * GEOAC_PATH_NF doubles), its caustic events caustic[caustic_offset[i] .. caustic_offset[i+1]) (GEOAC_CAUSTIC_NF doubles);
 * path_offset / caustic_offset hold n_rays + 1 entries.  The rows are gathered on the device, so only rows that exist cross
 * PCIe (WriteRays=True on a config-2-size batch: 1.2 GB instead of the 3.3 GB of the dense [ray][cap] layout).  path_cap /
 * caustic_cap still bound the rows kept PER RAY; *_total_cap are the capacities of the output buffers in rows -- if one is too
 * small the call returns GEOAC_ERR_TOO_LARGE with the offsets filled in (the last offset is the number of rows to allocate). */
int geoac_trace_paths_compact(geoac_ctx* ctx, int64_t n_rays, const double* theta, const double* phi,
                              double* rec, int32_t* status, int32_t* n_steps,
                              int path_stride, int64_t path_cap, int64_t path_total_cap, double* path, int64_t* path_offset,
                              int64_t caustic_cap, int64_t caustic_total_cap, double* caustic, int64_t* caustic_offset);

/* ---- several devices behind one call (SURVEY 8b / 8e; the data-parallel axis is the launch-angle loop, Code/GeoAc3D_main.cpp:226-227) ----
 * A front end creates one context per device (geoac_create_multi, or geoac_create in a loop), gives every context the same
 * atmosphere and parameters (the geoac_multi_set_* helpers do that from one host thread per context) and traces with
 * geoac_trace_multi: the ray list is dealt to the contexts in interleaved blocks of GEOAC_SHARD_BLOCK rays, one host thread
 * per context stages its share through pinned memory owned by that context, traces it, and writes the records back at the
 * rays' own places in rec / status / n_steps (same layout as geoac_trace for the whole batch).  There is no exchange between
 * devices.  The result is bitwise what a single context returns.  device_ids may name a device twice (two contexts on one
 * GPU -- that is how the tests exercise the path on a one-GPU box).  Contexts are destroyed one by one with geoac_destroy.
 * On failure the message of the failing context is copied to ctxs[0] (geoac_last_error(ctxs[0])). */
enum { GEOAC_SHARD_BLOCK = 4096 };
int geoac_create_multi(int variant, const int* device_ids, int n_devices, geoac_ctx** ctxs, int* status);
int geoac_multi_set_atmosphere_1d(geoac_ctx* const* ctxs, int n_ctx, int n, const double* z, const double* T,
                                  const double* u, const double* v, const double* rho);
int geoac_multi_set_atmosphere_3d(geoac_ctx* const* ctxs, int n_ctx, int n0, int n1, int nz,
                                  const double* ax0, const double* ax1, const double* axz,
                                  const double* T, const double* u, const double* v, const double* rho);
int geoac_multi_set_params(geoac_ctx* const* ctxs, int n_ctx, const geoac_params* p);
int geoac_trace_multi(geoac_ctx* const* ctxs, int n_ctx, int64_t n_rays, const double* theta, const double* phi,
                      double* rec, int32_t* status, int32_t* n_steps);

/* Optional: page-locked host memory for the arrays handed to geoac_trace / geoac_trace_paths* / geoac_trace_multi (launch angles,
 * records, status, step counts, raypath rows).  The reference keeps its results in `new double*[...]` arrays
 * (GeoAc_BuildSolutionArray, Code/GeoAc/GeoAc.Interface.cpp:53-58), i.e. pageable memory, which the CUDA driver copies through
 * its own staging at a fraction of the PCIe rate; with buffers from geoac_host_alloc the 151 MB of records of a config-2 pass
 * cross at full rate (what bench.py's `e2e` leg measures with pinned buffers).  Any host memory works; this is the fast kind.
 * Returns NULL on failure (no device, out of memory).  geoac_host_free(NULL) is a no-op. */
void* geoac_host_alloc(size_t bytes);
void  geoac_host_free(void* p);

/* Optional: allocate the device staging geoac_trace() needs for batches of up to n_rays rays (with the current
 * `bounces`) ahead of time, so that the first trace call does not pay for it.  geoac_trace() grows it on demand anyway. */
int geoac_reserve(geoac_ctx* ctx, int64_t n_rays);

/* Total RK4 steps of the last trace on this ctx (sum of n_steps), and its duration in milliseconds (CUDA events).  After
 * the host-buffer calls the duration covers the work between the angle upload and the record download.  After
 * geoac_trace_device it covers the call's work on the caller's stream (zeroing, claim order, trace launches, join); both
 * values are valid once that stream has been synchronised, and kernel_ms is NaN while the work has not completed. */
int geoac_last_trace_stats(geoac_ctx* ctx, int64_t* total_steps, double* kernel_ms);

/* Host helper mirroring Load_G2S (Code/Atmo/G2S_Spline1D.cpp:109-142): read a .met profile ("zTuvdp" or "zuvwTdp"),
 * convert winds m/s -> km/s and apply the ground taper with `z_grnd_taper` (the mains always use 0, App. A-10).
 * `global_taper` selects the Global file's arithmetic (z is offset by r_earth before the taper, which changes
 * rounding).  Arrays must hold `cap` entries; *n receives the row count. */
int geoac_load_met_1d(const char* path, const char* format, double z_grnd_taper, int global_taper,
                      int cap, int* n, double* z, double* T, double* u, double* v, double* rho);

/* Host helper mirroring Load_G2S_Multi (Code/Atmo/G2S_MultiDimSpline3D.cpp:139-189, G2S_GlobalMultiDimSpline3D.cpp:142-199):
 * reads `<prefix><i0*n1+i1>.met` for every horizontal node plus the two node-coordinate files (x/y [km], or lat/lon
 * [deg] converted to radians when `global`), converts winds m/s -> km/s and applies the loader's ground taper.
 * Outputs are what geoac_set_atmosphere_3d expects; fields are [n0][n1][nz] with nz taken from the first profile
 * (T, u, v, rho must hold cap0*cap1*capz doubles if the node counts are not known in advance). */
int geoac_load_met_grid(const char* prefix, const char* loc0, const char* loc1, const char* format, int global,
                        int cap0, int cap1, int capz, int* n0, int* n1, int* nz,
                        double* ax0, double* ax1, double* axz, double* T, double* u, double* v, double* rho);

/* ---- eigenray search (SURVEY 8f-1): -eig_search of GeoAc3D, GeoAc3D.RngDep, GeoAcGlobal, GeoAcGlobal.RngDep ----
 * Replaces the loop of GeoAc3D_RunEigSearch (Code/GeoAc3D_main.cpp:531-541; GeoAc3D.RngDep_main.cpp likewise) including
 * GeoAc_EstimateEigenray (Code/GeoAc/GeoAc.Eigenray.cpp:30-121) and GeoAc_3DEigenray_LM (:123-335), and the Global
 * counterparts (Code/GeoAcGlobal_main.cpp:573-583, Code/GeoAc/GeoAc.Eigenray.Global.cpp:46-136, :139-320), for one source
 * and n_rcvr receivers at once.  Same decisions as the reference's one-ray-at-a-time search; the rays of all
 * receivers, bounce counts and brackets are traced in batches on the GPU (geoac_b200/csrc/eigenray.cu). */
typedef struct geoac_eig_opts {
    double theta_min, theta_max;   /* inclination limits [deg], 0.5 / 45 (GeoAc3D_main.cpp:461)                        */
    double azimuth_err_lim;        /* [deg] 2.0                                                                         */
    double d_theta_big;            /* 0.25  (Eigenray.cpp:20)                                                           */
    double d_theta_small;          /* 0.002 (Eigenray.cpp:21)                                                           */
    double tolerance;              /* [km] arrival-to-receiver distance that ends the LM search, 0.1 (Eigenray.cpp:139) */
    double src_lat_deg, src_lon_deg; /* Global variants only: the source as the Global mains hold it, in DEGREES (30, 0;
                                      GeoAcGlobal_main.cpp:497); the search launches from lat*Pi/180, lon*Pi/180 and
                                      params.src[0] (altitude).  Receivers are (lat, lon) in degrees there            */
    int32_t bnc_min, bnc_max;      /* bounce counts searched, 0 / 0                                                     */
    int32_t iterations;            /* LM iteration limit, 25                                                            */
    int32_t max_rounds;            /* safety limit on trace batches, 4096                                               */
} geoac_eig_opts;
int geoac_default_eig_opts(geoac_eig_opts* o);

/* One row per GeoAc_EstimateEigenray call, in the reference's order (receiver, bounce count, theta_start ascending):
 *  0 receiver index   1 bounce count   2 estimate succeeded   3 theta_estimate [deg]   4 phi_estimate [deg from the x axis]
 *  5 theta_next       6 eigenray found 7 theta [deg]          8 phi [deg from the x axis; azimuth = 90 - phi]
 *  9 travel time [s] 10 celerity [km/s] 11 amplitude (linear; the reference prints 20 log10)   12 absorption [dB], positive
 * 13 arrival inclination [deg]  14 back azimuth [deg]  15 azimuth deviation [deg]  16 LM iterations used  17 status of the
 *    final trace.  7, 8, 16 are set whenever the estimate succeeded (angles where the LM search stopped); 9-15, 17 only for
 *    eigenrays found.  A ray that ends on the step limit counts as having left the region (the reference would go on with
 *    the state at the limit). */
enum { GEOAC_EIG_NF = 18 };
/* rcvr_xy: n_rcvr pairs (x, y) [km], or (lat, lon) [deg] for the Global variants (phi columns 4, 8 are then 90 - azimuth, as
 * inside the reference).  rows: cap_rows * GEOAC_EIG_NF doubles; *n_rows = rows produced (GEOAC_ERR_TOO_LARGE
 * if more than cap_rows).  stats (may be NULL): [0] trace batches, [1] rays traced, [2] eigenrays found.  The raypath file
 * of an eigenray (<title>_Eigenray-N.dat) is geoac_trace_paths at (theta, phi) with accum_per_segment = 1, stride 25.
 * While it runs the call sets bounces / calc_amp / accum_per_segment (Global: the source) on the context and restores the
 * caller's parameters before it returns, on the error paths too. */
int geoac_eigenray_search(geoac_ctx* ctx, const geoac_eig_opts* opts, int n_rcvr, const double* rcvr_xy,
                          int64_t cap_rows, double* rows, int64_t* n_rows, int64_t* stats);

/* -eig_direct (GeoAc3D_RunEigDirect, Code/GeoAc3D_main.cpp:546-601, and the other three 3-D mains): GeoAc_3DEigenray_LM
 * alone, from caller-supplied estimates.  n searches at once: receiver i = rcvr_xy[2i..], estimates[3i..] = { theta_est
 * [deg], phi_est [deg from the x axis = 90 - azimuth], bounces }.  rows: n * GEOAC_EIG_NF doubles, same columns as above
 * (columns 3, 4 repeat the estimate; bnc_min / bnc_max / theta limits of opts are not used).  GeoAc3D (stratified) only:
 * in this mode the reference evaluates `if(GeoAc_AtmoStrat) M_Comps = ...` (Eigenray.cpp:130-135) before anything has set
 * that flag (GeoAc_ConfigureCalcAmp, :146), so it iterates with uninitialised Mach components; this entry point uses the
 * ones -eig_search uses, and finds the same eigenray within `tolerance` rather than the same digits. */
int geoac_eigenray_direct(geoac_ctx* ctx, const geoac_eig_opts* opts, int n, const double* rcvr_xy, const double* estimates,
                          double* rows, int64_t* stats);

/* Variant the context was created for; c, u, v, rho at the source point (device-sampled), 4 doubles. */
int geoac_get_variant(const geoac_ctx* ctx);
int geoac_source_state(geoac_ctx* ctx, double* out4);

/* Atmosphere as the kernels evaluate it, at n points given in the variant's own coordinates (the reference's Atmo_State.h
 * argument order): 2D / 3D / 3D.RngDep (x, y, z) [km]; Global / Global.RngDep (r [km from the Earth's centre, i.e.
 * r_earth + altitude], lat [rad], lon [rad]).  Stratified atmospheres use only the vertical coordinate.  Coordinates outside
 * the table / grid are clamped exactly as every reference look-up clamps them.  out: GEOAC_ATM_NF * n doubles, SoA,
 * out[f * n + i].  Absorption uses the context's params (freq, tweak_abs, z_grnd).  Synchronous, on ctx's stream; the same
 * concurrency contract as the trace calls.  Does not change anything a later trace reads or reports.
 * Replaces, as callers see them, c/u/v/rho, c_diff/u_diff/v_diff along the vertical, SuthBass_Alpha and Eval_Spline_AllOrder2
 * (Code/Atmo/Atmo_State.h:11-36).  Every point is evaluated as the reference would with cold cursors (accel = 0): a point
 * exactly on knot m falls in interval m-1 in the lower half of an axis and in interval m in the upper half.
 * Errors: GEOAC_ERR_BAD_ARG (NULL context, n < 0, a NULL pointer with n > 0, a non-finite coordinate -- the message names
 * the first such index), GEOAC_ERR_NO_ATMO; n == 0 writes nothing.  Points go through the device in passes of
 * GEOAC_SAMPLE_BLOCK. */
int geoac_sample_atmosphere(geoac_ctx* ctx, int64_t n, const double* p0, const double* p1, const double* p2, double* out);

/* Number of state equations for (variant, calc_amp): GeoAc_SetEqCnt, Code/GeoAc/GeoAc.Interface.cpp:21-41. */
int geoac_eq_count(int variant, int calc_amp);

/* Scheduling counters of the last trace.  warp_trips: trips round the kernel's step loop summed over warps -- lane
 * occupancy = total_steps / (32 * warp_trips), i.e. how full the warps were on average (ray lifetimes differ; finished
 * lanes are refilled until the batch is exhausted).  kernel_launches: kernels the call enqueued (1 trace kernel; plus, when the
 * longest-ray-first claim order was built, the cost scout and the sort: for the range-dependent sets the cost dilation (unless
 * knob "dilate" is 0), 3 counting-sort kernels and, with a long region of its own, a second trace launch; for the stratified sets
 * 8 kernels, whose order is (cost, inclination, batch index) in two stable passes).  Either pointer may be NULL. */
int geoac_last_trace_counters(geoac_ctx* ctx, int64_t* warp_trips, int64_t* kernel_launches);

/* Scheduling facts of the last trace on ctx (8 values): [0] reserved (0), [1] packets of the range-dependent sets in the long
 * region (predicted to outlast the pass on a loaded SM), [2] CTAs of the concurrent launch that traced them on SMs of their own, [3] kernels enqueued, [4] the longest of the long packets
 * that were split over four warps (quarter claims, four lanes per ray), [5..7] reserved (0). */
int geoac_last_schedule(geoac_ctx* ctx, int64_t* out8);
/* Test / diagnosis hook: the RK4 step counts the cost scout PREDICTED for the rays of the last trace (n entries, batch order). */
int geoac_get_costs(geoac_ctx* ctx, int64_t n, uint32_t* cost);
/* Durations [ms] of the trace kernel launch(es) of the last completed trace: ms2[0] main launch, ms2[1] long-region launch (or 0). */
int geoac_last_launch_ms(geoac_ctx* ctx, double* ms2);

/* Device self-test of the kernel's branch-free FP64 primitives against the CUDA math library on n_per_thread random
 * operands per thread: max_err[7] = maximum relative error of reciprocal, reciprocal square root, square root, exp, 10^x
 * and maximum absolute error of sin, cos (arguments within a few turns), in that order. */
int geoac_selftest_math(geoac_ctx* ctx, int n_per_thread, double* max_rel_err);

/* Test hook: copy the range-dependent node tables out of device memory exactly as the kernels read them --
 * tuv[n0][n1][nz][18] (per field T,u,v: f, z-slope, z-slope of df/dax0, z-slope of df/dax1, df/dax0, df/dax1) and
 * rho[n0][n1][nz][2] (f, z-slope).  These are what Set_Slopes_Multi builds (Code/Atmo/G2S_MultiDimSpline3D.cpp:306-425,
 * G2S_GlobalMultiDimSpline3D.cpp:313-431); geoac_set_atmosphere_3d builds them ON THE DEVICE (one thread per column and
 * quantity), and the parity tests compare them bit for bit with the reference's recurrences. cap_* in doubles. */
int geoac_get_grid_tables(geoac_ctx* ctx, int64_t cap_tuv, double* tuv, int64_t cap_rho, double* rho);

/* Tuning / experiment knobs of a context (DESIGN.md section 6).  Their defaults are read from the GEOAC_B200_* environment
 * variables ONCE, in geoac_create; nothing on the launch path reads the environment.  Names: "lpt" (claim order: 0 natural,
 * 1 automatic, 2 always), "scout_coarse", "cost_shift", "coop", "sbpoly", "host_tables", "long_alpha", "long_sm_pct", "exclusive",
 * "quarter", "quarter_alpha", "dilate"; any other name is GEOAC_ERR_BAD_ARG.
 * No knob changes a record bit except "sbpoly" (absorption sum to 1e-11) -- that is what the tests use them to prove. */
int geoac_set_knob(geoac_ctx* ctx, const char* name, int value);

/* FP64 DFMA micro-benchmark on ctx's device: returns measured TFLOP/s (2 flops per DFMA) -- the roofline denominator. */
double geoac_measure_fp64_peak(geoac_ctx* ctx, double* out_ms);

#ifdef __cplusplus
}
#endif
#endif /* GEOAC_B200_H_ */
