// trace_ensemble.cu -- the ensemble kernels of geoac_trace_ensemble: trace_kernel and scout_kernel over TraceArgsEns (each ray
// traced through its own member of an ensemble of 1-D profiles, with that member's invariants and table, both read from
// global memory) for the three stratified sets x calc_amp, and the set-up of the members' invariants and absorption
// polynomials.  Kept out of capi.cu so that the kernels there compile exactly as without them (trace_kernel.cuh:
// msrc_trace_kernel).
#define GEOAC_TRACE_KERNELS_ONLY
#include "core.cuh"
#include "eq_cartesian.cuh"
#include "eq_global.cuh"
#include "trace_kernel.cuh"

namespace geoac {

template <class EQ, int BLOCK>
const void* ens_trace_kernel() { return (const void*)trace_kernel<EQ, BLOCK, false, false, TraceArgsEns>; }
template <class EQ>
const void* ens_scout_kernel() { return (const void*)scout_kernel<EQ, false, TraceArgsEns>; }

// the (equation set, lanes per CTA) pairs of capi.cu: dispatch_trace
template const void* ens_trace_kernel<Eq2D<true>, 512>();
template const void* ens_trace_kernel<Eq2D<false>, 512>();
template const void* ens_trace_kernel<Eq3D<true>, 384>();
template const void* ens_trace_kernel<Eq3D<false>, 512>();
template const void* ens_trace_kernel<EqGlobal<true>, 384>();
template const void* ens_trace_kernel<EqGlobal<false>, 512>();
template const void* ens_scout_kernel<Eq2D<false>>();
template const void* ens_scout_kernel<Eq3D<false>>();
template const void* ens_scout_kernel<EqGlobal<false>>();

// One thread per member: the invariants of member m, as capi.cu's setup_consts_kernel builds them for a single table.
__global__ void ens_setup_consts_kernel(LaunchConsts* out, const LaunchConsts in, const Table1D* tab, int n_atm, int variant) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n_atm) return;
    const Table1D T = tab[m];
    LaunchConsts L = in;
    fill_launch_consts_1d(L, T, variant);
    out[m] = L;
}

// One thread per (member, interval): interval k of member m (iv_off[m] <= k < iv_off[m + 1]) with m's invariants, as capi.cu's
// build_sbpoly_kernel builds them for a single table.  Member m's block starts at poly + iv_off[m] * SBP_STRIDE.
__global__ void ens_build_sbpoly_kernel(const LaunchConsts* Lc, const Table1D* tab, const int64_t* iv_off, int n_atm, int64_t n_iv,
                                        int glob, double* poly) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_iv) return;
    int lo = 0, hi = n_atm - 1;                          // the member m with iv_off[m] <= k < iv_off[m + 1]
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (iv_off[mid] <= k) lo = mid; else hi = mid - 1; }
    const Table1D T = tab[lo];
    double o[SBP_STRIDE];
    sbpoly_build_interval(Lc[lo], T, glob != 0, (int)(k - iv_off[lo]), o);
    for (int i = 0; i < SBP_STRIDE; i++) poly[(size_t)k * SBP_STRIDE + i] = o[i];
}

cudaError_t ens_setup(LaunchConsts* out, const LaunchConsts& in, const Table1D* tab, int n_atm, const int64_t* iv_off, int64_t n_iv,
                      int variant, double* poly, cudaStream_t st) {
    ens_setup_consts_kernel<<<(n_atm + 31) / 32, 32, 0, st>>>(out, in, tab, n_atm, variant);
    ens_build_sbpoly_kernel<<<(unsigned)((n_iv + 63) / 64), 64, 0, st>>>(out, tab, iv_off, n_atm, n_iv, variant == GEOAC_GLOBAL, poly);
    return cudaGetLastError();
}

}  // namespace geoac
