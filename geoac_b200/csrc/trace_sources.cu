// trace_sources.cu -- the many-source record kernels of geoac_trace_sources: trace_kernel and scout_kernel over TraceArgsMS
// (each ray traced with the invariants of its own source), for the five variants x calc_amp and both table placements of the
// stratified sets.  Kept out of capi.cu so that the single-source kernels there compile exactly as without them
// (trace_kernel.cuh: msrc_trace_kernel).
#define GEOAC_TRACE_KERNELS_ONLY
#include "core.cuh"
#include "eq_cartesian.cuh"
#include "eq_global.cuh"
#include "eq_rngdep.cuh"
#include "trace_kernel.cuh"

namespace geoac {

template <class EQ, int BLOCK, bool TABLE_IN_SMEM>
const void* msrc_trace_kernel() { return (const void*)trace_kernel<EQ, BLOCK, TABLE_IN_SMEM, false, TraceArgsMS>; }
template <class EQ, bool TABLE_IN_SMEM>
const void* msrc_scout_kernel() { return (const void*)scout_kernel<EQ, TABLE_IN_SMEM, TraceArgsMS>; }

// the (equation set, lanes per CTA) pairs of capi.cu: dispatch_trace
#define GEOAC_MSRC_STRATIFIED(EQ, BLOCK) \
    template const void* msrc_trace_kernel<EQ, BLOCK, true>(); template const void* msrc_trace_kernel<EQ, BLOCK, false>();
GEOAC_MSRC_STRATIFIED(Eq2D<true>, 512)
GEOAC_MSRC_STRATIFIED(Eq2D<false>, 512)
GEOAC_MSRC_STRATIFIED(Eq3D<true>, 384)
GEOAC_MSRC_STRATIFIED(Eq3D<false>, 512)
GEOAC_MSRC_STRATIFIED(EqGlobal<true>, 384)
GEOAC_MSRC_STRATIFIED(EqGlobal<false>, 512)
#undef GEOAC_MSRC_STRATIFIED
template const void* msrc_trace_kernel<Eq3DRD<true>, 128, false>();
template const void* msrc_trace_kernel<Eq3DRD<false>, 128, false>();
template const void* msrc_trace_kernel<EqGlobalRD<true>, 128, false>();
template const void* msrc_trace_kernel<EqGlobalRD<false>, 128, false>();

template const void* msrc_scout_kernel<Eq2D<false>, true>();
template const void* msrc_scout_kernel<Eq2D<false>, false>();
template const void* msrc_scout_kernel<Eq3D<false>, true>();
template const void* msrc_scout_kernel<Eq3D<false>, false>();
template const void* msrc_scout_kernel<EqGlobal<false>, true>();
template const void* msrc_scout_kernel<EqGlobal<false>, false>();
template const void* msrc_scout_kernel<Eq3DRD<false>, false>();
template const void* msrc_scout_kernel<EqGlobalRD<false>, false>();

}  // namespace geoac
