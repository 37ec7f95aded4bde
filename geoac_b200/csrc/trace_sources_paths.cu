// trace_sources_paths.cu -- the many-source capture kernels of geoac_trace_sources_paths_compact: trace_kernel over TraceArgsMS
// with PATHS = true (raypath rows and caustic events of rays from many sources), for the five variants x calc_amp and both
// table placements of the stratified sets.  The cost scout is the record path's (trace_sources.cu).  Kept out of capi.cu
// and trace_sources.cu so that the kernels there compile exactly as without them (trace_kernel.cuh: msrc_trace_kernel).
#define GEOAC_TRACE_KERNELS_ONLY
#include "core.cuh"
#include "eq_cartesian.cuh"
#include "eq_global.cuh"
#include "eq_rngdep.cuh"
#include "trace_kernel.cuh"

namespace geoac {

template <class EQ, int BLOCK, bool TABLE_IN_SMEM>
const void* msrc_paths_trace_kernel() { return (const void*)trace_kernel<EQ, BLOCK, TABLE_IN_SMEM, true, TraceArgsMS>; }

// the (equation set, lanes per CTA) pairs of capi.cu: dispatch_trace
#define GEOAC_MSRC_PATHS_STRATIFIED(EQ, BLOCK) \
    template const void* msrc_paths_trace_kernel<EQ, BLOCK, true>(); template const void* msrc_paths_trace_kernel<EQ, BLOCK, false>();
GEOAC_MSRC_PATHS_STRATIFIED(Eq2D<true>, 512)
GEOAC_MSRC_PATHS_STRATIFIED(Eq2D<false>, 512)
GEOAC_MSRC_PATHS_STRATIFIED(Eq3D<true>, 384)
GEOAC_MSRC_PATHS_STRATIFIED(Eq3D<false>, 512)
GEOAC_MSRC_PATHS_STRATIFIED(EqGlobal<true>, 384)
GEOAC_MSRC_PATHS_STRATIFIED(EqGlobal<false>, 512)
#undef GEOAC_MSRC_PATHS_STRATIFIED
template const void* msrc_paths_trace_kernel<Eq3DRD<true>, 128, false>();
template const void* msrc_paths_trace_kernel<Eq3DRD<false>, 128, false>();
template const void* msrc_paths_trace_kernel<EqGlobalRD<true>, 128, false>();
template const void* msrc_paths_trace_kernel<EqGlobalRD<false>, 128, false>();

}  // namespace geoac
