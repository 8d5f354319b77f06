// vrj_batch_inst.cu -- explicit instantiations of run_batch (vrj_batch.cuh); compiled once per value of VRJ_INST so that the
// kernel variants of the three (box type, real type) combinations, with and without traversal counters, build in parallel.
#include "vrj_batch.cuh"

#ifndef VRJ_INST
#error "compile with -DVRJ_INST=0..5"
#endif

namespace vrjimpl {
#if VRJ_INST == 0
template VrjStatus run_batch<float, double, false>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *); // the default path
#elif VRJ_INST == 1
template VrjStatus run_batch<float, double, true>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
#elif VRJ_INST == 2
template VrjStatus run_batch<double, double, false>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *); // VRJ_FILTER_F64
#elif VRJ_INST == 3
template VrjStatus run_batch<double, double, true>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
#elif VRJ_INST == 4
template VrjStatus run_batch<float, float, false>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *); // VRJ_PRECISION_F32_FAST
#else
template VrjStatus run_batch<float, float, true>(const VrjScene *, Scratch *, const RenderConst &, bool, int, uint64_t *);
#endif
} // namespace vrjimpl
