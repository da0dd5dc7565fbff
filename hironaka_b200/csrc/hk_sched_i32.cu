// census-scheduled thread-per-game kernel, int32_t state
#include "hk_sched_launch.inl"
namespace hk {
template int dispatch_sched<int32_t, false>(const StepParams&, int, cudaStream_t);
}  // namespace hk
