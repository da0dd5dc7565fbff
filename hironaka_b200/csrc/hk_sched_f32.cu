// census-scheduled thread-per-game kernel, float state
#include "hk_sched_launch.inl"
namespace hk {
template int dispatch_sched<float, false>(const StepParams&, int, cudaStream_t);
}  // namespace hk
