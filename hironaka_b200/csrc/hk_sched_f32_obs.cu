// census-scheduled thread-per-game kernel with the fused observation, float state
#include "hk_sched_launch.inl"
namespace hk {
template int dispatch_sched<float, true>(const StepParams&, int, cudaStream_t);
}  // namespace hk
