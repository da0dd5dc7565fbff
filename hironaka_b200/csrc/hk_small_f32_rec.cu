// thread-per-game kernel, float state: recorded rollouts (hk_rollout_record)
#include "hk_small_launch.inl"
namespace hk {
template int dispatch_small<float, SmallVariant::Rec>(const StepParams&, int, cudaStream_t);
}  // namespace hk
