// thread-per-game kernel, int32 state: recorded rollouts (hk_rollout_record)
#include "hk_small_launch.inl"
namespace hk {
template int dispatch_small<int32_t, SmallVariant::Rec>(const StepParams&, int, cudaStream_t);
}  // namespace hk
