// thread-per-game kernel, int32 state: rollouts with a value threshold, plain and recorded (hk_rollout_threshold)
#include "hk_small_launch.inl"
namespace hk {
template int dispatch_small<int32_t, SmallVariant::Thr>(const StepParams&, int, cudaStream_t);
template int dispatch_small<int32_t, SmallVariant::ThrRec>(const StepParams&, int, cudaStream_t);
}  // namespace hk
