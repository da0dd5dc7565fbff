// warp-per-game kernel, int32 state: rollouts with a value threshold, plain and recorded (hk_rollout_threshold)
#include "hk_generic_launch.inl"
namespace hk {
template int dispatch_generic<int32_t, GenericVariant::Thr>(const StepParams&, int, cudaStream_t);
template int dispatch_generic<int32_t, GenericVariant::ThrRec>(const StepParams&, int, cudaStream_t);
}  // namespace hk
