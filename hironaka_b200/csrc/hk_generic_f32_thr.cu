// warp-per-game kernel, float state: rollouts with a value threshold, plain and recorded (hk_rollout_threshold)
#include "hk_generic_launch.inl"
namespace hk {
template int dispatch_generic<float, GenericVariant::Thr>(const StepParams&, int, cudaStream_t);
template int dispatch_generic<float, GenericVariant::ThrRec>(const StepParams&, int, cudaStream_t);
}  // namespace hk
