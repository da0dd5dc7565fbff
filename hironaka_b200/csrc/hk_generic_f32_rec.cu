// warp-per-game kernel, float state: recorded rollouts (hk_rollout_record)
#include "hk_generic_launch.inl"
namespace hk {
template int dispatch_generic<float, GenericVariant::Rec>(const StepParams&, int, cudaStream_t);
}  // namespace hk
