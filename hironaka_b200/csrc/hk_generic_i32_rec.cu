// warp-per-game kernel, int32 state: recorded rollouts (hk_rollout_record)
#include "hk_generic_launch.inl"
namespace hk {
template int dispatch_generic<int32_t, GenericVariant::Rec>(const StepParams&, int, cudaStream_t);
}  // namespace hk
