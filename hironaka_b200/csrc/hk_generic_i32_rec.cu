// warp-per-game kernel, int32 state, recorded rollouts (hk_rollout_record)
#include "hk_generic_launch.inl"
namespace hk {
int launch_generic_i32_rec(const StepParams& p, int dev, cudaStream_t stream) { return dispatch_generic_record<int32_t>(p, dev, stream); }
}  // namespace hk
