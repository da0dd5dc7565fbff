// warp-per-game kernel, float state, recorded rollouts (hk_rollout_record)
#include "hk_generic_launch.inl"
namespace hk {
int launch_generic_f32_rec(const StepParams& p, int dev, cudaStream_t stream) { return dispatch_generic_record<float>(p, dev, stream); }
}  // namespace hk
