// warp-per-game kernel, float state, rollouts with a value threshold (hk_rollout_threshold)
#include "hk_generic_launch.inl"
namespace hk {
int launch_generic_f32_thr(const StepParams& p, bool rec, int dev, cudaStream_t stream) { return dispatch_generic_threshold<float>(p, rec, dev, stream); }
}  // namespace hk
