// thread-per-game kernel, float state, rollouts with a value threshold (hk_rollout_threshold)
#include "hk_small_launch.inl"
namespace hk {
int launch_small_f32_thr(const StepParams& p, bool rec, int dev, cudaStream_t stream) { return dispatch_small_threshold<float>(p, rec, dev, stream); }
}  // namespace hk
