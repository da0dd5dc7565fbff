// thread-per-game kernel, float state, recorded rollouts (hk_rollout_record)
#include "hk_small_launch.inl"
namespace hk {
int launch_small_f32_rec(const StepParams& p, int dev, cudaStream_t stream) { return dispatch_small_record<float>(p, dev, stream); }
}  // namespace hk
