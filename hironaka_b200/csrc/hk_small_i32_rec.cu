// thread-per-game kernel, int32 state, recorded rollouts (hk_rollout_record)
#include "hk_small_launch.inl"
namespace hk {
int launch_small_i32_rec(const StepParams& p, int dev, cudaStream_t stream) { return dispatch_small_record<int32_t>(p, dev, stream); }
}  // namespace hk
