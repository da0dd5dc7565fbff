// thread-per-game kernel, float state: steps and rollouts
#include "hk_small_launch.inl"
namespace hk {
template int dispatch_small<float, SmallVariant::Step>(const StepParams&, int, cudaStream_t);
}  // namespace hk
