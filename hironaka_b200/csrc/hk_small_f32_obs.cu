// thread-per-game kernel, float state: steps with observation features
#include "hk_small_launch.inl"
namespace hk {
template int dispatch_small<float, SmallVariant::Obs>(const StepParams&, int, cudaStream_t);
}  // namespace hk
