// thread-per-game kernel, int32 state: steps with observation features
#include "hk_small_launch.inl"
namespace hk {
template int dispatch_small<int32_t, SmallVariant::Obs>(const StepParams&, int, cudaStream_t);
}  // namespace hk
