// warp-per-game kernel, int32 state: steps and rollouts (with the hot and census instantiations), and observation features
#include "hk_generic_launch.inl"
namespace hk {
template int dispatch_generic<int32_t, GenericVariant::Plain>(const StepParams&, int, cudaStream_t);
template int dispatch_generic<int32_t, GenericVariant::Obs>(const StepParams&, int, cudaStream_t);
}  // namespace hk
