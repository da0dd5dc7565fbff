// warp-per-game kernel, float state: steps and rollouts (with the hot and census instantiations), and observation features
#include "hk_generic_launch.inl"
namespace hk {
template int dispatch_generic<float, GenericVariant::Plain>(const StepParams&, int, cudaStream_t);
template int dispatch_generic<float, GenericVariant::Obs>(const StepParams&, int, cudaStream_t);
}  // namespace hk
