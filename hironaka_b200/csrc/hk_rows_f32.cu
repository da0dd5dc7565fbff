// small games of large padded shapes (hk_rows.cuh), float state
#include "hk_rows_launch.inl"
namespace hk {
template int dispatch_rows<float>(const StepParams&, int, cudaStream_t);
}  // namespace hk
