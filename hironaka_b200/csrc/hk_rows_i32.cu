// small games of large padded shapes (hk_rows.cuh), int32_t state
#include "hk_rows_launch.inl"
namespace hk {
template int dispatch_rows<int32_t>(const StepParams&, int, cudaStream_t);
}  // namespace hk
