// hk_launch.cuh — launch helpers shared by the translation units of the library, and the
// launchers each unit defines.  The kernels are split over several .cu files (hk_small_*.cu,
// hk_generic_*.cu, hk_sched_*.cu, hk_rows_*.cu) only so that they compile in parallel; hk_capi.cu
// holds the extern "C" boundary and dispatches to these launchers.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstring>

#include "hk_common.cuh"

namespace hk {

constexpr int kMaxDevices = 64;

int device_sms(int dev);  // hk_capi.cu
bool use_pdl();           // hk_capi.cu (hk_debug_set_pdl)

// per-kernel, per-device launch facts (dynamic smem opt-in + resident CTAs per SM), computed once
struct KernelFacts {
    std::atomic<int> ctas_per_sm[kMaxDevices];
    KernelFacts() {
        for (auto& c : ctas_per_sm) c.store(0);
    }
};

template <typename K>
int kernel_ctas_per_sm(K kernel, KernelFacts& facts, int dev, int threads, size_t smem, cudaError_t* err) {
    int v = facts.ctas_per_sm[dev].load(std::memory_order_acquire);
    if (v > 0) return v;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
        *err = e;
        return 0;
    }
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, kernel, threads, smem);
    if (e != cudaSuccess) {
        *err = e;
        return 0;
    }
    if (v < 1) v = 1;
    facts.ctas_per_sm[dev].store(v, std::memory_order_release);
    return v;
}

__host__ __device__ constexpr bool is_small_shape(int N, int d) { return d == 3 && (N == 20 || N == 10 || N == 5); }

// one-launch paths of the two kernel families, one instantiation per (dtype, variant) in the hk_small_*.cu and
// hk_generic_*.cu units (hk_small_launch.inl, hk_generic_launch.inl)
template <typename T, SmallVariant V>
int dispatch_small(const StepParams& p, int dev, cudaStream_t stream);  // thread-per-game (hk_small.cuh)
template <typename T, GenericVariant V>
int dispatch_generic(const StepParams& p, int dev, cudaStream_t stream);  // warp-per-game (hk_generic.cuh)
extern template int dispatch_small<int32_t, SmallVariant::Step>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<int32_t, SmallVariant::Obs>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<int32_t, SmallVariant::Rec>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<int32_t, SmallVariant::Thr>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<int32_t, SmallVariant::ThrRec>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<float, SmallVariant::Step>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<float, SmallVariant::Obs>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<float, SmallVariant::Rec>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<float, SmallVariant::Thr>(const StepParams&, int, cudaStream_t);
extern template int dispatch_small<float, SmallVariant::ThrRec>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<int32_t, GenericVariant::Plain>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<int32_t, GenericVariant::Obs>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<int32_t, GenericVariant::Rec>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<int32_t, GenericVariant::Thr>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<int32_t, GenericVariant::ThrRec>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<float, GenericVariant::Plain>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<float, GenericVariant::Obs>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<float, GenericVariant::Rec>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<float, GenericVariant::Thr>(const StepParams&, int, cudaStream_t);
extern template int dispatch_generic<float, GenericVariant::ThrRec>(const StepParams&, int, cudaStream_t);
// census paths: the census-scheduled thread-per-game kernel (hk_sched.cuh), in-place single steps with p.census, OBS
// with the fused observation (sorted modes); and the small games of large padded shapes, thread-per-game on census
// masks (hk_rows.cuh).  One instantiation per unit (hk_sched_*.cu, hk_rows_*.cu)
template <typename T, bool OBS>
int dispatch_sched(const StepParams& p, int dev, cudaStream_t stream);
template <typename T>
int dispatch_rows(const StepParams& p, int dev, cudaStream_t stream);
extern template int dispatch_sched<int32_t, false>(const StepParams&, int, cudaStream_t);
extern template int dispatch_sched<int32_t, true>(const StepParams&, int, cudaStream_t);
extern template int dispatch_sched<float, false>(const StepParams&, int, cudaStream_t);
extern template int dispatch_sched<float, true>(const StepParams&, int, cudaStream_t);
extern template int dispatch_rows<int32_t>(const StepParams&, int, cudaStream_t);
extern template int dispatch_rows<float>(const StepParams&, int, cudaStream_t);
constexpr int ROWS_K = 8;  // = ROWS_MAX_K of hk_rows.cuh
__host__ __device__ constexpr bool rows_shape(int N, int d) { return N <= 64 && d >= 2 && d <= 5; }

}  // namespace hk
