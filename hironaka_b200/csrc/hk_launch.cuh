// hk_launch.cuh — launch helpers shared by the translation units of the library, and the
// per-dtype launcher functions each unit defines.  The kernels are split over several .cu files
// (hk_small_*.cu, hk_generic_*.cu) only so that they compile in parallel; hk_capi.cu holds the
// extern "C" boundary and dispatches to these launchers.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstring>

#include "hk_common.cuh"

namespace hk {

constexpr int kMaxDevices = 64;

int device_sms(int dev);  // hk_capi.cu
bool use_pdl();           // hk_capi.cu (hk_debug_set_pdl)
int sched_geometry();     // hk_capi.cu (hk_debug_set_sched_geometry)

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

inline bool is_small_shape(int N, int d) { return d == 3 && (N == 20 || N == 10 || N == 5); }

// thread-per-game family (hk_small.cuh); `obs` selects the instantiation that builds features
int launch_small_i32(const StepParams& p, bool obs, int dev, cudaStream_t stream);
int launch_small_f32(const StepParams& p, bool obs, int dev, cudaStream_t stream);
// census-scheduled thread-per-game kernel (hk_sched.cuh): in-place single steps with p.census
int launch_sched_i32(const StepParams& p, int dev, cudaStream_t stream);
int launch_sched_f32(const StepParams& p, int dev, cudaStream_t stream);
int launch_sched_i32_obs(const StepParams& p, int dev, cudaStream_t stream);  // + fused observation (sorted modes)
int launch_sched_f32_obs(const StepParams& p, int dev, cudaStream_t stream);
// small games of large padded shapes, thread-per-game on census masks (hk_rows.cuh)
int launch_rows_i32(const StepParams& p, int dev, cudaStream_t stream);
int launch_rows_f32(const StepParams& p, int dev, cudaStream_t stream);
constexpr int ROWS_K = 8;  // = ROWS_MAX_K of hk_rows.cuh
inline bool rows_shape(int N, int d) { return N <= 64 && d >= 2 && d <= 5; }
// warp-per-game family (hk_generic.cuh)
int launch_generic_i32(const StepParams& p, bool obs, int dev, cudaStream_t stream);
int launch_generic_f32(const StepParams& p, bool obs, int dev, cudaStream_t stream);
// recorded rollouts (hk_rollout_record), instantiations of their own in both families
int launch_small_i32_rec(const StepParams& p, int dev, cudaStream_t stream);
int launch_small_f32_rec(const StepParams& p, int dev, cudaStream_t stream);
int launch_generic_i32_rec(const StepParams& p, int dev, cudaStream_t stream);
int launch_generic_f32_rec(const StepParams& p, int dev, cudaStream_t stream);
// rollouts with a value threshold (hk_rollout_threshold), recorded (`rec`) or not, instantiations of their own in both families
int launch_small_i32_thr(const StepParams& p, bool rec, int dev, cudaStream_t stream);
int launch_small_f32_thr(const StepParams& p, bool rec, int dev, cudaStream_t stream);
int launch_generic_i32_thr(const StepParams& p, bool rec, int dev, cudaStream_t stream);
int launch_generic_f32_thr(const StepParams& p, bool rec, int dev, cudaStream_t stream);

}  // namespace hk
