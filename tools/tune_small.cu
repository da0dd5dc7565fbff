// tune_small.cu — standalone tuning harness for the thread-per-game kernel (not part of the product).
// Plays R random-play rollouts of the C2 workload (N=20, d=3, 1 Mi games) with several warps-per-CTA
// counts and prints the mean launch time by rollout step for each, plus a state checksum.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o tune_small tools/tune_small.cu
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

#include "../hironaka_b200/csrc/hk_small.cuh"

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

constexpr int N = 20, D = 3, T = 20;
#ifndef TUNE_EXTRA_FLAGS
#define TUNE_EXTRA_FLAGS 0u
#endif

template <int WARPS, bool OBS = false>
float launch(const hk::StepParams& p, cudaStream_t st, int sms, bool time_it, cudaEvent_t e0, cudaEvent_t e1) {
    using L = hk::SmallLayout<N, D, OBS, WARPS>;
    auto k = hk::hk_small_kernel<int32_t, N, D, false, WARPS, true, OBS ? hk::SmallVariant::Obs : hk::SmallVariant::Step>;
    static int per_sm = 0;
    if (!per_sm) {
        CK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::SMEM_BYTES));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, WARPS * 32, L::SMEM_BYTES));
        printf("  [W=%d OBS=%d] smem/CTA=%zu B, CTAs/SM=%d, warps/SM=%d\n", WARPS, (int)OBS, L::SMEM_BYTES, per_sm, per_sm * WARPS);
    }
    long long ntiles = (p.B + 31) / 32;
    long long ctas = (ntiles + WARPS - 1) / WARPS;
    long long cap = (long long)sms * per_sm;
    if (ctas > cap) ctas = cap;
    if (time_it) CK(cudaEventRecord(e0, st));
    k<<<(unsigned)ctas, WARPS * 32, L::SMEM_BYTES, st>>>(p);
    if (time_it) CK(cudaEventRecord(e1, st));
    CK(cudaGetLastError());
    return 0.f;
}

template <int WARPS, bool OBS = false>
void run_variant(int B, int R, const std::vector<int32_t>& pts, const std::vector<int32_t>& ha, const std::vector<int32_t>& ax) {
    int sms = 148;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    int32_t *d_state, *d_ha, *d_ax; uint8_t* d_done; float* d_rew;
    size_t sbytes = (size_t)B * N * D * 4;
    CK(cudaMalloc(&d_state, sbytes * R)); CK(cudaMalloc(&d_ha, (size_t)R * T * B * 4)); CK(cudaMalloc(&d_ax, (size_t)R * T * B * 4));
    CK(cudaMalloc(&d_done, B)); CK(cudaMalloc(&d_rew, (size_t)B * 4));
    float* d_obs = nullptr;
    if (OBS) CK(cudaMalloc(&d_obs, sbytes));
    CK(cudaMemcpy(d_state, pts.data(), sbytes * R, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ha, ha.data(), (size_t)R * T * B * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ax, ax.data(), (size_t)R * T * B * 4, cudaMemcpyHostToDevice));
    cudaStream_t st; CK(cudaStreamCreate(&st));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    hk::StepParams p; memset(&p, 0, sizeof(p));
    p.B = B; p.N = N; p.d = D; p.T = 1; p.pad = -1.f; p.threshold = 1e8f;
    std::vector<double> by_step(T, 0.0); double init_ms = 0;
    for (int r = 0; r < R; ++r) {
        int32_t* s = d_state + (size_t)r * B * N * D;
        p.in = s; p.out = s; p.ops = HK_OP_NEWTON | HK_OP_REPOSITION; p.flags = 0; p.host_action = nullptr; p.axis = nullptr; p.done = nullptr; p.reward = nullptr;
        launch<WARPS, false>(p, st, sms, true, e0, e1);
        CK(cudaEventSynchronize(e1)); float ms; CK(cudaEventElapsedTime(&ms, e0, e1)); init_ms += ms;
        p.ops = HK_OP_SHIFT | HK_OP_REPOSITION | HK_OP_NEWTON; p.flags = HK_F_ACT_DISCRETE | TUNE_EXTRA_FLAGS; p.done = d_done; p.reward = d_rew;
        if (OBS) { p.obs = d_obs; p.flags |= HK_F_OBS_SORT_LEX | HK_F_OBS_RESCALE; }
        for (int t = 0; t < T; ++t) {
            p.host_action = d_ha + ((size_t)r * T + t) * B; p.axis = d_ax + ((size_t)r * T + t) * B;
            launch<WARPS, OBS>(p, st, sms, true, e0, e1);
            CK(cudaEventSynchronize(e1)); CK(cudaEventElapsedTime(&ms, e0, e1));
            if (r > 0) by_step[t] += ms;  // rollout 0 is warm-up
        }
    }
    {   // floor of this data path: the same kernel with no op selected (load tile, store tile), and a plain D2D memcpy
        p.ops = 0; p.flags = 0; p.host_action = nullptr; p.axis = nullptr; p.done = nullptr; p.reward = nullptr; p.obs = nullptr;
        double cp = 0, mc = 0; float ms;
        for (int i = 0; i < 12; ++i) {
            int32_t* s = d_state + (size_t)(i % R) * B * N * D; p.in = s; p.out = s;
            launch<WARPS, false>(p, st, sms, true, e0, e1);
            CK(cudaEventSynchronize(e1)); CK(cudaEventElapsedTime(&ms, e0, e1)); if (i >= 2) cp += ms;
        }
        for (int i = 0; i < 12; ++i) {
            CK(cudaEventRecord(e0, st));
            CK(cudaMemcpyAsync(d_state + (size_t)((i + 1) % R) * B * N * D, d_state + (size_t)(i % R) * B * N * D, sbytes, cudaMemcpyDeviceToDevice, st));
            CK(cudaEventRecord(e1, st));
            CK(cudaEventSynchronize(e1)); CK(cudaEventElapsedTime(&ms, e0, e1)); if (i >= 2) mc += ms;
        }
        printf("  copy-only kernel %.2f us (%.0f GB/s r+w) | cudaMemcpy D2D %.2f us (%.0f GB/s r+w)\n", 1e3 * cp / 10, 2.0 * sbytes / (cp / 10 * 1e-3) / 1e9,
               1e3 * mc / 10, 2.0 * sbytes / (mc / 10 * 1e-3) / 1e9);
    }
    CK(cudaStreamSynchronize(st));
    std::vector<int32_t> out((size_t)B * N * D);
    CK(cudaMemcpy(out.data(), d_state, sbytes, cudaMemcpyDeviceToHost));
    unsigned long long cs = 1469598103934665603ull;
    for (size_t i = 0; i < out.size(); ++i) cs = (cs ^ (unsigned)out[i]) * 1099511628211ull;
    double tot = 0; for (int t = 0; t < T; ++t) { by_step[t] /= (R - 1); tot += by_step[t]; }
    printf("W=%d OBS=%d: init %.1f us | mean/step %.2f us (%.3f of 6543.7 GB/s) | t0..t4: %.1f %.1f %.1f %.1f %.1f | t5..19 mean %.2f | checksum %016llx\n",
           WARPS, (int)OBS, 1e3 * init_ms / R, 1e3 * tot / T, (double)B * (OBS ? 733 : 493) / (tot / T * 1e-3) / 6543.7e9,
           1e3 * by_step[0], 1e3 * by_step[1], 1e3 * by_step[2], 1e3 * by_step[3], 1e3 * by_step[4],
           1e3 * (tot - by_step[0] - by_step[1] - by_step[2] - by_step[3] - by_step[4]) / 15, cs);
    cudaFree(d_state); cudaFree(d_ha); cudaFree(d_ax); cudaFree(d_done); cudaFree(d_rew);
}

// one-launch T-step rollouts (hk_rollout): state read and written once per T steps
template <int WARPS>
void run_rollout(int B, int R, const std::vector<int32_t>& pts, const std::vector<int32_t>& ha, const std::vector<int32_t>& ax) {
    int sms = 148;
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, 0));
    int32_t *d_state, *d_ha, *d_ax, *d_cnt;
    size_t sbytes = (size_t)B * N * D * 4;
    CK(cudaMalloc(&d_state, sbytes * R)); CK(cudaMalloc(&d_ha, (size_t)R * T * B * 4)); CK(cudaMalloc(&d_ax, (size_t)R * T * B * 4));
    CK(cudaMalloc(&d_cnt, T * 4)); CK(cudaMemset(d_cnt, 0, T * 4));
    CK(cudaMemcpy(d_state, pts.data(), sbytes * R, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ha, ha.data(), (size_t)R * T * B * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_ax, ax.data(), (size_t)R * T * B * 4, cudaMemcpyHostToDevice));
    cudaStream_t st; CK(cudaStreamCreate(&st));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    hk::StepParams p; memset(&p, 0, sizeof(p));
    p.B = B; p.N = N; p.d = D; p.pad = -1.f; p.threshold = 1e8f;
    double tot = 0;
    for (int r = 0; r < R; ++r) {
        int32_t* s = d_state + (size_t)r * B * N * D;
        p.in = s; p.out = s; p.T = 1; p.ops = HK_OP_NEWTON | HK_OP_REPOSITION; p.flags = 0; p.host_action = nullptr; p.axis = nullptr; p.done_count = nullptr;
        launch<WARPS>(p, st, sms, false, e0, e1);
        p.T = T; p.ops = HK_OP_SHIFT | HK_OP_REPOSITION | HK_OP_NEWTON; p.flags = HK_F_ACT_DISCRETE; p.done_count = d_cnt;
        p.host_action = d_ha + (size_t)r * T * B; p.axis = d_ax + (size_t)r * T * B;
        launch<WARPS>(p, st, sms, true, e0, e1);
        CK(cudaEventSynchronize(e1)); float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
        if (r > 0) tot += ms;
    }
    std::vector<int32_t> out((size_t)B * N * D);
    CK(cudaMemcpy(out.data(), d_state, sbytes, cudaMemcpyDeviceToHost));
    unsigned long long cs = 1469598103934665603ull;
    for (size_t i = 0; i < out.size(); ++i) cs = (cs ^ (unsigned)out[i]) * 1099511628211ull;
    printf("ROLLOUT W=%d: %.3f ms per %d-step rollout = %.3e game-steps/s | checksum %016llx\n", WARPS, tot / (R - 1), T,
           (double)B * T / (tot / (R - 1) * 1e-3), cs);
    cudaFree(d_state); cudaFree(d_ha); cudaFree(d_ax); cudaFree(d_cnt);
}

int main(int argc, char** argv) {
    int B = 1 << 20, R = 4;
    std::mt19937 rng(7);
    std::vector<int32_t> pts((size_t)R * B * N * D), ha((size_t)R * T * B), ax((size_t)R * T * B);
    for (auto& v : pts) v = rng() % 20;
    for (auto& v : ha) v = rng() % 4;
    for (auto& v : ax) v = rng() % 3;
#include "tune_variants.inc"
    return 0;
}
