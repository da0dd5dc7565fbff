// hk_capi.cu — the extern "C" boundary declared in include/hironaka_b200.h.
//
// Device entry points validate arguments, pick the kernel family for (dtype, N, d) and launch
// on the caller's stream; they never allocate or synchronise.  Host-buffer sessions own the
// device state of one shard and wrap the same launches with explicit H2D / D2H copies.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <new>

#include "hk_census.cuh"
#include "hk_experience.cuh"
#include "hk_launch.cuh"
#include "hk_value.cuh"

using hk::GenericVariant;
using hk::SmallVariant;
using hk::StepParams;
using hk::kMaxDevices;

namespace {

std::atomic<int> g_use_pdl{0};  // programmatic dependent launch of the thread-per-game kernel (hk_debug_set_pdl)

struct DevInfo {
    std::atomic<int> sms{0};
};
DevInfo g_dev[kMaxDevices];

int device_sms_impl(int dev) {
    if (dev < 0 || dev >= kMaxDevices) return 148;
    int v = g_dev[dev].sms.load(std::memory_order_relaxed);
    if (v == 0) {
        cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev);
        if (v <= 0) v = 148;
        g_dev[dev].sms.store(v, std::memory_order_relaxed);
    }
    return v;
}

int check_shape(long long B, int N, int d, int dtype) {
    if (B < 0 || N < 1 || d < 1) return HK_ERR_BAD_ARG;
    if (dtype != HK_DTYPE_I32 && dtype != HK_DTYPE_F32) return HK_ERR_BAD_ARG;
    if (d > HK_MAX_DIM || N > HK_MAX_POINTS || (long long)N * d > HK_MAX_GAME_WORDS) return HK_ERR_UNSUPPORTED;
    return HK_OK;
}

// the variant of the one-launch kernels a call needs, from the outputs it asks for
SmallVariant rollout_variant(const StepParams& p) {
    const bool rec = p.obs_t || p.host_mask_t || p.axis_played_t;
    if (p.over_step || p.stop_at_threshold) return rec ? SmallVariant::ThrRec : SmallVariant::Thr;
    if (rec) return SmallVariant::Rec;
    return p.obs ? SmallVariant::Obs : SmallVariant::Step;
}

// the thread-per-game family (`small`) or the warp-per-game family, in variant V
template <typename T, SmallVariant V>
int launch_variant(const StepParams& p, bool small, int dev, cudaStream_t stream) {
    return small ? hk::dispatch_small<T, V>(p, dev, stream) : hk::dispatch_generic<T, hk::generic_variant(V)>(p, dev, stream);
}

template <typename T>
int launch_family(const StepParams& p, bool small, int dev, cudaStream_t stream) {
    switch (rollout_variant(p)) {
        case SmallVariant::Step: return launch_variant<T, SmallVariant::Step>(p, small, dev, stream);
        case SmallVariant::Obs: return launch_variant<T, SmallVariant::Obs>(p, small, dev, stream);
        case SmallVariant::Rec: return launch_variant<T, SmallVariant::Rec>(p, small, dev, stream);
        case SmallVariant::Thr: return launch_variant<T, SmallVariant::Thr>(p, small, dev, stream);
        case SmallVariant::ThrRec: return launch_variant<T, SmallVariant::ThrRec>(p, small, dev, stream);
    }
    return HK_ERR_UNSUPPORTED;
}

int run(StepParams& p, int dtype, int force_generic, cudaStream_t stream) {
    int rc = check_shape(p.B, p.N, p.d, dtype);
    if (rc != HK_OK) return rc;
    if (p.B == 0) return HK_OK;  // empty batch: nothing to do (an empty tensor has a null data pointer)
    if (p.in == nullptr) return HK_ERR_BAD_ARG;
    if ((((uintptr_t)p.in) & 3u) || (((uintptr_t)p.out) & 3u)) return HK_ERR_ALIGN;
    {
        const bool host_fixed = p.flags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER | HK_F_HOST_RANDOM);
        const bool agent_fixed = p.flags & (HK_F_AGENT_FIRST | HK_F_AGENT_LAST | HK_F_AGENT_RANDOM);
        if ((p.flags & HK_F_HOST_RANDOM) && (p.flags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER))) return HK_ERR_BAD_ARG;
        if ((p.flags & HK_F_AGENT_RANDOM) && (p.flags & (HK_F_AGENT_FIRST | HK_F_AGENT_LAST))) return HK_ERR_BAD_ARG;
        if ((p.flags & HK_F_HOST_ALL_COORD) && (p.flags & HK_F_HOST_ZEILLINGER)) return HK_ERR_BAD_ARG;
        if ((p.flags & HK_F_AGENT_FIRST) && (p.flags & HK_F_AGENT_LAST)) return HK_ERR_BAD_ARG;
        const bool nibble = p.flags & HK_F_ACT_NIBBLE;
        const bool packed = (p.flags & HK_F_ACT_PACKED) || nibble;
        if ((p.flags & HK_F_ACT_PACKED) && nibble) return HK_ERR_BAD_ARG;
        if (packed && (host_fixed || agent_fixed || p.d > 5)) return HK_ERR_BAD_ARG;
        if (nibble && (p.d > 3 || !(p.flags & HK_F_ACT_DISCRETE))) return HK_ERR_BAD_ARG;
        if (host_fixed) p.host_action = nullptr;
        if (agent_fixed || packed) p.axis = nullptr;
        if ((p.ops & HK_OP_SHIFT) &&
            ((!host_fixed && p.host_action == nullptr) || (!agent_fixed && !packed && p.axis == nullptr)))
            return HK_ERR_BAD_ARG;
    }
    if ((p.ops & HK_OP_RESCALE) && dtype != HK_DTYPE_F32) return HK_ERR_UNSUPPORTED;
    if (p.ops & ~(HK_OP_SHIFT | HK_OP_REPOSITION | HK_OP_NEWTON | HK_OP_RESCALE | HK_OP_DEDUPE)) return HK_ERR_BAD_ARG;
    {
        const uint32_t sm = p.flags & (HK_F_OBS_SORT_COORD0 | HK_F_OBS_SORT_LEX | HK_F_OBS_SORT_LEX_FIRST);
        if (sm & (sm - 1)) return HK_ERR_BAD_ARG;  // at most one sort mode
    }
    if (p.T < 1) return HK_ERR_BAD_ARG;
    if (p.B == 0) return HK_OK;
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    const bool obs = p.obs != nullptr;
    if (p.done_bits && !p.census) return HK_ERR_UNSUPPORTED;  // the bit mask is an output of the census path
    if (p.census) {
        // the census path: in-place single steps without fused observation or in-kernel players
        const bool policy = p.flags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER | HK_F_AGENT_FIRST | HK_F_AGENT_LAST);
        if (p.out != p.in || p.T != 1 || policy || p.host_out || p.ops == 0) return HK_ERR_UNSUPPORTED;
        const bool sched = hk::is_small_shape(p.N, p.d) && !force_generic && !(p.ops & HK_OP_DEDUPE);
        // a fused observation rides on the census only for the thread-per-game shapes and the sorted modes (the
        // observation of a game at rest is then a constant)
        if (obs && !(sched && (p.flags & (HK_F_OBS_SORT_COORD0 | HK_F_OBS_SORT_LEX | HK_F_OBS_SORT_LEX_FIRST))))
            return HK_ERR_UNSUPPORTED;
        if (sched && obs)
            return dtype == HK_DTYPE_I32 ? hk::dispatch_sched<int32_t, true>(p, dev, stream)
                                         : hk::dispatch_sched<float, true>(p, dev, stream);
        if (sched)
            return dtype == HK_DTYPE_I32 ? hk::dispatch_sched<int32_t, false>(p, dev, stream)
                                         : hk::dispatch_sched<float, false>(p, dev, stream);
        // Large padded shapes with at most 64 rows: the census carries a live mask per game after the bytes, and the
        // games with few live rows are stepped thread-per-game on their live rows alone (hk_rows_kernel) before
        // the warp-per-game kernel takes the rest.
        if (hk::rows_shape(p.N, p.d) && !(p.ops & HK_OP_DEDUPE)) {
            p.live_mask = reinterpret_cast<uint64_t*>(p.census + hk::census_mask_offset(p.B));
            int rc2 = dtype == HK_DTYPE_I32 ? hk::dispatch_rows<int32_t>(p, dev, stream) : hk::dispatch_rows<float>(p, dev, stream);
            if (rc2 != HK_OK) return rc2;
            p.rows_k = hk::ROWS_K;
        } else if (p.done_bits) {  // the warp-per-game kernel ORs the bits in, one game at a time
            e = cudaMemsetAsync(p.done_bits, 0, (size_t)((p.B + 31) / 32) * 4, stream);
            if (e != cudaSuccess) return (int)e;
        }
        return dtype == HK_DTYPE_I32 ? hk::dispatch_generic<int32_t, GenericVariant::Plain>(p, dev, stream)
                                     : hk::dispatch_generic<float, GenericVariant::Plain>(p, dev, stream);
    }
    // remove_repeated alone is not on the step path: it runs on the warp-per-game kernel for every shape
    const bool small = hk::is_small_shape(p.N, p.d) && !force_generic && !(p.ops & HK_OP_DEDUPE);
    return dtype == HK_DTYPE_I32 ? launch_family<int32_t>(p, small, dev, stream) : launch_family<float>(p, small, dev, stream);
}

StepParams make_params(const void* in, void* out, long long B, int N, int d, float pad) {
    StepParams p;
    memset(&p, 0, sizeof(p));
    p.in = in;
    p.out = out;
    p.B = B;
    p.N = N;
    p.d = d;
    p.T = 1;
    p.pad = pad;
    p.threshold = 1e8f;
    return p;
}

// the parameters of the one-launch rollouts (hk_rollout, hk_rollout_seeded, hk_rollout_record, and hk_rollout_threshold
// before its threshold).  Without a random player the seed and step offset are 0; the streams of a random player are
// dropped (run() drops them for every fixed or random player).
StepParams rollout_params(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
                          float* obs_t, int32_t agent_obs, int32_t* host_mask_t, int32_t* axis_played_t, uint8_t* done_t,
                          float* reward_t, int32_t* done_count, int32_t* length, long long B, int N, int d, int T,
                          uint32_t ops, uint32_t flags, float padding_value, uint64_t seed, int32_t step_offset) {
    const bool random = flags & (HK_F_HOST_RANDOM | HK_F_AGENT_RANDOM);
    StepParams p = make_params(state_in, state_out, B, N, d, padding_value);
    p.host_action = (flags & HK_F_HOST_RANDOM) ? nullptr : host_action_t;
    p.axis = (flags & HK_F_AGENT_RANDOM) ? nullptr : axis_t;
    p.obs_t = obs_t;
    p.agent_obs = agent_obs ? 1 : 0;
    p.host_mask_t = host_mask_t;
    p.axis_played_t = axis_played_t;
    p.done = done_t;
    p.reward = reward_t;
    p.done_count = done_count;
    p.length = length;
    p.T = T;
    p.ops = ops;
    p.flags = flags;
    p.seed = random ? seed : 0;
    p.step_offset = random ? step_offset : 0;
    return p;
}

std::atomic<int> g_force_generic{0};
std::atomic<int> g_no_session_graphs{0};  // test / tuning hook (hk_debug_set_session_graphs)

}  // namespace

namespace hk {
int device_sms(int dev) { return device_sms_impl(dev); }
bool use_pdl() { return g_use_pdl.load(std::memory_order_relaxed) != 0; }
}  // namespace hk

extern "C" {

int hk_version(void) { return HK_VERSION; }

const char* hk_error_string(int code) {
    switch (code) {
        case HK_OK: return "ok";
        case HK_ERR_BAD_ARG: return "bad argument (null pointer, non-positive size or bad flag combination)";
        case HK_ERR_UNSUPPORTED: return "unsupported shape or op for this dtype";
        case HK_ERR_ALIGN: return "state pointer is not 4-byte aligned";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown error";
    }
}

int hk_kernel_class(int N, int d) {
    if (check_shape(1, N, d, HK_DTYPE_I32) != HK_OK) return HK_ERR_UNSUPPORTED;
    return (hk::is_small_shape(N, d) && !g_force_generic.load()) ? 1 : 0;
}

// tuning hook: programmatic dependent launch on/off
int hk_debug_set_pdl(int on) {
    g_use_pdl.store(on ? 1 : 0);
    return HK_OK;
}

int64_t hk_census_bytes(int64_t B, int32_t N, int32_t d) {
    return B < 0 ? 0 : hk::census_bytes(B, N, d);
}

// test / tuning hook: host-buffer rollouts replayed as CUDA graphs (on by default)
int hk_debug_set_session_graphs(int on) {
    g_no_session_graphs.store(on ? 0 : 1);
    return HK_OK;
}

// test hook: route small shapes through the generic warp-per-game kernel as well
int hk_debug_force_generic(int on) {
    g_force_generic.store(on ? 1 : 0);
    return HK_OK;
}

int hk_step(const void* state_in, void* state_out, const int32_t* host_action, const int32_t* axis, uint8_t* done,
            float* reward, int32_t* num_points, float* obs, const int32_t* obs_coord, int32_t* exceed_flag,
            int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t ops, uint32_t flags, float padding_value,
            float value_threshold, void* stream) {
    StepParams p = make_params(state_in, state_out, B, N, d, padding_value);
    p.host_action = host_action;
    p.axis = axis;
    p.done = done;
    p.reward = reward;
    p.num_points = num_points;
    p.obs = obs;
    p.obs_coord = obs_coord;
    p.exceed_flag = exceed_flag;
    p.ops = ops;
    p.flags = flags;
    p.threshold = value_threshold;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_step_census_obs(void* state, const int32_t* host_action, const int32_t* axis, uint8_t* done, uint32_t* done_bits,
                       float* reward, int32_t* num_points, float* obs, const int32_t* obs_coord, uint8_t* census,
                       int32_t* done_count, int32_t* exceed_flag, int64_t B, int32_t N, int32_t d, int32_t dtype,
                       uint32_t ops, uint32_t flags, float padding_value, float value_threshold, void* stream) {
    if (census == nullptr || state == nullptr) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state, state, B, N, d, padding_value);
    p.host_action = host_action;
    p.axis = axis;
    p.done = done;
    p.done_bits = done_bits;
    p.reward = reward;
    p.num_points = num_points;
    p.obs = obs;
    p.obs_coord = obs_coord;
    p.census = census;
    p.done_count = done_count;
    p.exceed_flag = exceed_flag;
    p.ops = ops;
    p.flags = flags;
    p.threshold = value_threshold;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_step_census(void* state, const int32_t* host_action, const int32_t* axis, uint8_t* done, uint32_t* done_bits,
                   float* reward, int32_t* num_points, uint8_t* census, int32_t* done_count, int32_t* exceed_flag, int64_t B, int32_t N,
                   int32_t d, int32_t dtype, uint32_t ops, uint32_t flags, float padding_value, float value_threshold,
                   void* stream) {
    return hk_step_census_obs(state, host_action, axis, done, done_bits, reward, num_points, nullptr, nullptr, census,
                              done_count, exceed_flag, B, N, d, dtype, ops, flags, padding_value, value_threshold, stream);
}

int hk_shift(const void* state_in, void* state_out, const int32_t* host_action, const int32_t* axis, int64_t B,
             int32_t N, int32_t d, int32_t dtype, uint32_t flags, float padding_value, void* stream) {
    if (state_out == nullptr) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state_in, state_out, B, N, d, padding_value);
    p.host_action = host_action;
    p.axis = axis;
    p.ops = HK_OP_SHIFT;
    p.flags = flags;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_reposition(const void* state_in, void* state_out, int64_t B, int32_t N, int32_t d, int32_t dtype,
                  float padding_value, void* stream) {
    if (state_out == nullptr) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state_in, state_out, B, N, d, padding_value);
    p.ops = HK_OP_REPOSITION;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_newton_polytope(const void* state_in, void* state_out, int64_t B, int32_t N, int32_t d, int32_t dtype,
                       float padding_value, void* stream) {
    if (state_out == nullptr) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state_in, state_out, B, N, d, padding_value);
    p.ops = HK_OP_NEWTON;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_rescale(const void* state_in, void* state_out, int64_t B, int32_t N, int32_t d, int32_t dtype,
               float padding_value, void* stream) {
    if (state_out == nullptr) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state_in, state_out, B, N, d, padding_value);
    p.ops = HK_OP_RESCALE;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_features(const void* state_in, float* obs, const int32_t* obs_coord, int64_t B, int32_t N, int32_t d,
                int32_t dtype, uint32_t flags, float padding_value, void* stream) {
    if (obs == nullptr) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state_in, nullptr, B, N, d, padding_value);
    p.obs = obs;
    p.obs_coord = obs_coord;
    p.flags = flags;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_dones(const void* state_in, uint8_t* done, int32_t* num_points, int64_t B, int32_t N, int32_t d,
             int32_t dtype, void* stream) {
    if (done == nullptr && num_points == nullptr) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state_in, nullptr, B, N, d, -1.0f);
    p.done = done;
    p.num_points = num_points;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_host_policy(const void* state_in, int32_t* coord_mask, int64_t B, int32_t N, int32_t d, int32_t dtype,
                   uint32_t flags, float padding_value, void* stream) {
    if (coord_mask == nullptr) return HK_ERR_BAD_ARG;
    const uint32_t host = flags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER);
    if (host == 0 || host == (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER)) return HK_ERR_BAD_ARG;
    StepParams p = make_params(state_in, nullptr, B, N, d, padding_value);
    p.ops = HK_OP_SHIFT;  // the players are evaluated where the shift would use them; nothing is moved or written
    p.flags = host | HK_F_AGENT_FIRST;  // (the agent's choice is not used: nothing moves)
    p.host_out = coord_mask;
    return run(p, dtype, 1 /* the warp-per-game family evaluates it for every shape */, (cudaStream_t)stream);
}

int hk_rollout(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
               uint8_t* done_t, float* reward_t, int32_t* done_count, int32_t* length, int64_t B, int32_t N,
               int32_t d, int32_t T, int32_t dtype, uint32_t ops, uint32_t flags, float padding_value,
               void* stream) {
    if (T < 1) return HK_ERR_BAD_ARG;
    StepParams p = rollout_params(state_in, state_out, host_action_t, axis_t, nullptr, 0, nullptr, nullptr, done_t, reward_t,
                                  done_count, length, B, N, d, T, ops, flags, padding_value, 0, 0);
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_rollout_seeded(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
                      uint8_t* done_t, float* reward_t, int32_t* done_count, int32_t* length, int64_t B, int32_t N,
                      int32_t d, int32_t T, int32_t dtype, uint32_t ops, uint32_t flags, float padding_value,
                      uint64_t seed, int32_t step_offset, void* stream) {
    if (T < 1 || !(flags & (HK_F_HOST_RANDOM | HK_F_AGENT_RANDOM))) return HK_ERR_BAD_ARG;
    StepParams p = rollout_params(state_in, state_out, host_action_t, axis_t, nullptr, 0, nullptr, nullptr, done_t, reward_t,
                                  done_count, length, B, N, d, T, ops, flags, padding_value, seed, step_offset);
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_rollout_record(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
                      float* obs_t, int32_t agent_obs, int32_t* host_mask_t, int32_t* axis_played_t, uint8_t* done_t,
                      float* reward_t, int32_t* done_count, int32_t* length, int64_t B, int32_t N, int32_t d, int32_t T,
                      int32_t dtype, uint32_t ops, uint32_t flags, float padding_value, uint64_t seed, int32_t step_offset,
                      void* stream) {
    if (T < 1 || (agent_obs && !obs_t)) return HK_ERR_BAD_ARG;
    StepParams p = rollout_params(state_in, state_out, host_action_t, axis_t, obs_t, agent_obs, host_mask_t, axis_played_t,
                                  done_t, reward_t, done_count, length, B, N, d, T, ops, flags, padding_value, seed,
                                  step_offset);
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_rollout_threshold(const void* state_in, void* state_out, const int32_t* host_action_t, const int32_t* axis_t,
                         float* obs_t, int32_t agent_obs, int32_t* host_mask_t, int32_t* axis_played_t, uint8_t* done_t,
                         float* reward_t, int32_t* done_count, int32_t* length, int64_t B, int32_t N, int32_t d, int32_t T,
                         int32_t dtype, uint32_t ops, uint32_t flags, float padding_value, uint64_t seed, int32_t step_offset,
                         float value_threshold, int32_t stop_at_threshold, int32_t* over_step, void* stream) {
    if (T < 1 || (agent_obs && !obs_t) || value_threshold != value_threshold) return HK_ERR_BAD_ARG;
    const bool never = value_threshold == INFINITY;
    // int32 state: inputs below the threshold give shift sums below 2^30, the range in which the kernels are exact
    if (dtype == HK_DTYPE_I32 && !never && d >= 1 && (double)value_threshold > (double)((1 << 30) / d)) return HK_ERR_BAD_ARG;
    StepParams p = rollout_params(state_in, state_out, host_action_t, axis_t, obs_t, agent_obs, host_mask_t, axis_played_t,
                                  done_t, reward_t, done_count, length, B, N, d, T, ops, flags, padding_value, seed,
                                  step_offset);
    // without over_step and without a stop (+inf stops nothing) the call is the recorded rollout as it is
    p.threshold = value_threshold;
    p.over_step = over_step;
    p.stop_at_threshold = (stop_at_threshold && !never) ? 1 : 0;
    return run(p, dtype, g_force_generic.load(), (cudaStream_t)stream);
}

int hk_random_actions(int32_t* host_action_t, int32_t* axis_t, int64_t B, int32_t d, int32_t T, uint64_t seed,
                      int32_t step_offset, void* stream) {
    if (B < 0 || T < 1 || d < 1 || d > HK_MAX_DIM || (!host_action_t && !axis_t)) return HK_ERR_BAD_ARG;
    if (B == 0) return HK_OK;
    const long long total = (long long)B * T;
    const unsigned blocks = (unsigned)((total + 255) / 256 > 148 * 32 ? 148 * 32 : (total + 255) / 256);
    hk::hk_random_actions_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(host_action_t, axis_t, B, d, T, seed, step_offset);
    return (int)cudaGetLastError();
}

int64_t hk_experience_scratch_words(int64_t B) {
    if (B < 0) return 0;
    return (B + hk::EXP_ROWS_PER_BLOCK - 1) / hk::EXP_ROWS_PER_BLOCK + 4;
}

int hk_experience_append(const uint8_t* skip, const float* obs, const float* next_obs, int32_t obs_width,
                         const float* coords, const float* next_coords, int32_t coord_width, const int32_t* action,
                         const float* reward, const uint8_t* done, float* buf_obs, float* buf_next_obs,
                         float* buf_coords, float* buf_next_coords, int32_t* buf_action, float* buf_reward,
                         uint8_t* buf_done, int64_t capacity, int64_t* pos, int32_t* full, int32_t* appended,
                         int32_t* scratch, int64_t B, void* stream) {
    if (B < 0 || capacity < 1 || !skip || !pos || !full || !scratch) return HK_ERR_BAD_ARG;
    if ((buf_obs && (!obs || obs_width < 1)) || (buf_next_obs && (!next_obs || obs_width < 1))) return HK_ERR_BAD_ARG;
    if ((buf_coords && (!coords || coord_width < 1)) || (buf_next_coords && (!next_coords || coord_width < 1)))
        return HK_ERR_BAD_ARG;
    if ((buf_action && !action) || (buf_reward && !reward) || (buf_done && !done)) return HK_ERR_BAD_ARG;
    if (B == 0) return HK_OK;
    hk::ExpParams p;
    memset(&p, 0, sizeof(p));
    p.skip = skip;
    p.obs = obs;
    p.next_obs = next_obs;
    p.coords = coords;
    p.next_coords = next_coords;
    p.action = action;
    p.reward = reward;
    p.done = done;
    p.buf_obs = buf_obs;
    p.buf_next_obs = buf_next_obs;
    p.buf_coords = buf_coords;
    p.buf_next_coords = buf_next_coords;
    p.buf_action = buf_action;
    p.buf_reward = buf_reward;
    p.buf_done = buf_done;
    p.capacity = capacity;
    p.pos = (long long*)pos;
    p.full = full;
    p.appended = appended;
    p.scratch = scratch;
    p.B = B;
    p.ow = obs_width;
    p.cw = coord_width;
    p.nblocks = (int)((B + hk::EXP_ROWS_PER_BLOCK - 1) / hk::EXP_ROWS_PER_BLOCK);
    cudaStream_t st = (cudaStream_t)stream;
    hk::hk_exp_count_kernel<<<p.nblocks, hk::EXP_THREADS, 0, st>>>(p);
    hk::hk_exp_scan_kernel<<<1, 1024, 0, st>>>(p);
    hk::hk_exp_scatter_kernel<<<p.nblocks, hk::EXP_THREADS, 0, st>>>(p);
    return (int)cudaGetLastError();
}

int hk_value_targets(const float* obs, const int32_t* num_points, int32_t* num_points_out, float* value, int64_t B,
                     int32_t T, int32_t W, int32_t dimension, int32_t offset, float discount, int32_t est_sign,
                     int32_t reward_sign, int32_t unified, void* stream) {
    if (B < 0 || T < 1 || T > hk::VALUE_MAX_T || !value || (!obs && !num_points)) return HK_ERR_BAD_ARG;
    if (obs && !num_points && (W < 1 || dimension < 1)) return HK_ERR_BAD_ARG;
    if (B == 0) return HK_OK;
    hk::ValueParams p;
    memset(&p, 0, sizeof(p));
    p.obs = obs;
    p.num_points = num_points;
    p.num_points_out = num_points_out;
    p.value = value;
    p.B = B;
    p.T = T;
    p.W = W;
    p.dimension = dimension;
    p.offset = offset;
    p.discount = discount;
    p.est_sign = est_sign;
    p.reward_sign = reward_sign;
    p.unified = unified;
    const int warps = 8;
    const size_t smem = (size_t)warps * T * sizeof(int32_t);
    long long ctas = (B + warps - 1) / warps;
    if (ctas > 148 * 8) ctas = 148 * 8;
    hk::hk_value_targets_kernel<<<(unsigned)ctas, warps * 32, smem, (cudaStream_t)stream>>>(p);
    return (int)cudaGetLastError();
}

int hk_overflow(const void* state, uint8_t* overflow, int64_t B, int32_t N, int32_t d, int32_t dtype, float value_threshold,
                int32_t strict, void* stream) {
    int rc = check_shape(B, N, d, dtype);
    if (rc != HK_OK) return rc;
    if (B == 0) return HK_OK;
    if (!state || !overflow) return HK_ERR_BAD_ARG;
    const int warps = 8;
    long long ctas = (B + warps - 1) / warps;
    if (ctas > 148 * 16) ctas = 148 * 16;
    if (dtype == HK_DTYPE_I32)
        hk::hk_overflow_kernel<int32_t><<<(unsigned)ctas, warps * 32, 0, (cudaStream_t)stream>>>(
            (const int32_t*)state, overflow, B, N * d, value_threshold, strict);
    else
        hk::hk_overflow_kernel<float><<<(unsigned)ctas, warps * 32, 0, (cudaStream_t)stream>>>(
            (const float*)state, overflow, B, N * d, value_threshold, strict);
    return (int)cudaGetLastError();
}

int hk_pack_coords(const void* coords, int32_t src_dtype, int32_t* mask, int64_t B, int32_t d, void* stream) {
    if (B < 0 || d < 1 || d > 31 || !mask || (!coords && B > 0)) return HK_ERR_BAD_ARG;
    if (B == 0) return HK_OK;
    const unsigned blocks = (unsigned)((B + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    switch (src_dtype) {
        case 0: hk::hk_pack_coords_kernel<int32_t><<<blocks, 256, 0, st>>>((const int32_t*)coords, mask, B, d); break;
        case 1: hk::hk_pack_coords_kernel<float><<<blocks, 256, 0, st>>>((const float*)coords, mask, B, d); break;
        case 2: hk::hk_pack_coords_kernel<long long><<<blocks, 256, 0, st>>>((const long long*)coords, mask, B, d); break;
        case 3: hk::hk_pack_coords_kernel<uint8_t><<<blocks, 256, 0, st>>>((const uint8_t*)coords, mask, B, d); break;
        default: return HK_ERR_BAD_ARG;
    }
    return (int)cudaGetLastError();
}

// ---- host-buffer sessions ----------------------------------------------------------------------
struct hk_session {
    int device;
    long long B;
    int N, d, dtype;
    float pad;
    cudaStream_t stream;
    cudaStream_t copy_stream;  // host -> device (actions)
    cudaStream_t back_stream;  // device -> host (per-step results), so that the two directions overlap
    cudaEvent_t ready[2], freed[2], drained[2];
    void* state;
    int32_t* host_action;  // two slots of B int32 each (double buffer for hk_session_rollout)
    int32_t* axis;
    int32_t* counts;       // per-step finished-game counts of a rollout (device)
    int32_t* counts_pinned; // pinned host mirror: a D2H copy into pageable memory would block the host every step
    int counts_cap;
    uint8_t* done;         // two slots of B bytes (double buffer for the per-step read-back of hk_session_rollout_ex)
    uint32_t* done_bits;   // two slots of ceil(B/32) words (hk_session_rollout_bits)
    float* reward;
    int32_t* done_count;
    uint8_t* census;       // [B] census of the resident state (hk_step_census); zeroed whenever the state is set
    // hk_session_rollout_ex replayed as a CUDA graph: the second call with the same arguments captures the
    // three-stream schedule once, later calls launch it (a rollout is ~10 API calls per step otherwise, and the
    // steps of a census rollout are shorter than that)
    cudaEvent_t fork, join_copy, join_back;
    cudaGraphExec_t rollout_exec;
    struct RolloutKey {
        const void* ha;
        const void* ax;
        int32_t* dc;
        uint8_t* done;
        uint32_t* bits;
        int32_t T;
        uint32_t ops, flags;
        int force_generic;
    } last_key, exec_key;
};

// page-locked host memory?  (copies from pageable memory are staged by the driver and cannot be captured)
static bool is_pinned(const void* ptr) {
    if (!ptr) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, ptr) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeHost;
}

static bool same_key(const hk_session::RolloutKey& a, const hk_session::RolloutKey& b) {
    return a.ha == b.ha && a.ax == b.ax && a.dc == b.dc && a.done == b.done && a.bits == b.bits && a.T == b.T && a.ops == b.ops &&
           a.flags == b.flags && a.force_generic == b.force_generic;
}

// bytes of one step's action array of B games under the action-format flags
static size_t action_bytes(long long B, uint32_t flags) {
    if (flags & HK_F_ACT_NIBBLE) return (size_t)((B + 1) / 2);
    return (size_t)B * ((flags & (HK_F_ACT_U8 | HK_F_ACT_PACKED)) ? 1 : 4);
}

// the census step serves in-place single steps without fused observation or in-kernel players
static bool census_eligible(uint32_t ops, uint32_t flags) {
    return ops != 0 && !(flags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER | HK_F_AGENT_FIRST | HK_F_AGENT_LAST));
}

// sessions switch to their device for the duration of a call and restore the caller's device
struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

#define HK_CUDA(x)                       \
    do {                                 \
        cudaError_t e_ = (x);            \
        if (e_ != cudaSuccess) return (int)e_; \
    } while (0)

int hk_session_create(hk_session** out, int device, int64_t B, int32_t N, int32_t d, int32_t dtype,
                      float padding_value) {
    if (out == nullptr || B < 1) return HK_ERR_BAD_ARG;
    int rc = check_shape(B, N, d, dtype);
    if (rc != HK_OK) return rc;
    DeviceGuard guard_(device);
    hk_session* s = new (std::nothrow) hk_session();
    if (!s) return HK_ERR_BAD_ARG;
    memset(s, 0, sizeof(*s));
    s->device = device;
    s->B = B;
    s->N = N;
    s->d = d;
    s->dtype = dtype;
    s->pad = padding_value;
    cudaError_t e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->back_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && e == cudaSuccess; ++i) {
        e = cudaEventCreateWithFlags(&s->ready[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->freed[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->drained[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->join_copy, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->join_back, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(&s->state, (size_t)B * N * d * 4);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->host_action, (size_t)B * 4 * 2);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->axis, (size_t)B * 4 * 2);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->done, (size_t)B * 2);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->done_bits, (size_t)((B + 31) / 32) * 4 * 2);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->census, (size_t)hk_census_bytes(B, N, d));
    if (e == cudaSuccess) e = cudaMemsetAsync(s->census, 0, (size_t)B, s->stream);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->reward, (size_t)B * 4);
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->done_count, 4);
    // per-step count buffers of hk_session_rollout are sized here (allocating later would put a
    // device-synchronising cudaMallocHost on the step path); they grow only for T > 1024
    if (e == cudaSuccess) e = cudaMalloc((void**)&s->counts, 1024 * 4);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&s->counts_pinned, 1024 * 4);
    if (e == cudaSuccess) s->counts_cap = 1024;
    if (e != cudaSuccess) {
        hk_session_destroy(s);
        return (int)e;
    }
    *out = s;
    return HK_OK;
}

int hk_session_destroy(hk_session* s) {
    if (!s) return HK_OK;
    DeviceGuard guard_(s->device);
    if (s->stream) cudaStreamSynchronize(s->stream);
    cudaFree(s->state);
    cudaFree(s->host_action);
    cudaFree(s->axis);
    cudaFree(s->done);
    cudaFree(s->done_bits);
    cudaFree(s->census);
    cudaFree(s->reward);
    cudaFree(s->done_count);
    cudaFree(s->counts);
    if (s->counts_pinned) cudaFreeHost(s->counts_pinned);
    for (int i = 0; i < 2; ++i) {
        if (s->ready[i]) cudaEventDestroy(s->ready[i]);
        if (s->freed[i]) cudaEventDestroy(s->freed[i]);
        if (s->drained[i]) cudaEventDestroy(s->drained[i]);
    }
    if (s->rollout_exec) cudaGraphExecDestroy(s->rollout_exec);
    if (s->fork) cudaEventDestroy(s->fork);
    if (s->join_copy) cudaEventDestroy(s->join_copy);
    if (s->join_back) cudaEventDestroy(s->join_back);
    if (s->copy_stream) cudaStreamDestroy(s->copy_stream);
    if (s->back_stream) cudaStreamDestroy(s->back_stream);
    if (s->stream) cudaStreamDestroy(s->stream);
    delete s;
    return HK_OK;
}

int hk_session_set_state(hk_session* s, const void* state_host) {
    if (!s || !state_host) return HK_ERR_BAD_ARG;
    DeviceGuard guard_(s->device);
    HK_CUDA(cudaMemcpyAsync(s->state, state_host, (size_t)s->B * s->N * s->d * 4, cudaMemcpyHostToDevice, s->stream));
    HK_CUDA(cudaMemsetAsync(s->census, 0, (size_t)s->B, s->stream));  // every game unknown again
    HK_CUDA(cudaStreamSynchronize(s->stream));
    return HK_OK;
}

int hk_session_get_state(hk_session* s, void* state_host) {
    if (!s || !state_host) return HK_ERR_BAD_ARG;
    DeviceGuard guard_(s->device);
    HK_CUDA(cudaMemcpyAsync(state_host, s->state, (size_t)s->B * s->N * s->d * 4, cudaMemcpyDeviceToHost, s->stream));
    HK_CUDA(cudaStreamSynchronize(s->stream));
    return HK_OK;
}

int hk_session_step(hk_session* s, const int32_t* host_action_host, const int32_t* axis_host, uint8_t* done_host,
                    float* reward_host, int32_t* done_count_host, uint32_t ops, uint32_t flags) {
    if (!s) return HK_ERR_BAD_ARG;
    DeviceGuard guard_(s->device);
    const bool packed = flags & (HK_F_ACT_PACKED | HK_F_ACT_NIBBLE);
    const size_t abytes = action_bytes(s->B, flags);
    if ((ops & HK_OP_SHIFT) && host_action_host)
        HK_CUDA(cudaMemcpyAsync(s->host_action, host_action_host, abytes, cudaMemcpyHostToDevice, s->stream));
    if ((ops & HK_OP_SHIFT) && axis_host && !packed)
        HK_CUDA(cudaMemcpyAsync(s->axis, axis_host, abytes, cudaMemcpyHostToDevice, s->stream));
    StepParams p = make_params(s->state, s->state, s->B, s->N, s->d, s->pad);
    p.host_action = host_action_host ? s->host_action : nullptr;
    p.axis = (axis_host && !packed) ? s->axis : nullptr;
    p.done = done_host ? s->done : nullptr;
    p.reward = reward_host ? s->reward : nullptr;
    p.ops = ops;
    p.flags = flags;
    if (done_count_host) {
        HK_CUDA(cudaMemsetAsync(s->done_count, 0, 4, s->stream));
        p.done_count = s->done_count;
    }
    if (census_eligible(ops, flags)) p.census = s->census;
    int rc = run(p, s->dtype, g_force_generic.load(), s->stream);
    if (rc != HK_OK) return rc;
    if (!p.census && ops != 0) HK_CUDA(cudaMemsetAsync(s->census, 0, (size_t)s->B, s->stream));  // stepped without it: stale
    if (done_host) HK_CUDA(cudaMemcpyAsync(done_host, s->done, (size_t)s->B, cudaMemcpyDeviceToHost, s->stream));
    if (reward_host) HK_CUDA(cudaMemcpyAsync(reward_host, s->reward, (size_t)s->B * 4, cudaMemcpyDeviceToHost, s->stream));
    if (done_count_host) HK_CUDA(cudaMemcpyAsync(done_count_host, s->done_count, 4, cudaMemcpyDeviceToHost, s->stream));
    HK_CUDA(cudaStreamSynchronize(s->stream));
    return HK_OK;
}

// the three-stream schedule of one rollout, enqueued (or captured: every call below is capturable)
static int enqueue_rollout(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                           int32_t* done_count_host, uint8_t* done_host, uint32_t* bits_host, uint32_t ops, uint32_t flags,
                           int force_generic) {
    const bool packed = flags & (HK_F_ACT_PACKED | HK_F_ACT_NIBBLE);
    const size_t abytes = action_bytes(s->B, flags);
    const size_t bwords = (size_t)((s->B + 31) / 32);
    const bool use_census = census_eligible(ops, flags);
    HK_CUDA(cudaMemsetAsync(s->counts, 0, (size_t)T * 4, s->stream));
    // uploads and read-backs branch off the step stream here and join it again at the end
    HK_CUDA(cudaEventRecord(s->fork, s->stream));
    HK_CUDA(cudaStreamWaitEvent(s->copy_stream, s->fork, 0));
    HK_CUDA(cudaStreamWaitEvent(s->back_stream, s->fork, 0));
    // Three streams: uploads (copy_stream), steps (stream), read-backs (back_stream).  Step t uses slot t & 1 of
    // the action and done buffers; the upload of step t waits until step t - 2 has run (freed), the read-back of
    // step t waits for step t, and step t + 2 waits until that read-back has drained the slot (drained).
    auto read_back = [&](int t) -> int {
        const int slot = t & 1;
        HK_CUDA(cudaStreamWaitEvent(s->back_stream, s->freed[slot], 0));
        if (done_count_host)
            HK_CUDA(cudaMemcpyAsync(s->counts_pinned + t, s->counts + t, 4, cudaMemcpyDeviceToHost, s->back_stream));
        if (done_host)
            HK_CUDA(cudaMemcpyAsync(done_host + (size_t)t * s->B, s->done + (size_t)slot * s->B, (size_t)s->B,
                                    cudaMemcpyDeviceToHost, s->back_stream));
        if (bits_host)
            HK_CUDA(cudaMemcpyAsync(bits_host + (size_t)t * bwords, s->done_bits + (size_t)slot * bwords, bwords * 4,
                                    cudaMemcpyDeviceToHost, s->back_stream));
        HK_CUDA(cudaEventRecord(s->drained[slot], s->back_stream));
        return HK_OK;
    };
    for (int t = 0; t < T; ++t) {
        const int slot = t & 1;
        int32_t* ha = s->host_action + (size_t)slot * s->B;
        int32_t* ax = s->axis + (size_t)slot * s->B;
        if (t >= 2) {
            HK_CUDA(cudaStreamWaitEvent(s->copy_stream, s->freed[slot], 0));
            int rb = read_back(t - 2);
            if (rb != HK_OK) return rb;
        }
        HK_CUDA(cudaMemcpyAsync(ha, (const char*)host_action_host + (size_t)t * abytes, abytes, cudaMemcpyHostToDevice,
                                s->copy_stream));
        if (!packed)
            HK_CUDA(cudaMemcpyAsync(ax, (const char*)axis_host + (size_t)t * abytes, abytes, cudaMemcpyHostToDevice,
                                    s->copy_stream));
        HK_CUDA(cudaEventRecord(s->ready[slot], s->copy_stream));
        HK_CUDA(cudaStreamWaitEvent(s->stream, s->ready[slot], 0));
        if (t >= 2 && (done_host || bits_host)) HK_CUDA(cudaStreamWaitEvent(s->stream, s->drained[slot], 0));
        StepParams p = make_params(s->state, s->state, s->B, s->N, s->d, s->pad);
        p.host_action = ha;
        p.axis = packed ? nullptr : ax;
        p.done_count = s->counts + t;
        p.done = done_host ? s->done + (size_t)slot * s->B : nullptr;
        p.done_bits = bits_host ? s->done_bits + (size_t)slot * bwords : nullptr;
        p.census = use_census ? s->census : nullptr;
        p.ops = ops;
        p.flags = flags;
        int rc = run(p, s->dtype, force_generic, s->stream);
        if (rc != HK_OK) return rc;
        HK_CUDA(cudaEventRecord(s->freed[slot], s->stream));
    }
    if (!use_census) HK_CUDA(cudaMemsetAsync(s->census, 0, (size_t)s->B, s->stream));
    for (int t = (T >= 2 ? T - 2 : 0); t < T; ++t) {  // the results of the last two steps
        int rb = read_back(t);
        if (rb != HK_OK) return rb;
    }
    HK_CUDA(cudaEventRecord(s->join_copy, s->copy_stream));
    HK_CUDA(cudaEventRecord(s->join_back, s->back_stream));
    HK_CUDA(cudaStreamWaitEvent(s->stream, s->join_copy, 0));
    HK_CUDA(cudaStreamWaitEvent(s->stream, s->join_back, 0));
    return HK_OK;
}

static int session_rollout(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                           int32_t* done_count_host, uint8_t* done_host, uint32_t* bits_host, uint32_t ops, uint32_t flags) {
    const bool packed = flags & (HK_F_ACT_PACKED | HK_F_ACT_NIBBLE);
    if (!s || T < 1 || !(ops & HK_OP_SHIFT) || !host_action_host || (!axis_host && !packed)) return HK_ERR_BAD_ARG;
    if (bits_host && !census_eligible(ops, flags)) return HK_ERR_UNSUPPORTED;
    DeviceGuard guard_(s->device);
    if (s->counts_cap < T) {
        if (s->rollout_exec) {  // the graph holds the old buffers
            cudaGraphExecDestroy(s->rollout_exec);
            s->rollout_exec = nullptr;
        }
        cudaFree(s->counts);
        if (s->counts_pinned) cudaFreeHost(s->counts_pinned);
        s->counts = nullptr;
        s->counts_pinned = nullptr;
        s->counts_cap = 0;
        HK_CUDA(cudaMalloc((void**)&s->counts, (size_t)T * 4));
        HK_CUDA(cudaMallocHost((void**)&s->counts_pinned, (size_t)T * 4));
        s->counts_cap = T;
    }
    const int fg = g_force_generic.load();
    const hk_session::RolloutKey key = {host_action_host, axis_host, done_count_host, done_host, bits_host, T, ops, flags, fg};
    int rc = HK_OK;
    if (s->rollout_exec && same_key(key, s->exec_key)) {
        HK_CUDA(cudaGraphLaunch(s->rollout_exec, s->stream));
    } else if (same_key(key, s->last_key) && !g_no_session_graphs.load() && is_pinned(host_action_host) &&
               is_pinned(axis_host) && is_pinned(done_host) && is_pinned(bits_host)) {
        // second call with these arguments (the first ran eagerly, so every kernel is set up): capture and keep
        if (s->rollout_exec) {
            cudaGraphExecDestroy(s->rollout_exec);
            s->rollout_exec = nullptr;
        }
        cudaGraph_t graph = nullptr;
        HK_CUDA(cudaStreamBeginCapture(s->stream, cudaStreamCaptureModeThreadLocal));
        rc = enqueue_rollout(s, host_action_host, axis_host, T, done_count_host, done_host, bits_host, ops, flags, fg);
        cudaError_t e = cudaStreamEndCapture(s->stream, &graph);
        if (rc == HK_OK && e != cudaSuccess) rc = (int)e;
        if (rc == HK_OK) {
            e = cudaGraphInstantiate(&s->rollout_exec, graph, 0);
            if (e != cudaSuccess) {
                s->rollout_exec = nullptr;
                rc = (int)e;
            }
        }
        if (graph) cudaGraphDestroy(graph);
        if (rc != HK_OK) {
            cudaGetLastError();
            return rc;
        }
        s->exec_key = key;
        HK_CUDA(cudaGraphLaunch(s->rollout_exec, s->stream));
    } else {
        rc = enqueue_rollout(s, host_action_host, axis_host, T, done_count_host, done_host, bits_host, ops, flags, fg);
        if (rc != HK_OK) return rc;
    }
    s->last_key = key;
    HK_CUDA(cudaStreamSynchronize(s->stream));  // (the other two streams were joined into this one)
    if (done_count_host) memcpy(done_count_host, s->counts_pinned, (size_t)T * 4);
    return HK_OK;
}

int hk_session_rollout_ex(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                          int32_t* done_count_host, uint8_t* done_host, uint32_t ops, uint32_t flags) {
    return session_rollout(s, host_action_host, axis_host, T, done_count_host, done_host, nullptr, ops, flags);
}

int hk_session_rollout_bits(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                            int32_t* done_count_host, uint32_t* done_bits_host, uint32_t ops, uint32_t flags) {
    return session_rollout(s, host_action_host, axis_host, T, done_count_host, nullptr, done_bits_host, ops, flags);
}

int hk_session_rollout(hk_session* s, const void* host_action_host, const void* axis_host, int32_t T,
                       int32_t* done_count_host, uint32_t ops, uint32_t flags) {
    return session_rollout(s, host_action_host, axis_host, T, done_count_host, nullptr, nullptr, ops, flags);
}

void* hk_session_state_ptr(hk_session* s) { return s ? s->state : nullptr; }
void* hk_session_stream(hk_session* s) { return s ? (void*)s->stream : nullptr; }

}  // extern "C"
