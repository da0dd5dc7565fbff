// hk_small.cuh — thread-per-game step kernel for small games (N <= 32, N*d words in registers).
//
// Mapping (DESIGN.md "K-small"): one lane owns one game; a warp owns tiles of 32 consecutive
// games.  Each warp has a private shared-memory stage of one tile:
// lane 0 issues one TMA bulk load per tile (32*N*d*4 contiguous bytes), all lanes wait on the warp's
// mbarrier and read their own game with conflict-free vector LDS (game stride N*d words: 16-byte
// reads are conflict-free when N*d/4 is odd, 8-byte when N*d/2 is odd, 4-byte when N*d is odd —
// true for (20,3), (10,3), (5,3)).  The warp picks a tier from the largest live count among its 32
// games, every lane gathers its live rows into that many register rows and runs the step there
// (small tiers fully unrolled, 12 and 16 rows with a rolled victim loop).  Only games that changed
// are written back when the call is in place: one TMA bulk store of the tile when many did, one
// coalesced copy per game when few did, nothing when none did.  The fused observation features
// (OBS) are a second phase on the new state: a sorting network on packed row keys.  No CTA-wide
// barrier exists anywhere; warps drift freely, which overlaps one warp's loads with another's ALU phase.
// Single steps of int32 state with small values run on PACKED tiers instead (tier_packed below: one 32-bit word per
// row, one sort after which only earlier rows can dominate, dominance as one subtraction), and in-place callers that
// own the stage (the census kernel) may take their DIRECT route: stage handed back after the gather, changed rows
// stored straight to global memory.
#pragma once
#include <type_traits>

#include "hk_common.cuh"

namespace hk {

constexpr int SMALL_BAR_BYTES = 256;
#ifndef HK_SPARSE_STORE_MAX
#define HK_SPARSE_STORE_MAX 16  // at most this many changed games of a tile are written one by one (tools/tune_small.cu: 4 -> 71.2, 8 -> 68.3, 16 -> 67.3, 32 -> 75.7 us/step at C2)
#endif

// WARPS warps per CTA, each with a private stage of one tile (and the obs tile with OBS).
template <int N, int D, bool OBS, int WARPS>
struct SmallLayout {
    static_assert(WARPS * 8 <= SMALL_BAR_BYTES, "mbarrier area too small");
    static constexpr int W = N * D;
    static constexpr int TILE_WORDS = 32 * W;
    static constexpr int OBS_W = W + D;
    static constexpr int OBS_WORDS = OBS ? 32 * OBS_W : 0;
    static constexpr int WARP_WORDS = TILE_WORDS + OBS_WORDS;
    static constexpr size_t SMEM_BYTES = SMALL_BAR_BYTES + (size_t)WARPS * WARP_WORDS * 4;
};

// ---- game <-> shared memory -------------------------------------------------------------------
template <typename T, int W>
__device__ __forceinline__ void load_game(const uint32_t* s, T (&x)[W]) {
    if constexpr (W % 4 == 0) {
        const uint4* p = reinterpret_cast<const uint4*>(s);
#pragma unroll
        for (int q = 0; q < W / 4; ++q) {
            uint4 v = p[q];
            x[4 * q + 0] = Elem<T>::from_bits(v.x);
            x[4 * q + 1] = Elem<T>::from_bits(v.y);
            x[4 * q + 2] = Elem<T>::from_bits(v.z);
            x[4 * q + 3] = Elem<T>::from_bits(v.w);
        }
    } else if constexpr (W % 2 == 0) {
        const uint2* p = reinterpret_cast<const uint2*>(s);
#pragma unroll
        for (int q = 0; q < W / 2; ++q) {
            uint2 v = p[q];
            x[2 * q + 0] = Elem<T>::from_bits(v.x);
            x[2 * q + 1] = Elem<T>::from_bits(v.y);
        }
    } else {
#pragma unroll
        for (int q = 0; q < W; ++q) x[q] = Elem<T>::from_bits(s[q]);
    }
}

template <typename T, int W>
__device__ __forceinline__ void store_game(uint32_t* s, const T (&x)[W]) {
    if constexpr (W % 4 == 0) {
        uint4* p = reinterpret_cast<uint4*>(s);
#pragma unroll
        for (int q = 0; q < W / 4; ++q)
            p[q] = make_uint4((uint32_t)Elem<T>::bits(x[4 * q]), (uint32_t)Elem<T>::bits(x[4 * q + 1]),
                              (uint32_t)Elem<T>::bits(x[4 * q + 2]), (uint32_t)Elem<T>::bits(x[4 * q + 3]));
    } else if constexpr (W % 2 == 0) {
        uint2* p = reinterpret_cast<uint2*>(s);
#pragma unroll
        for (int q = 0; q < W / 2; ++q)
            p[q] = make_uint2((uint32_t)Elem<T>::bits(x[2 * q]), (uint32_t)Elem<T>::bits(x[2 * q + 1]));
    } else {
#pragma unroll
        for (int q = 0; q < W; ++q) s[q] = (uint32_t)Elem<T>::bits(x[q]);
    }
}

// ---- the per-game ops, state in registers --------------------------------------------------------
template <typename T, int N, int D>
__device__ __forceinline__ uint32_t live_mask(const T (&x)[N * D]) {
    uint32_t lm = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) lm |= (x[i * D] >= Elem<T>::zero()) ? (1u << i) : 0u;
    return lm;
}

// shift: x_a <- sum_{j in S} x_j on live rows (shift_torch _torch_ops.py:46-110, shift_jax _jax_ops.py:76-90)
template <typename T, int N, int D>
__device__ __forceinline__ void op_shift(T (&x)[N * D], uint32_t lm, uint32_t cm, int a, bool apply) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
        T s = Elem<T>::zero();
#pragma unroll
        for (int k = 0; k < D; ++k) {
            if constexpr (Elem<T>::is_float) {
                s = ((cm >> k) & 1u) ? s + x[i * D + k] : s;
            } else {
                s = (T)((uint32_t)s + (((cm >> k) & 1u) ? (uint32_t)x[i * D + k] : 0u));
            }
        }
        const bool upd = apply && ((lm >> i) & 1u);
#pragma unroll
        for (int k = 0; k < D; ++k) x[i * D + k] = (upd && k == a) ? s : x[i * D + k];
    }
}

// reposition: per coordinate subtract the min over live rows (reposition_torch _torch_ops.py:113-133)
template <typename T, int N, int D>
__device__ __forceinline__ void op_reposition(T (&x)[N * D], uint32_t lm) {
#pragma unroll
    for (int k = 0; k < D; ++k) {
        T mn = Elem<T>::big();
#pragma unroll
        for (int i = 0; i < N; ++i) {
            T v = ((lm >> i) & 1u) ? x[i * D + k] : Elem<T>::big();
            mn = v < mn ? v : mn;
        }
#pragma unroll
        for (int i = 0; i < N; ++i) x[i * D + k] = ((lm >> i) & 1u) ? x[i * D + k] - mn : x[i * D + k];
    }
}

// Newton polytope (approx): fused dedupe + dominance (remove_repeated _fn.py:192-213 followed by
// get_newton_polytope_approx_torch _torch_ops.py:8-39).  Row i dies iff some row j != i has
// x_j <= x_i componentwise and (x_j != x_i or j < i).  With t = OR_k bits(x_i[k] - x_j[k]):
//   sign(t) = 0  <=> x_j <= x_i;  t == 0 <=> equal.  For j > i the tie must not kill, which is
//   sign(t - 1) = 0 <=> t > 0.  The AND over j of these words has sign 0 iff some j kills i.
// Dead rows are parked at +BIG so they dominate nothing and no liveness test is needed per pair.
template <typename T, int N, int D>
__device__ __forceinline__ uint32_t op_newton(T (&x)[N * D], uint32_t lm) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int k = 0; k < D; ++k) x[i * D + k] = ((lm >> i) & 1u) ? x[i * D + k] : Elem<T>::big();
    }
    uint32_t kill = 0;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        int32_t acc = (int32_t)0x80000000;
#pragma unroll
        for (int j = 0; j < N; ++j) {
            if (j == i) continue;
            int32_t t = Elem<T>::bits(x[i * D] - x[j * D]);
#pragma unroll
            for (int k = 1; k < D; ++k) t |= Elem<T>::bits(x[i * D + k] - x[j * D + k]);
            if (j > i) t -= 1;
            acc &= t;
        }
        kill |= (acc >= 0) ? (1u << i) : 0u;
    }
    return lm & ~kill;
}

// The same filter with the victim loop ROLLED (code size K times smaller: the fully unrolled
// N = 20 body is 33 KB of SASS, more than the 32 KB instruction cache, and warps of one SM run
// different tiers at the same time).  Victim i is re-read from the lane's shared-memory scratch
// (a register array cannot be indexed dynamically); dominators j stay in registers with static
// indices.  The tie-break needs j >= i at run time: t - (j >= i) also neutralises the self pair
// (t_ii = 0 -> -1).  RS = scratch row stride in words (4 => one conflict-free LDS.128 per victim).
template <typename T, int K, int D, int RS>
__device__ __forceinline__ uint32_t op_newton_rolled(T (&y)[K * D], uint32_t clm, uint32_t* scratch) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
#pragma unroll
        for (int c = 0; c < D; ++c) y[k * D + c] = ((clm >> k) & 1u) ? y[k * D + c] : Elem<T>::big();
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if constexpr (RS == 4 && D == 3) {
            *reinterpret_cast<uint4*>(scratch + k * 4) =
                make_uint4((uint32_t)Elem<T>::bits(y[k * 3]), (uint32_t)Elem<T>::bits(y[k * 3 + 1]),
                           (uint32_t)Elem<T>::bits(y[k * 3 + 2]), 0u);
        } else {
#pragma unroll
            for (int c = 0; c < D; ++c) scratch[k * RS + c] = (uint32_t)Elem<T>::bits(y[k * D + c]);
        }
    }
    uint32_t kill = 0;
    // compact rows fill from 0: rows past the highest one that is live in SOME game of the warp are dead
    // in every lane and need no pass (the tier is chosen by the maximum, so this trims its rounding)
    const int kb = 32 - __clz((int)__reduce_or_sync(0xffffffffu, clm));
#pragma unroll 1
    for (int i = 0; i < kb; ++i) {
        T v[D];
        if constexpr (RS == 4 && D == 3) {
            const uint4 q = *reinterpret_cast<const uint4*>(scratch + i * 4);
            v[0] = Elem<T>::from_bits(q.x);
            v[1] = Elem<T>::from_bits(q.y);
            v[2] = Elem<T>::from_bits(q.z);
        } else {
#pragma unroll
            for (int c = 0; c < D; ++c) v[c] = Elem<T>::from_bits(scratch[i * RS + c]);
        }
        int32_t acc = (int32_t)0x80000000;
#pragma unroll
        for (int j = 0; j < K; ++j) {
            int32_t t = Elem<T>::bits(v[0] - y[j * D]);
#pragma unroll
            for (int c = 1; c < D; ++c) t |= Elem<T>::bits(v[c] - y[j * D + c]);
            t -= (j >= i) ? 1 : 0;
            acc &= t;
        }
        kill |= ((acc >= 0) ? 1u : 0u) << i;
    }
    return clm & ~kill;
}

// rescale (float state): live entries / game max, max == 0 -> 1 (rescale_torch _torch_ops.py:136-146);
// `eps`: a maximum <= 1e-8 leaves the game unchanged (calculate_rescale _jax_ops.py:93-98; x / 1 == x)
template <int N, int D>
__device__ __forceinline__ void op_rescale(float (&x)[N * D], uint32_t lm, bool eps) {
    float mx = -1.0f, mnpos = 3.0e38f;
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int k = 0; k < D; ++k) {
            const float v = x[i * D + k];
            const bool lv = (lm >> i) & 1u;
            mx = lv ? fmaxf(mx, v) : mx;
            mnpos = (lv && v > 0.0f) ? fminf(mnpos, v) : mnpos;
        }
    }
    if (mx == 0.0f || (eps && mx > 0.0f && mx <= 1e-8f)) mx = 1.0f;
    // Dead rows are parked at +BIG and zeros are common after reposition; neither goes through
    // the divider (0 / mx = 0 exactly, dead rows are rewritten with the padding value).
    // The choice of the division routine is warp-uniform; the vote is taken by ALL lanes, outside
    // the per-game condition (a game without live rows has nothing to divide).
    const bool act = mx > 0.0f;
    const GameDivider g = make_divider(act ? mx : 1.0f, mnpos);
    const bool fast = __all_sync(0xffffffffu, !act || g.safe);
    if (act) {
        if (fast) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const bool lv = (lm >> i) & 1u;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    const float v = x[i * D + k];
                    const bool use = lv && (v != 0.0f);
                    const float q = divide_by_game_max(use ? v : mx, g);
                    x[i * D + k] = use ? q : v;
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const bool lv = (lm >> i) & 1u;
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    const float v = x[i * D + k];
                    const bool use = lv && (v != 0.0f);
                    const float q = divide_ieee(use ? v : mx, mx);
                    x[i * D + k] = use ? q : v;
                }
            }
        }
    }
}

template <typename T, int N, int D>
__device__ __forceinline__ bool exceeds(const T (&x)[N * D], uint32_t lm, float threshold) {
    bool e = false;
#pragma unroll
    for (int i = 0; i < N; ++i) {
#pragma unroll
        for (int k = 0; k < D; ++k) e |= ((lm >> i) & 1u) && (Elem<T>::to_float(x[i * D + k]) >= threshold);
    }
    return e;
}

// One full step of one game in registers.  Returns the new live mask; x holds garbage in dead rows.
// Zeillinger's host, thread-per-game: the K compact rows are written (as floats) to the lane's
// shared-memory scratch at stride ZS and an (i, j) double loop walks them in flat order.  The walk
// is a separate NON-inlined function on shared memory only, so that this rarely used policy adds
// a few stores and a call to each tier instead of its whole body (the tiers' hot loops have to
// stay inside the instruction cache), and no register array escapes through a pointer.
template <int D>
__device__ __noinline__ uint32_t zeillinger_scratch(const uint32_t* scratch, int K, int ZS, uint32_t clm) {
    ZeilBest b;
    b.L = __int_as_float(0x7f800000);
    b.S = b.L;
    b.i = -1;
    b.j = -1;
#pragma unroll 1
    for (int i = 0; i < K; ++i) {
        if (!((clm >> i) & 1u)) continue;
        float vi[D];
#pragma unroll
        for (int c = 0; c < D; ++c) vi[c] = __uint_as_float(scratch[i * ZS + c]);
#pragma unroll 1
        for (int j = 0; j < K; ++j) {
            if (!((clm >> j) & 1u)) continue;
            float vj[D];
#pragma unroll
            for (int c = 0; c < D; ++c) vj[c] = __uint_as_float(scratch[j * ZS + c]);
            zeillinger_consider<D>(b, vi, vj, i, j);
        }
    }
    const bool found = b.i >= 0;
    float vi[D], vj[D];
#pragma unroll
    for (int c = 0; c < D; ++c) {
        vi[c] = found ? __uint_as_float(scratch[b.i * ZS + c]) : 0.0f;
        vj[c] = found ? __uint_as_float(scratch[b.j * ZS + c]) : 0.0f;
    }
    return zeillinger_mask_from_diff<D>(vi, vj, found);
}

template <typename T, int K, int D, int ZS>
__device__ __forceinline__ uint32_t zeillinger_rows(const T (&y)[K * D], uint32_t clm, uint32_t* scratch) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
#pragma unroll
        for (int c = 0; c < D; ++c) scratch[k * ZS + c] = __float_as_uint(Elem<T>::to_float(y[k * D + c]));
    }
    return zeillinger_scratch<D>(scratch, K, ZS, clm);
}

// POLICY: instantiation that can evaluate the fixed players (kept out of the ordinary step kernels)
// REC: recorded rollouts; `played` receives the coordinate bitmask and the axis the shift used (a fixed host on a game
// without live rows records 0, as hk_host_policy reports it)
// THR: rollouts with a value threshold; a game stopped there (`frozen`) takes part in the warp-wide votes of the step
// with no live row and keeps its live mask and its live rows as they are (dead rows may change: they are padded on the
// way out).  The Newton filter runs on its rows as they are (it only rewrites dead rows) and its result is dropped.
template <typename T, int N, int D, int RS = 0, bool POLICY = false, bool REC = false, bool THR = false>
__device__ __forceinline__ uint32_t game_step(T (&x)[N * D], uint32_t lm, uint32_t ops, uint32_t flags, int32_t ha,
                                              int32_t ax_in, uint32_t* scratch = nullptr, uint32_t* played = nullptr,
                                              bool frozen = false) {
    const uint32_t lm_in = lm;
    if constexpr (THR) lm = frozen ? 0u : lm;
    if (ops & HK_OP_SHIFT) {
        uint32_t cm;
        int ax = ax_in;
        if constexpr (POLICY) {
            if (flags & HK_F_HOST_ALL_COORD) {
                cm = (1u << D) - 1u;
            } else if (flags & HK_F_HOST_ZEILLINGER) {
                cm = zeillinger_rows<T, N, D, D>(x, lm, scratch);
            } else {
                cm = action_mask(ha, flags);
            }
            ax = agent_policy_axis(cm, ax_in, flags, D);
        } else {
            cm = action_mask(ha, flags);
        }
        if constexpr (REC) {
            played[0] = (POLICY && (flags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER)) && lm == 0) ? 0u : cm;
            played[1] = (uint32_t)ax;
        }
        bool apply = (ax >= 0) && (ax < D);
        if (flags & HK_F_NOOP_INVALID) apply = apply && ((cm >> (ax & 31)) & 1u);
        if (flags & HK_F_FREEZE_ENDED) apply = apply && (__popc(lm) >= 2);
        op_shift<T, N, D>(x, lm, cm, ax, apply);
    }
    if (ops & HK_OP_REPOSITION) op_reposition<T, N, D>(x, lm);
    if (ops & HK_OP_NEWTON) {
        const uint32_t lm_f = THR ? (frozen ? lm_in : lm) : lm;
        uint32_t nl;
        if constexpr (RS > 0) {
            nl = op_newton_rolled<T, N, D, RS>(x, lm_f, scratch);
        } else {
            nl = op_newton<T, N, D>(x, lm_f);
        }
        lm = (THR && frozen) ? 0u : nl;
    }
    if constexpr (Elem<T>::is_float) {
        if (ops & HK_OP_RESCALE) op_rescale<N, D>(x, lm, flags & HK_F_RESCALE_EPS);
    }
    if constexpr (THR) lm = frozen ? lm_in : lm;
    return lm;
}

// one element of the lane's shared-memory game area (float: -0.0 canonicalised to +0.0)
template <typename T>
__device__ __forceinline__ T x_row_value(const uint32_t* row, int w) {
    T v = Elem<T>::from_bits(row[w]);
    if constexpr (Elem<T>::is_float) v = v + 0.0f;
    return v;
}

// ---- compacted tiers ------------------------------------------------------------------------------
// Under real play few of the N slots are live (mean 6 of 20 after the root filter, 3 after two
// steps), and the O(K^2 d) filter only needs the live rows.  Each warp therefore picks a tier
// K in {2, 4, 8, 12, 16, N} from the maximum live count over its 32 games (warp-uniform, no
// divergence), gathers every lane's live rows into K register rows through the lane's own
// shared-memory copy of the game (slot order is kept, so the lowest-index-wins dedupe rule is
// unchanged), runs the steps on the K rows and scatters the survivors back to their slots.  In a
// multi-step rollout the warp drops to a smaller tier as soon as its live counts allow it.
struct LaneState {
    long long g;
    bool valid, shift;
    int32_t ha, ax;
    int cnt;
    int32_t len;
    bool origin;  // census only: no live row, or the lone live row sits at the origin (a fixed point of every op)
    uint32_t played[2];  // recorded rollouts: the host's coordinate bitmask and the axis of the last step (0 without a shift)
    int32_t over;        // value thresholds: the crossing step as p.over_step reports it (T + 1 while below)
};

__host__ __device__ constexpr int next_lower_tier(int K) {
    return K > 16 ? 16 : (K > 12 ? 12 : (K > 8 ? 8 : (K > 4 ? 4 : 0)));  // (the 2-row tier is for single steps only)
}

// Runs steps [st, T) of one tile on K compact rows; returns the step index at which it stopped
// (T, or earlier when every game of the warp fits the next lower tier; REC: after one step).  The lane's game area in
// shared memory (`row`) holds the current state on entry and on exit.
// THR (hk_rollout_threshold): after every step a game that has not crossed yet compares its live entries with the
// threshold; with p.stop_at_threshold a game that has crossed sits out the later steps (game_step, `frozen`) and writes
// its per-step outputs as an ended game that does not change: its done flag again, no reward, (REC) no action.
template <typename T, int N, int D, int K, bool POLICY, bool REC = false, bool THR = false>
__device__ __forceinline__ int tier_steps(const StepParams& p, LaneState& ls, uint32_t* row, uint32_t lm, int st,
                                          bool& exceed, bool& chg) {
    const long long B = p.B;
    const T padv = Elem<T>::pad(p.pad);
    const bool mutate = p.ops != 0;
    // tiers of 12 and 16 rows run the filter with a rolled victim loop through the lane's own
    // shared-memory game area (scratch); the area is rebuilt from registers at the end
    constexpr bool ROLLED = (K >= 12) && (K < N) && ((N * D) % 4 == 0);
    constexpr int RS = !ROLLED ? 0 : ((D == 3 && 4 * K <= N * D) ? 4 : D);
    constexpr int LOWER = next_lower_tier(K);
    T y[K * D];
    int idx[K];
    uint32_t clm = 0, cvalid = 0;
    if constexpr (K == N) {
        // (read again from the lane's game area: the caller keeps no register copy of the game across the tiers)
        load_game<T, N * D>(row, y);
        if constexpr (Elem<T>::is_float) {
#pragma unroll
            for (int q = 0; q < N * D; ++q) y[q] = y[q] + 0.0f;
        }
        clm = lm;
        cvalid = (N == 32) ? 0xffffffffu : ((1u << N) - 1u);
    } else {
        uint32_t m = lm;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const bool v = m != 0;
            const int i = v ? (__ffs((int)m) - 1) : 0;
            m &= m - 1;
            idx[k] = i;
            clm |= v ? (1u << k) : 0u;
#pragma unroll
            for (int c = 0; c < D; ++c) y[k * D + c] = x_row_value<T>(row, i * D + c);
        }
        cvalid = clm;
    }
    // Did the game change?  Exact for the games that matter, those with at most one live row (the
    // ended games of a long rollout, nearly all of which sit at a fixed point): their only row is
    // compact row 0 and it is compared before and after the step.  A game with two or more live
    // rows counts as changed, as does every game of a busier tile (tiers above 4 rows).
    bool tchg = (K > 4 || p.T > 1) ? true : chg;  // (a multi-step rollout changes every game that is worth playing)
    for (; st < p.T;) {
        T before[D];
#pragma unroll
        for (int c = 0; c < D; ++c) before[c] = y[c];
        const uint32_t clm_before = clm;
        int32_t ha_n = 3, ax_n = 0;
        if (ls.shift && st + 1 < p.T) {  // prefetch the next step's actions
            load_actions(p, p.flags, ls.g, st + 1, ha_n, ax_n);
        }
        const bool prev_done = ls.cnt < 2;
        if constexpr (REC) ls.played[0] = ls.played[1] = 0u;
        const bool frozen = THR && p.stop_at_threshold && ls.over <= st;
        clm = game_step<T, K, D, RS, POLICY, REC, THR>(y, clm, p.ops, p.flags, ls.ha, ls.ax, row, ls.played, frozen);
        if constexpr (THR) {
            if constexpr (REC) {
                if (frozen) {
                    ls.played[0] = 0u;
                    ls.played[1] = 0xffffffffu;  // axis -1: no move
                }
            }
            if (ls.over > p.T && exceeds<T, K, D>(y, clm, p.threshold)) ls.over = st + 1;
        }
        if (K <= 4 && p.T == 1) {
            bool diff = (clm != clm_before) || (clm_before > 1u);  // compact rows fill from 0: > 1 means two or more rows
#pragma unroll
            for (int c = 0; c < D; ++c) diff = diff || ((clm & 1u) && (Elem<T>::bits(y[c]) != Elem<T>::bits(before[c])));
            tchg = tchg || diff;
        }
        ls.cnt = __popc(clm);
        const bool dn = ls.cnt < 2;
        if (ls.valid) {
            if (p.done) p.done[(long long)st * B + ls.g] = dn ? 1 : 0;
            if (p.reward) p.reward[(long long)st * B + ls.g] = step_reward(p.flags, dn, prev_done);
        }
        if (p.done_count) {
            const int c = __popc(__ballot_sync(0xffffffffu, ls.valid && dn));
            if ((threadIdx.x & 31) == 0 && c) atomicAdd(p.done_count + st, c);
        }
        if (dn && !prev_done) ls.len = st + 1;
        ls.ha = ha_n;
        ls.ax = ax_n;
        ++st;
        if constexpr (REC) break;  // the recorder reads the state in the lane's game area after every step
        if constexpr (LOWER > 0) {
            if (st < p.T && __reduce_max_sync(0xffffffffu, ls.valid ? ls.cnt : 0) <= LOWER) break;  // re-tier
        }
    }
    chg = tchg;
    const bool last = st >= p.T;
    if (last && p.exceed_flag) exceed = exceeds<T, K, D>(y, clm, p.threshold);
    if (p.census) {  // (warp-uniform) is the game at rest?  Only ended games can be.
        if (K <= 4 || __any_sync(0xffffffffu, ls.cnt <= 1)) {
            uint32_t nz = 0;
#pragma unroll
            for (int k = 0; k < K; ++k) {
                uint32_t o = 0;
#pragma unroll
                for (int c = 0; c < D; ++c) o |= (uint32_t)Elem<T>::bits(y[k * D + c]);
                nz |= ((clm >> k) & 1u) ? o : 0u;
            }
            ls.origin = (nz == 0);
        } else {
            ls.origin = false;
        }
    }
    if (mutate) {
        if constexpr (K == N) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
#pragma unroll
                for (int c = 0; c < D; ++c) y[i * D + c] = ((clm >> i) & 1u) ? y[i * D + c] : padv;
            }
            store_game<T, N * D>(row, y);
        } else {
            if (ROLLED || (POLICY && (p.flags & HK_F_HOST_ZEILLINGER))) {  // the scratch overwrote the game area: all padding, then the survivors
                const uint32_t pw = (uint32_t)Elem<T>::bits(padv);
                if constexpr ((N * D) % 4 == 0) {
#pragma unroll
                    for (int q = 0; q < (N * D) / 4; ++q) reinterpret_cast<uint4*>(row)[q] = make_uint4(pw, pw, pw, pw);
                } else {
#pragma unroll
                    for (int q = 0; q < N * D; ++q) row[q] = pw;
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if ((cvalid >> k) & 1u) {
                    const bool lv = (clm >> k) & 1u;
#pragma unroll
                    for (int c = 0; c < D; ++c)
                        row[idx[k] * D + c] = (uint32_t)Elem<T>::bits(lv ? y[k * D + c] : padv);
                }
            }
        }
    }
    return st;
}

// ---- packed tiers: one 32-bit word per live row -------------------------------------------------------
// While every live value of the warp's games stays small (after the shift: <= 2^(27/D - 1) - 1, i.e. 255
// for D = 3 — true for whole warps through the first steps of real play, where the games with many rows
// are), a row fits ONE word: coordinate c in a field of FB = 27/D bits at bit 5 + FB c, the field's top bit
// kept clear as a guard, the row's slot index in the low 5 bits.  Then
//   * a single unsigned sort of the K words (sorting network, two min/max per compare-exchange) orders the
//     rows so that a row can only be dominated by rows BEFORE it: x_j <= x_i componentwise and x_j != x_i
//     implies word_j < word_i whatever the slots, and equal rows sort by slot, so "an equal row with a lower
//     slot kills" (remove_repeated, _fn.py:192-213) and "a dominating row kills" (_torch_ops.py:8-39,
//     _jax_ops.py:32-73) become ONE rule: row b dies iff some row a < b (sorted order) has x_a <= x_b;
//   * that test is one subtraction: (word_b | guards | 31) - word_a keeps every guard bit iff no field
//     borrows, i.e. iff x_a <= x_b in every coordinate: K (K - 1) / 2 pairs of 2.5 instructions each (IADD,
//     LOP3, half a three-input minimum) against K (K - 1) pairs of 5.5 - 7 in the exact tiers;
//   * reposition (the per-coordinate minima do not depend on the filter) is one subtraction per row.
// The tier's K words replace 3 K registers, nothing is rolled through shared memory, and the survivors go
// back to their slots from the index bits.  The vote is warp-uniform; a warp that fails it (large values,
// negative entries in live rows) has touched nothing and takes the exact tiers.  Single steps of int32
// state only.
#ifndef HK_PACKED_MIN
#define HK_PACKED_MIN 2  // smallest warp maximum of live rows that takes a packed tier (2 against 3: C2 steps 4-6 77 61 50 -> 72 52 44 us, the direct route serves the two-row chunks of the sorted order)
#endif

template <int N>
__device__ __forceinline__ void sort_words_asc(uint32_t (&k)[N]) {
#define HK_CE(i, j)                          \
    {                                        \
        const uint32_t a_ = k[i], b_ = k[j]; \
        k[i] = min(a_, b_);                  \
        k[j] = max(a_, b_);                  \
    }
#include "hk_sortnet.inc"
#undef HK_CE
}

template <int D>
struct PackedRow {
    static constexpr int FB = 27 / D;
    static constexpr uint32_t VMAX = (1u << (FB - 1)) - 1u;
    static constexpr uint32_t FMASK = (1u << FB) - 1u;
    __host__ __device__ static constexpr uint32_t guards() {
        uint32_t g = 0;
        for (int c = 0; c < D; ++c) g |= 1u << (5 + FB * c + FB - 1);
        return g;
    }
};

// One step (p.T == 1, ops include the Newton filter) of the tile on K packed rows, K >= the warp's largest
// live count `lmax`.  Returns false, with nothing written, when the values of some game do not pack.
// DIRECT (in-place single steps of a kernel that owns no other use of the stage): once the rows are gathered and the
// vote has passed, nothing reads the lane's game area again — `release()` lets the caller refill the stage at once
// (the next tile's load then runs in the shadow of this tile's arithmetic: what a second stage would buy, without its
// shared memory), and the changed rows go straight to global memory at `gdst` (the lane's game), 12 bytes per row that
// was live: dead rows are normalised and stay, the game area is left stale and `chg` is not raised.
struct NoRelease {
    __device__ __forceinline__ void operator()() const {}
};

template <int N, int D, int K, bool DIRECT = false, typename Release = NoRelease>
__device__ __forceinline__ bool tier_packed(const StepParams& p, LaneState& ls, uint32_t* row, uint32_t lm_in, int lmax, int st,
                                            bool& exceed, bool& chg, uint32_t* gdst = nullptr, Release release = Release()) {
    using P = PackedRow<D>;
    constexpr uint32_t G = P::guards();
    const uint32_t lm = ls.valid ? lm_in : 0u;  // a lane without a game to step gathers and scatters nothing
    const int cnt0 = __popc(lm);
    // The shift and the packing are ONE multiply-add chain per row: with the chosen coordinates S and the axis a,
    //   word = slot + sum_c x_c * M_c,   M_c = [c != a] 2^sh(c) + [c in S] 2^sh(a)   (shift applied)
    //                                    M_c = 2^sh(c)                               (no shift),
    // the M_c per-game constants.  The row sum s = sum_{c in S} x_c is formed beside it for the vote and the minima.
    uint32_t M[D], csel[D];
    const int ax = ls.ax;
    bool apply = false;
    {
        uint32_t cm = 0;
        if (p.ops & HK_OP_SHIFT) {
            cm = action_mask(ls.ha, p.flags);
            apply = (ax >= 0) && (ax < D);
            if (p.flags & HK_F_NOOP_INVALID) apply = apply && ((cm >> (ax & 31)) & 1u);
            if (p.flags & HK_F_FREEZE_ENDED) apply = apply && (cnt0 >= 2);
        }
        const uint32_t into = apply ? (1u << (5 + P::FB * ax)) : 0u;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            csel[c] = apply ? ((cm >> c) & 1u) : 0u;
            M[c] = ((apply && c == ax) ? 0u : (1u << (5 + P::FB * c))) + csel[c] * into;
        }
    }
    constexpr int KLOW = (K > 16) ? 16 : ((K > 12) ? 12 : (K > 8 ? 8 : (K > 4 ? 4 : 0)));  // the tier below: lmax > KLOW
    uint32_t w[K];
    uint32_t uor = 0, orig0 = 0, orig_hi = 0;
    uint32_t mn[D], mns = 0xffffffffu;
#pragma unroll
    for (int c = 0; c < D; ++c) mn[c] = 0xffffffffu;
    {
        uint32_t m = lm;
        int i = 0;
        uint32_t pa[D], ps = 0xffffffffu;  // the previous row (the minima take rows in pairs: one three-input minimum each)
#pragma unroll
        for (int c = 0; c < D; ++c) pa[c] = 0xffffffffu;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            if (k >= KLOW && k >= lmax) {  // (warp-uniform) past the warp's largest live count: parked in every lane
                w[k] = 0xffffffffu;
                continue;
            }
            // compact rows fill from 0; past the last live row the last one is read again (its values change
            // neither the vote nor the minima) and the word is parked above every live word
            const bool v = m != 0;
            i = v ? (__ffs((int)m) - 1) : i;
            m &= m - 1;
            uint32_t a[D];
#pragma unroll
            for (int c = 0; c < D; ++c) a[c] = row[i * D + c];
            if (k == 0) {  // the first row as it was (a value that does not fit its field counts as moved)
#pragma unroll
                for (int c = 0; c < D; ++c) {
                    orig0 += a[c] << (5 + P::FB * c);
                    orig_hi |= a[c];
                }
            }
            uint32_t q = (uint32_t)i, sum = 0;
#pragma unroll
            for (int c = 0; c < D; ++c) {
                q += a[c] * M[c];
                sum += a[c] * csel[c];
                uor |= a[c];
            }
            uor |= sum;
            if (k & 1) {
#pragma unroll
                for (int c = 0; c < D; ++c) mn[c] = __vimin3_u32(mn[c], pa[c], a[c]);
                mns = __vimin3_u32(mns, ps, sum);
            } else {
#pragma unroll
                for (int c = 0; c < D; ++c) pa[c] = a[c];
                ps = sum;
            }
            w[k] = v ? q : 0xffffffffu;
        }
        // (an odd row count: the last row is still pending)
#pragma unroll
        for (int c = 0; c < D; ++c) mn[c] = min(mn[c], pa[c]);
        mns = min(mns, ps);
    }
    // every value of the game, before and after the shift, fits a field (the OR of values <= 2^n - 1 is <= 2^n - 1)
    if (!__all_sync(0xffffffffu, cnt0 == 0 || uor <= P::VMAX)) return false;
    if constexpr (DIRECT) release();  // (after the vote: every lane has read its rows)
    // (DIRECT, measured and not kept: storing only the coordinates the step can have changed — the shifted axis and those
    // with a non-zero minimum — instead of whole 12-byte rows: 4-byte fragments, steps 3-4 of C2 5 % slower)
    if (p.ops & HK_OP_REPOSITION) {
        uint32_t pm = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) pm += ((apply && c == ax) ? mns : mn[c]) << (5 + P::FB * c);
        pm = cnt0 ? pm : 0u;
        // (parked words keep their top guard: every field stays >= 2^(FB-1), above every live word)
#pragma unroll
        for (int k = 0; k < K; ++k) w[k] -= pm;
    }
    sort_words_asc<K>(w);
    // the lone row of an ended game, before and after: everything else counts as changed
    const bool lone_moved = (((w[0] ^ orig0) >> 5) != 0) || (orig_hi > P::VMAX);
    uint32_t kill = 0;
#pragma unroll
    for (int b = 1; b < K; ++b) {
        if (b < lmax) {  // (warp-uniform) rows past the warp's largest live count are parked in every lane
            const uint32_t pb = w[b] | (G | 31u);
            uint32_t acc = 0xffffffffu;
#pragma unroll
            for (int a = 0; a + 1 < b; a += 2) acc = __vimin3_u32(acc, ~(pb - w[a]) & G, ~(pb - w[a + 1]) & G);
            if (b & 1) acc = min(acc, ~(pb - w[b - 1]) & G);
            kill |= (acc == 0u) ? (1u << b) : 0u;
        }
    }
    const uint32_t live0 = (cnt0 >= 32) ? 0xffffffffu : ((1u << cnt0) - 1u);
    const uint32_t alive = live0 & ~kill;
    const int cnt = __popc(alive);
    const bool prev_done = cnt0 < 2, dn = cnt < 2;
    if (ls.valid) {
        if (p.done) p.done[(long long)st * p.B + ls.g] = dn ? 1 : 0;
        if (p.reward) p.reward[(long long)st * p.B + ls.g] = step_reward(p.flags, dn, prev_done);
    }
    if (p.done_count) {
        const int c = __popc(__ballot_sync(0xffffffffu, ls.valid && dn));
        if ((threadIdx.x & 31) == 0 && c) atomicAdd(p.done_count + st, c);
    }
    if (dn && !prev_done) ls.len = st + 1;
    ls.cnt = cnt;
    ls.origin = (cnt == 0) || (cnt == 1 && (w[0] >> 5) == 0u);
    const bool gchg = (cnt0 >= 2) || (cnt0 == 1 && lone_moved);
    if constexpr (!DIRECT) chg = chg || gchg;
    if (p.exceed_flag && st + 1 >= p.T) {
        uint32_t hi = 0;
#pragma unroll
        for (int b = 0; b < K; ++b) {
#pragma unroll
            for (int c = 0; c < D; ++c) hi = ((alive >> b) & 1u) ? max(hi, (w[b] >> (5 + P::FB * c)) & P::VMAX) : hi;
        }
        exceed = (cnt > 0) && ((float)hi >= p.threshold);
    }
    const uint32_t padw = (uint32_t)(int32_t)p.pad;
#pragma unroll
    for (int b = 0; b < K; ++b) {
        if (b < lmax) {
            if (gchg && b < cnt0) {
                const bool lv = (alive >> b) & 1u;
                const int i = (int)(w[b] & 31u);
                uint32_t* dst = DIRECT ? (gdst + i * D) : (row + i * D);
                if constexpr (DIRECT && D == 3) {
                    // a 12-byte row is one 8-byte and one 4-byte store whatever its alignment (two requests instead of three)
                    uint32_t v[3];
#pragma unroll
                    for (int c = 0; c < 3; ++c) v[c] = lv ? ((w[b] >> (5 + P::FB * c)) & P::FMASK) : padw;
                    const bool ev = ((reinterpret_cast<uintptr_t>(dst) >> 2) & 1u) == 0;
                    *reinterpret_cast<uint2*>(dst + (ev ? 0 : 1)) = ev ? make_uint2(v[0], v[1]) : make_uint2(v[1], v[2]);
                    dst[ev ? 2 : 0] = ev ? v[2] : v[0];
                } else {
#pragma unroll
                    for (int c = 0; c < D; ++c) dst[c] = lv ? ((w[b] >> (5 + P::FB * c)) & P::FMASK) : padw;
                }
            }
        }
    }
    return true;
}

// Descending sort of N 32-bit keys in registers by a merge-exchange network (tools/gen_sortnet.py):
// one compare-exchange is two min/max instructions, there is no branch and no memory access.
template <int N>
__device__ __forceinline__ void sort_keys_desc(uint32_t (&k)[N]) {
#define HK_CE(i, j)                   \
    {                                 \
        const uint32_t a_ = k[i], b_ = k[j]; \
        k[i] = max(a_, b_);           \
        k[j] = min(a_, b_);           \
    }
#include "hk_sortnet.inc"
#undef HK_CE
}

// Observation features, fast path: every slot of the game becomes ONE
// 32-bit key that holds the whole row -- the coordinates in sort order, 27/D bits each, and the
// slot tag N - i (5 bits; lower slots sort first, so the sort is stable and keys of live rows are
// distinct and non-zero) -- dead slots get key 0.  The N keys are sorted in registers by a
// sorting network and the observation rows are DECODED from the sorted keys, rescaled and stored
// 16 bytes at a time: no gather, no rank counting, no loop, no shared-memory scratch.  Where the
// tag sits depends on the order: below all coordinates for the lexicographic orders, right
// below the primary coordinate for the coordinate-0 order (the remaining coordinates then ride
// along without influencing the order).  Unsorted features skip the network (slot order).
// Valid when every live value of the warp's games is an integer below 2^(27/D); the routine votes
// and returns false (warp-uniform) otherwise, and the caller falls back to features_rolled.
// The order of the raw integers is the order of the rescaled values (RN division by a positive
// constant is strictly monotonic on distinct integers below 2^23).
template <typename T, int N, int D>
__device__ __forceinline__ bool features_network(const T (&z)[N * D], uint32_t lm, int zmax, uint32_t flags, float padf,
                                                 float* orow) {
    static_assert(N <= 31 && D >= 2 && D <= 6, "5 tag bits, at least 4 bits per coordinate");
    constexpr int W = N * D;
    constexpr int BITS = 27 / D;
    constexpr uint32_t FMASK = (1u << BITS) - 1u;
    const bool sorted = flags & (HK_F_OBS_SORT_COORD0 | HK_F_OBS_SORT_LEX | HK_F_OBS_SORT_LEX_FIRST);
    const bool lex = flags & HK_F_OBS_SORT_LEX;  // last coordinate primary: field c holds coordinate D-1-c
    const bool coord0 = !lex && !(flags & HK_F_OBS_SORT_LEX_FIRST);

    // integer view of the state, its maximum over live rows (unsigned: a negative entry in a live
    // row disqualifies the game), and for float state the integrality of every live value
    uint32_t iv[W];
    uint32_t umax = 0;
    bool packable = true;
#pragma unroll
    for (int i = 0; i < N; ++i) {
        const bool lv = (lm >> i) & 1u;
        uint32_t rmax = 0;
#pragma unroll
        for (int c = 0; c < D; ++c) {
            if constexpr (Elem<T>::is_float) {
                const int q = __float2int_rz(z[i * D + c]);
                packable = packable && (!lv || ((float)q == z[i * D + c]));
                iv[i * D + c] = (uint32_t)q;
            } else {
                iv[i * D + c] = (uint32_t)z[i * D + c];
            }
            rmax = max(rmax, iv[i * D + c]);
        }
        umax = lv ? max(umax, rmax) : umax;
    }
    packable = packable && (umax <= FMASK);
    if (!__all_sync(0xffffffffu, packable)) return false;

    // field shifts (warp-uniform): field 0 on top, the tag below everything or right below field 0
    uint32_t sh[D];
    sh[0] = 5 + (D - 1) * BITS;
#pragma unroll
    for (int c = 1; c < D; ++c) sh[c] = (coord0 ? 0 : 5) + (D - 1 - c) * BITS;
    const uint32_t tag_sh = coord0 ? (D - 1) * BITS : 0;

    uint32_t key[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
        uint32_t q = (uint32_t)(N - i) << tag_sh;
#pragma unroll
        for (int c = 0; c < D; ++c) q |= (lex ? iv[i * D + (D - 1 - c)] : iv[i * D + c]) << sh[c];
        key[i] = ((lm >> i) & 1u) ? q : 0u;
    }
    if (sorted) sort_keys_desc<N>(key);

    // The sorted keys go to the TAIL of the lane's obs row (words W-N .. W-1) and the rows are decoded
    // from there in a rolled loop, four rows (= D 16-byte stores) per trip, so that the decode exists
    // once in the code instead of N*D times.  Writing rows 4t .. 4t+3 (words below 4 D (t+1))
    // overwrites only key words that have been read: key j sits at word W-N+j, so the keys hit are
    // j < 4 D (t+1) - (W-N) = 4(t+1) + (D-1)(4(t+1) - N) <= 4(t+1) for every trip but the last
    // (4(t+1) <= N), and the last trip has read all remaining keys before it writes.
    uint32_t* ks = reinterpret_cast<uint32_t*>(orow) + (W - N);
    const bool vec = (reinterpret_cast<uintptr_t>(orow) & 15u) == 0;
    if (N % 4 == 0 && (W - N) % 4 == 0 && vec) {
#pragma unroll
        for (int q = 0; q + 3 < N; q += 4) *reinterpret_cast<uint4*>(ks + q) = make_uint4(key[q], key[q + 1], key[q + 2], key[q + 3]);
    } else {
#pragma unroll
        for (int q = 0; q < N; ++q) ks[q] = key[q];
    }
    // rescale by the game maximum (max == 0 -> 1); the fast division is always safe here
    // (divisor and dividends are integers in [1, 2^BITS))
    const bool resc = flags & HK_F_OBS_RESCALE;
    const GameDivider g = make_divider(umax == 0 ? 1.0f : (float)umax, 1.0f);
#pragma unroll 1
    for (int r0 = 0; r0 < N; r0 += 4) {
        uint32_t kq[4];
        if (N % 4 == 0 && (W - N) % 4 == 0 && vec) {
            const uint4 t = *reinterpret_cast<const uint4*>(ks + r0);
            kq[0] = t.x, kq[1] = t.y, kq[2] = t.z, kq[3] = t.w;
        } else {
#pragma unroll
            for (int r = 0; r < 4; ++r) kq[r] = (r0 + r < N) ? ks[r0 + r] : 0u;
        }
        float v[4 * D];
        if (r0 < zmax || !sorted) {  // groups past the warp's live maximum are all padding
#pragma unroll
            for (int r = 0; r < 4; ++r) {
#pragma unroll
                for (int c = 0; c < D; ++c) {  // coordinate c of the row held by key kq[r]
                    const uint32_t fld = (kq[r] >> (lex ? sh[D - 1 - c] : sh[c])) & FMASK;
                    const float x = (float)fld;
                    const bool use = resc && (fld != 0);
                    const float q = divide_by_game_max(use ? x : g.b, g);
                    v[r * D + c] = (kq[r] == 0) ? padf : (use ? q : x);
                }
            }
        } else {
#pragma unroll
            for (int q = 0; q < 4 * D; ++q) v[q] = padf;
        }
        if (N % 4 == 0 && vec) {
#pragma unroll
            for (int q = 0; q < D; ++q)
                reinterpret_cast<float4*>(orow + r0 * D)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        } else {
#pragma unroll
            for (int q = 0; q < 4 * D; ++q) {
                if (r0 * D + q < W) orow[r0 * D + q] = v[q];
            }
        }
    }
    return true;
}

// Observation features, general path: ONE rolled, out-of-line routine for every live count.
// Unrolled per-tier versions (gather, rescale, K^2/2 lexicographic compares, scatter for K = 8, 12,
// 20) made the step+features kernel 240-460 KB of SASS; with the warps of an SM in different tiers
// it was instruction-fetch bound (ncu: icc hit rate 44-59 %, stall no_instruction).  Here the rows
// are walked in loops whose trip count is the warp's maximum live count `zmax`:
//   phase 0  per live row: game max / min-positive, and one 64-bit sort key
//            (live bit | coordinates in sort order, 19 bits each | 31 - k) into the scratch row;
//   phase 1  ranks by counting greater keys, four ranked rows per pass over the competitors; the
//            ranks are packed 5 bits each into two registers;
//   phase 2  the scratch row is filled with the padding value and every live row is read again from
//            the state tile, rescaled and written at its rank.
// Keys of distinct rows are distinct (the low bits break ties towards the lower slot: a stable
// sort), dead entries sort below every live row, and the order of the raw integers is the order
// of the rescaled values (RN division by a positive constant is strictly monotonic on distinct
// integers below 2^23).  When some live value of the warp's games is not an integer below 2^19
// (e.g. a rescaled float state) the rows are compared as rescaled floats instead (warp-uniform vote).
// `skew` (0 .. 3, from the lane and the row stride) makes the key accesses bank-conflict free.
template <typename T, int N, int D>
__device__ __noinline__ void features_rolled(const uint32_t* row, uint32_t lm, int zmax, uint32_t flags, float padf,
                                             float* orow, int skew) {
    static_assert(N <= 24 && D >= 2, "ranks are packed 5 bits each into two 64-bit registers; the scratch row holds 2N+8 words");
    constexpr int W = N * D;
    constexpr bool CAN_PACK = (D * 19 + 7 <= 64);
    constexpr int HI = N + 4;  // high key words after the low ones (+ the largest skew)
    const bool sorted = flags & (HK_F_OBS_SORT_COORD0 | HK_F_OBS_SORT_LEX | HK_F_OBS_SORT_LEX_FIRST);
    const bool lex = flags & HK_F_OBS_SORT_LEX;
    const bool lexf = flags & HK_F_OBS_SORT_LEX_FIRST;
    uint32_t* ks = reinterpret_cast<uint32_t*>(orow);

    // ---- phase 0 ----
    float mx = -1.0f, mnpos = 3.0e38f;
    bool packable = CAN_PACK;
    {
        uint32_t m = lm;
#pragma unroll 1
        for (int k = 0; k < zmax; ++k) {
            const bool v = m != 0;
            const int i = v ? (__ffs((int)m) - 1) : 0;
            m &= m - 1;
            uint32_t iv[D];
#pragma unroll
            for (int c = 0; c < D; ++c) {
                const T val = x_row_value<T>(row, i * D + c);
                const float fv = Elem<T>::to_float(val);
                if constexpr (Elem<T>::is_float) {
                    const int q = __float2int_rz(val);
                    iv[c] = (uint32_t)q;
                    packable = packable && (!v || ((float)q == val));
                } else {
                    iv[c] = (uint32_t)val;
                }
                packable = packable && (!v || iv[c] < (1u << 19));
                mx = v ? fmaxf(mx, fv) : mx;
                mnpos = (v && fv > 0.0f) ? fminf(mnpos, fv) : mnpos;
            }
            if constexpr (CAN_PACK) {
                uint64_t q = 0;
                if (lex) {  // last coordinate primary
#pragma unroll
                    for (int c = D - 1; c >= 0; --c) q = (q << 19) | (iv[c] & 0x7ffffu);
                } else if (lexf) {  // coordinate 0 primary
#pragma unroll
                    for (int c = 0; c < D; ++c) q = (q << 19) | (iv[c] & 0x7ffffu);
                } else {
                    q = iv[0] & 0x7ffffu;
                }
                const uint64_t key = v ? ((1ull << 62) | (q << 5) | (uint32_t)(31 - k)) : (uint64_t)(31 - k);
                ks[skew + k] = (uint32_t)key;
                ks[HI + skew + k] = (uint32_t)(key >> 32);
            }
        }
    }
    if (mx == 0.0f || ((flags & HK_F_RESCALE_EPS) && mx > 0.0f && mx <= 1e-8f)) mx = 1.0f;
    // both votes are taken by ALL lanes, outside any per-game condition
    const bool act = (flags & HK_F_OBS_RESCALE) && (mx > 0.0f);
    const GameDivider g = make_divider(act ? mx : 1.0f, mnpos);
    const bool fast = __all_sync(0xffffffffu, !act || g.safe);
    packable = __all_sync(0xffffffffu, packable);
    auto rescaled = [&](float v) -> float {
        const bool use = act && (v != 0.0f);  // 0 / mx = 0 exactly
        const float a = use ? v : g.b;
        const float q = fast ? divide_by_game_max(a, g) : __fdiv_rn(a, g.b);
        return use ? q : v;
    };

    // ---- phase 1 ----
    uint64_t rk0 = 0, rk1 = 0;  // rank of compact row k: 5 bits at 5k (k < 12) or 5(k - 12)
    if (sorted) {
        if (packable) {
#pragma unroll 1
            for (int kb = 0; kb < zmax; kb += 4) {
                uint64_t key[4];
                int r[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const bool ok = kb + q < zmax;
                    const uint32_t lo = ok ? ks[skew + kb + q] : 0xffffffffu;
                    const uint32_t hi = ok ? ks[HI + skew + kb + q] : 0xffffffffu;
                    key[q] = ((uint64_t)hi << 32) | lo;
                    r[q] = 0;
                }
#pragma unroll 1
                for (int j = 0; j < zmax; ++j) {
                    const uint64_t kj = ((uint64_t)ks[HI + skew + j] << 32) | ks[skew + j];
#pragma unroll
                    for (int q = 0; q < 4; ++q) r[q] += (kj > key[q]) ? 1 : 0;
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int kk = kb + q;
                    if (kk < zmax) {
                        if (kk < 12) rk0 |= (uint64_t)r[q] << (5 * kk);
                        else rk1 |= (uint64_t)r[q] << (5 * (kk - 12));
                    }
                }
            }
        } else {
            // rescaled float rows into the scratch row (dead entries negative: below every live row)
            uint32_t m = lm;
#pragma unroll 1
            for (int k = 0; k < zmax; ++k) {
                const bool v = m != 0;
                const int i = v ? (__ffs((int)m) - 1) : 0;
                m &= m - 1;
#pragma unroll
                for (int c = 0; c < D; ++c)
                    orow[k * D + c] = v ? rescaled(Elem<T>::to_float(x_row_value<T>(row, i * D + c))) : -1.0f;
            }
#pragma unroll 1
            for (int kb = 0; kb < zmax; kb += 4) {
                float fk[4][D];
                int r[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const bool ok = kb + q < zmax;
#pragma unroll
                    for (int c = 0; c < D; ++c) fk[q][c] = ok ? orow[(kb + q) * D + c] : 0.0f;
                    r[q] = 0;
                }
#pragma unroll 1
                for (int j = 0; j < zmax; ++j) {
                    float fj[D];
#pragma unroll
                    for (int c = 0; c < D; ++c) fj[c] = orow[j * D + c];
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        // does row j sort before row kb+q?  strictly greater key, or equal key and lower slot
                        bool gt = fj[0] > fk[q][0];
                        bool eq = fj[0] == fk[q][0];
                        if (lex) {
#pragma unroll
                            for (int c = 1; c < D; ++c) {
                                gt = (fj[c] > fk[q][c]) || ((fj[c] == fk[q][c]) && gt);
                                eq = eq && (fj[c] == fk[q][c]);
                            }
                        } else if (lexf) {
                            gt = fj[D - 1] > fk[q][D - 1];
                            eq = fj[D - 1] == fk[q][D - 1];
#pragma unroll
                            for (int c = D - 2; c >= 0; --c) {
                                gt = (fj[c] > fk[q][c]) || ((fj[c] == fk[q][c]) && gt);
                                eq = eq && (fj[c] == fk[q][c]);
                            }
                        }
                        r[q] += (gt || (eq && j < kb + q)) ? 1 : 0;
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int kk = kb + q;
                    if (kk < zmax) {
                        if (kk < 12) rk0 |= (uint64_t)r[q] << (5 * kk);
                        else rk1 |= (uint64_t)r[q] << (5 * (kk - 12));
                    }
                }
            }
        }
    }

    // ---- phase 2: all padding, then the live rows at their ranks ----
    if constexpr ((W & 3) == 0) {
        if ((reinterpret_cast<uintptr_t>(orow) & 15u) == 0) {
            const float4 pv = make_float4(padf, padf, padf, padf);
#pragma unroll 1
            for (int q = 0; q < W / 4; ++q) reinterpret_cast<float4*>(orow)[q] = pv;
        } else {
#pragma unroll 1
            for (int q = 0; q < W; ++q) orow[q] = padf;
        }
    } else {
#pragma unroll 1
        for (int q = 0; q < W; ++q) orow[q] = padf;
    }
    {
        uint32_t m = lm;
#pragma unroll 1
        for (int k = 0; k < zmax; ++k) {
            const bool v = m != 0;
            const int i = v ? (__ffs((int)m) - 1) : 0;
            m &= m - 1;
            const int rank = !sorted ? i : (int)(((k < 12) ? (rk0 >> (5 * k)) : (rk1 >> (5 * (k - 12)))) & 31u);
            if (v) {
#pragma unroll
                for (int c = 0; c < D; ++c)
                    orow[rank * D + c] = rescaled(Elem<T>::to_float(x_row_value<T>(row, i * D + c)));
            }
        }
    }
}

// One tile (the lane's game sits in `row`, its shared-memory area) through all p.T steps: liveness pass and
// dead-row check, the warp's tier by the largest live count, the steps on compact rows, per-step outputs.
// On return `row` holds the new state, ls.cnt / ls.len / ls.origin describe it, `chg` says whether the
// game must be written back.  Shared by the tile-ring kernel below and the census-scheduled kernel
// (hk_sched.cuh).
// `gdst` (optional, with `release`): the lane's game in global memory of an in-place call whose stage may be refilled
// as soon as the packed tiers have gathered their rows (tier_packed, DIRECT); returns true when that route was taken
// (the stage has been released, the game is already in global memory, `row` is stale).
// `rec` (recorded rollouts): rec(st, false) before step st with the state in `row`, rec(st, true) after it with
// ls.played set; the tiers then stop after every step.
struct NoRec {
    __device__ __forceinline__ void operator()(int, bool) const {}
};

// THR (hk_rollout_threshold): ls.over is set from the state on entry and kept by the tiers (tier_steps).
template <typename T, int N, int D, bool POLICY, bool PACKED = true, typename Release = NoRelease, typename Rec = NoRec,
          bool THR = false>
__device__ __forceinline__ bool small_process_tile(const StepParams& p, LaneState& ls, uint32_t* row, bool& exceed,
                                                   bool& chg, uint32_t* gdst = nullptr, Release release = Release(),
                                                   Rec rec = Rec()) {
    constexpr int W = N * D;
    constexpr bool REC = !std::is_same<Rec, NoRec>::value;
    static_assert(!(REC && PACKED), "a recorded rollout steps on the exact tiers only");
    static_assert(!(THR && PACKED), "a rollout with a value threshold steps on the exact tiers only");
    const T padv = Elem<T>::pad(p.pad);
    const bool mutate = p.ops != 0;
    bool normalised = false;
    ls.len = -1;
    int st = 0;
    do {
        const int st0 = st;
        if constexpr (REC) rec(st0, false);
        bool any_junk = false;
        uint32_t lm;
        {
        // (block scope: the register copy of the game lives for this pass only; the tiers read the lane's game area)
        T x[W];
        load_game<T, W>(row, x);
        if constexpr (Elem<T>::is_float) {
            uint32_t canon = 0;
#pragma unroll
            for (int q = 0; q < W; ++q) {  // canonicalise -0.0 (a game that held one counts as changed)
                const float c = x[q] + 0.0f;
                canon |= (uint32_t)__float_as_int(x[q]) ^ (uint32_t)__float_as_int(c);
                x[q] = c;
            }
            chg = chg || (canon != 0);
        }
        // Every reference op rewrites dead rows with the padding value.  States produced by these
        // kernels already satisfy that, so the tile is only CHECKED here (a dead row that holds anything
        // else counts as a change of its game) and the rewrite below runs only if some game needs it.
        // One pass yields the live mask (sign of coordinate 0) and the check.
        {
            const bool check = mutate && !normalised;
            const uint32_t pbits = (uint32_t)Elem<T>::bits(padv);
            uint32_t dead = 0, diff = 0;
#pragma unroll
            for (int i = 0; i < N; ++i) {
                const uint32_t sgn = (uint32_t)(Elem<T>::bits(x[i * D]) >> 31);  // all ones <=> dead row
                dead |= sgn & (1u << i);
                uint32_t dr = 0;
#pragma unroll
                for (int c = 0; c < D; ++c) dr |= (uint32_t)Elem<T>::bits(x[i * D + c]) ^ pbits;
                diff |= dr & sgn;
            }
            lm = ~dead & ((N == 32) ? 0xffffffffu : ((1u << N) - 1u));
            if constexpr (THR) {
                if (st == 0) ls.over = exceeds<T, N, D>(x, lm, p.threshold) ? 0 : p.T + 1;
            }
            if (check) {
                chg = chg || (diff != 0);
                any_junk = __any_sync(0xffffffffu, diff != 0);
            }
        }
        }
        ls.cnt = __popc(lm);
        if (ls.len < 0) ls.len = (ls.cnt < 2) ? 0 : p.T + 1;
        const int lmax = __reduce_max_sync(0xffffffffu, ls.valid ? ls.cnt : 0);
        // the gathered tiers scatter only live rows: dead rows that need it are rewritten first
        auto prestore = [&]() {
            if (mutate && !normalised) {
                if (any_junk) {
                    T x[W];
                    load_game<T, W>(row, x);
                    if constexpr (Elem<T>::is_float) {
#pragma unroll
                        for (int q = 0; q < W; ++q) x[q] = x[q] + 0.0f;
                    }
#pragma unroll
                    for (int i = 0; i < N; ++i) {
#pragma unroll
                        for (int c = 0; c < D; ++c) x[i * D + c] = ((lm >> i) & 1u) ? x[i * D + c] : padv;
                    }
                    store_game<T, W>(row, x);
                }
                normalised = true;
            }
        };
        // (Measured and not kept: dropping the exact 12- and 16-row tiers from the kernels that have packed ones — 3k
        // instructions less — sends warps whose values no longer pack, common from the fifth step on, to all N rows:
        // rollout mean 0.0449 -> 0.0470 ms per step.)
        constexpr bool HAS_PACKED = PACKED && !Elem<T>::is_float && !POLICY && D == 3;
        if constexpr (HAS_PACKED) {
            // (warp-uniform) single steps with the filter: packed rows while the values allow it.  (Measured and not kept
            // for one-launch rollouts: the game would go back to the lane's game area after every packed step and be
            // gathered again for the next one, 1.07 ms per 20-step C2 rollout against 0.64 ms with the exact tiers, which
            // keep their rows in registers from step to step.)
            if ((p.ops & HK_OP_NEWTON) && lmax <= 20 && (p.T == 1 && lmax >= HK_PACKED_MIN)) {
                prestore();
                int32_t ha_n = 3, ax_n = 0;
                if (ls.shift && st + 1 < p.T) load_actions(p, p.flags, ls.g, st + 1, ha_n, ax_n);  // the next step's actions
                bool ok = false, tried = false;
                if constexpr (!std::is_same<Release, NoRelease>::value) {
                    // (warp-uniform) direct route: in place, one step, no dead row had to be rewritten, nothing pending
                    // (up to 8 rows: the 12-byte row stores of a lane are uncoalesced, three store instructions per row
                    // slot — measured at C2: 18 % faster than the staged tile at 4 rows, 7 % at 8, 25 % SLOWER at 12 and
                    // 2.5 times slower on the 20-row root filter)
                    if (gdst != nullptr && p.T == 1 && lmax <= 8 && !any_junk && !__any_sync(0xffffffffu, chg)) {
                        if (lmax <= 4) ok = tier_packed<N, D, 4, true, Release>(p, ls, row, lm, lmax, st, exceed, chg, gdst, release);
                        else ok = tier_packed<N, D, 8, true, Release>(p, ls, row, lm, lmax, st, exceed, chg, gdst, release);
                        if (ok) return true;
                        tried = true;  // (the values do not pack: the exact tiers below)
                    }
                }
                if (!tried) {
                    if (lmax <= 4) ok = tier_packed<N, D, 4>(p, ls, row, lm, lmax, st, exceed, chg);
                    else if (lmax <= 8) ok = tier_packed<N, D, 8>(p, ls, row, lm, lmax, st, exceed, chg);
                    else if (lmax <= 12) ok = tier_packed<N, D, 12>(p, ls, row, lm, lmax, st, exceed, chg);
                    else if (N <= 16 || lmax <= 16) ok = tier_packed<N, D, 16>(p, ls, row, lm, lmax, st, exceed, chg);
                    else ok = tier_packed<N, D, (N > 16 ? 20 : 16)>(p, ls, row, lm, lmax, st, exceed, chg);  // (the root filter of (20,3))
                }
                if (ok) {
                    ls.ha = ha_n;
                    ls.ax = ax_n;
                    ++st;
                    continue;
                }
            }
        }
        if (N > 2 && p.T == 1 && lmax <= 2) {  // the tail of a rollout driven step by step: ended games and two-point games only
            prestore();
            st = tier_steps<T, N, D, (N > 2 ? 2 : N), POLICY, REC, THR>(p, ls, row, lm, st, exceed, chg);
        } else if (N > 4 && lmax <= 4) {
            prestore();
            st = tier_steps<T, N, D, (N > 4 ? 4 : N), POLICY, REC, THR>(p, ls, row, lm, st, exceed, chg);
        } else if (N > 8 && lmax <= 8) {
            prestore();
            st = tier_steps<T, N, D, (N > 8 ? 8 : N), POLICY, REC, THR>(p, ls, row, lm, st, exceed, chg);
        } else if (N > 12 && lmax <= 12) {
            if (W % 4 != 0) prestore();
            st = tier_steps<T, N, D, (N > 12 ? 12 : N), POLICY, REC, THR>(p, ls, row, lm, st, exceed, chg);
            normalised = normalised || (W % 4 == 0);
        } else if (N > 16 && lmax <= 16) {
            if (W % 4 != 0) prestore();
            st = tier_steps<T, N, D, (N > 16 ? 16 : N), POLICY, REC, THR>(p, ls, row, lm, st, exceed, chg);
            normalised = normalised || (W % 4 == 0);
        } else {
            st = tier_steps<T, N, D, N, POLICY, REC, THR>(p, ls, row, lm, st, exceed, chg);
            normalised = true;
        }
        if constexpr (REC) rec(st0, true);
    } while (st < p.T);
    return false;
}

// ---- a lane's observation row ---------------------------------------------------------------------
// Features of the game in the lane's row of the stage into orow (row stride OW words).  Every warp takes the same
// route whatever its live counts (sorting network; the rolled routine only when values do not pack): per-tier variants
// made the warps of an SM execute different code and the kernels instruction-fetch bound.  holds_game: the lane's row
// is a game of the batch (the others do not count towards the warp's largest live count).
template <typename T, int N, int D>
__device__ __forceinline__ void lane_features(const StepParams& p, const uint32_t* row, float* orow, int OW, int lane,
                                              const bool& holds_game) {
    constexpr int W = N * D;
    T z[W];
    load_game<T, W>(row, z);
    if constexpr (Elem<T>::is_float) {
#pragma unroll
        for (int q = 0; q < W; ++q) z[q] = z[q] + 0.0f;
    }
    const uint32_t zl = live_mask<T, N, D>(z);
    const int zmax = __reduce_max_sync(0xffffffffu, holds_game ? __popc(zl) : 0);
    bool built = false;
    if constexpr (D <= 6) built = features_network<T, N, D>(z, zl, zmax, p.flags, p.pad, orow);
    if (!built) {
        // rows of stride OW words: lanes 32/g apart share a bank (g = largest power of two in OW)
        const int gpow = (OW & -OW) > 32 ? 32 : (OW & -OW);
        features_rolled<T, N, D>(row, zl, zmax, p.flags, p.pad, orow, (lane * gpow) >> 5);
    }
}

// the coordinates p.obs_coord names for game g, as D floats 0/1 after the W feature words
template <int D>
__device__ __forceinline__ void append_obs_coord(const StepParams& p, long long g, const bool& holds_game, float* orow, int W) {
    if (!p.obs_coord) return;
    const uint32_t ocm = holds_game ? action_mask(load_action(p.obs_coord, g, p.flags), p.flags) : 0u;
#pragma unroll
    for (int k = 0; k < D; ++k) orow[W + k] = (float)((ocm >> k) & 1u);
}

// ---- tile movement -------------------------------------------------------------------------------
__device__ __forceinline__ void warp_copy_words(uint32_t* dst, const uint32_t* src, int words, int lane) {
    for (int w = lane; w < words; w += 32) dst[w] = src[w];
}

// The thread-per-game kernel: a warp-private stage of one tile of 32 games, WARPS warps per CTA, one persistent wave.
// PACKED = false: the instantiation of the one-launch rollouts (p.T > 1), which never take the packed tiers and are bound
// by instruction fetch: they do not carry that code.
// V (SmallVariant): Obs builds the features of the final state into the warp's obs tile.  Rec (recorded rollouts):
// before every step the features of the state go to the warp's obs tile, after it the played actions are written and
// the tile leaves with one bulk store into row st of p.obs_t.  Thr, ThrRec: rollouts with a value threshold, recorded or
// not; p.over_step leaves with length.
template <typename T, int N, int D, bool POLICY, int WARPS, bool PACKED, SmallVariant V>
__device__ __forceinline__ void small_kernel_body(const StepParams& p) {
    // (static: plain constexpr locals are captured by the [&] lambdas below, which changes the code the compiler emits)
    static constexpr bool OBS = is_obs(V), REC = is_rec(V), THR = is_thr(V);
    using L = SmallLayout<N, D, OBS || REC, WARPS>;
    constexpr int SMALL_WARPS = WARPS;
    // One stage per warp.  The stage index `s` below is always 0, but it stays a loop variable: with the index folded by
    // hand (one mbarrier, one phase bit, no rotation) ptxas emits different code for every variant.
    constexpr int SMALL_STAGES = 1;
    constexpr int W = L::W;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw) + warp * SMALL_STAGES;
    uint32_t* ring = reinterpret_cast<uint32_t*>(smem_raw + SMALL_BAR_BYTES) + (size_t)warp * L::WARP_WORDS;
    float* obs_tile = reinterpret_cast<float*>(ring + SMALL_STAGES * L::TILE_WORDS);

    const long long B = p.B;
    const long long ntiles = (B + 31) >> 5;
    const long long gw = (long long)blockIdx.x * SMALL_WARPS + warp;
    const long long nw = (long long)gridDim.x * SMALL_WARPS;
    const uint32_t* gin = reinterpret_cast<const uint32_t*>(p.in);
    uint32_t* gout = reinterpret_cast<uint32_t*>(p.out);
    const bool tma_base = aligned16(p.in) && aligned16(p.out);
    const int OW = W + ((REC ? p.agent_obs : p.obs_coord != nullptr) ? D : 0);
    const bool obs_tma = aligned16(p.obs);
    const T padv = Elem<T>::pad(p.pad);
    const bool write = (gout != nullptr);
    const bool inplace = (gout == gin) && !(p.flags & HK_F_STORE_ALL);

    pdl_launch_dependents();  // the next launch of the stream may begin its prologue as SMs free up
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < SMALL_STAGES; ++s) mbar_init(&bar[s], 1);
        mbar_fence_init();
    }
    __syncwarp();
    pdl_wait_prior_grid();  // everything below reads or writes global memory of the previous launch

    auto tile_words = [&](long long t) -> int {
        long long left = B - (t << 5);
        return (int)(left < 32 ? left : 32) * W;
    };
    auto tile_tma = [&](long long t) -> bool { return tma_base && ((tile_words(t) & 3) == 0); };
    auto issue_load = [&](long long t, int s) {
        if (t < ntiles && tile_tma(t)) {
            const uint32_t bytes = (uint32_t)tile_words(t) * 4u;
            mbar_expect_tx(&bar[s], bytes);
            bulk_load(ring + s * L::TILE_WORDS, gin + t * (long long)L::TILE_WORDS, bytes, &bar[s]);
        }
    };

    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < SMALL_STAGES; ++s) issue_load(gw + s * nw, s);
    }

    uint32_t phase_bits = 0;  // bit s = parity to wait for on stage s
    int s = 0;
    for (long long t = gw; t < ntiles; t += nw) {
        uint32_t* stage = ring + s * L::TILE_WORDS;
        uint32_t* row = stage + lane * W;
        float* orow = obs_tile + lane * OW;
        LaneState ls;
        ls.g = (t << 5) + lane;
        ls.valid = ls.g < B;
        const int words = tile_words(t);
        const bool tma = tile_tma(t);
        ls.shift = (p.ops & HK_OP_SHIFT) && ls.valid;
        ls.ha = 3;
        ls.ax = 0;
        if (ls.shift) {
            load_actions(p, p.flags, ls.g, 0, ls.ha, ls.ax);
        }

        // (measured and not kept: a prefetch of the warp's next tile into L2 here, cp.async.bulk.prefetch.L2, +5 % on the
        // first steps at 16 warps per SM, -8 % only at 8)
        if (tma) {
            mbar_wait(&bar[s], (phase_bits >> s) & 1u);
            phase_bits ^= (1u << s);
        } else {
            warp_copy_words(stage, gin + t * (long long)L::TILE_WORDS, words, lane);
            __syncwarp();
        }

        bool exceed = false;
        // Did this lane's game change?  Unchanged games of an in-place call are not written back
        // (everything is when out != in).
        bool chg = !inplace;
        if constexpr (REC) {
            const int nrows = words / W;
            auto rec = [&](int st, bool after) {
                if (!after) {
                    if (p.obs_t == nullptr) return;
                    if (lane == 0) bulk_wait_read<0>();  // the previous row's store has read the obs tile
                    __syncwarp();
                    lane_features<T, N, D>(p, row, orow, OW, lane, ls.valid);
                    return;
                }
                if (ls.valid) {
                    const long long o = (long long)st * B + ls.g;
                    if (p.host_mask_t) p.host_mask_t[o] = (int32_t)ls.played[0];
                    if (p.axis_played_t) p.axis_played_t[o] = (int32_t)ls.played[1];
                }
                if (p.obs_t == nullptr) return;
                if (p.agent_obs) {
#pragma unroll
                    for (int k = 0; k < D; ++k) orow[W + k] = (float)((ls.played[0] >> k) & 1u);
                }
                const int owords = nrows * OW;
                float* gobs = p.obs_t + ((long long)st * B + (t << 5)) * OW;
                if (aligned16(gobs) && (owords & 3) == 0) {
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        bulk_store(gobs, obs_tile, (uint32_t)owords * 4u);
                        bulk_commit();
                    }
                } else {
                    __syncwarp();
                    warp_copy_words(reinterpret_cast<uint32_t*>(gobs), reinterpret_cast<uint32_t*>(obs_tile), owords, lane);
                    __syncwarp();
                }
            };
            small_process_tile<T, N, D, POLICY, PACKED, NoRelease, decltype(rec), THR>(p, ls, row, exceed, chg, nullptr, NoRelease(),
                                                                                   rec);
        } else if constexpr (THR) {
            small_process_tile<T, N, D, POLICY, PACKED, NoRelease, NoRec, THR>(p, ls, row, exceed, chg);
        } else {
            // (measured and not kept: the direct route of the packed tiers here, as in the census kernel — C2 steps 2-4
            // 94 92 79 -> 82 73 67 us, but every later step 68 us instead of 50-60: rollout mean 0.0658 -> 0.0672 ms)
            small_process_tile<T, N, D, POLICY, PACKED>(p, ls, row, exceed, chg);
        }

        if (ls.valid) {
            if (p.num_points) p.num_points[ls.g] = ls.cnt;
            if (p.length) p.length[ls.g] = ls.len;
            if constexpr (THR) {
                if (p.over_step) p.over_step[ls.g] = ls.over;
            }
        }
        if (p.exceed_flag) {
            if (__any_sync(0xffffffffu, exceed && ls.valid) && lane == 0) *p.exceed_flag = 1;
        }

        // ---- write-back.  In a long rollout most games have ended and sit at a fixed point (a lone
        // point at the origin), so most games of an in-place step do not change: only changed games are
        // written.  Many changed games -> the whole tile in one bulk store (rewriting an unchanged game
        // is harmless); a few -> one coalesced copy per changed game; none -> nothing.
        bool stored = false;
        if (write) {
            const uint32_t dirty = __ballot_sync(0xffffffffu, ls.valid && chg);
            const int ndirty = __popc(dirty);
            if (ndirty > HK_SPARSE_STORE_MAX) {
                if (tma) {
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) bulk_store(gout + t * (long long)L::TILE_WORDS, stage, (uint32_t)words * 4u);
                    stored = true;
                } else {
                    __syncwarp();
                    warp_copy_words(gout + t * (long long)L::TILE_WORDS, stage, words, lane);
                    __syncwarp();
                }
            } else if (ndirty > 0) {
                __syncwarp();
                uint32_t m = dirty;
                while (m) {
                    const int gi = __ffs((int)m) - 1;
                    m &= m - 1;
                    const uint32_t* src = stage + gi * W;
                    uint32_t* dst = gout + (t * 32ll + gi) * W;
                    if (W % 4 == 0 && tma_base) {
                        if (lane < W / 4) reinterpret_cast<uint4*>(dst)[lane] = reinterpret_cast<const uint4*>(src)[lane];
                    } else {
                        warp_copy_words(dst, src, W, lane);
                    }
                }
                __syncwarp();
            }
        }
        if constexpr (OBS) {
            if (p.obs) {
                // Observation features of the FINAL state of the tile (survivors scattered back to their slots), as a
                // phase of its own after the steps
                lane_features<T, N, D>(p, row, orow, OW, lane, ls.valid);
                append_obs_coord<D>(p, ls.g, ls.valid, orow, W);
                const int owords = (words / W) * OW;
                float* gobs = p.obs + t * 32ll * OW;
                if (obs_tma && ((owords & 3) == 0)) {
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) bulk_store(gobs, obs_tile, (uint32_t)owords * 4u);
                    stored = true;
                } else {
                    __syncwarp();
                    warp_copy_words(reinterpret_cast<uint32_t*>(gobs), reinterpret_cast<uint32_t*>(obs_tile), owords,
                                    lane);
                    __syncwarp();
                }
            }
        }
        // the lanes wrote this stage with st.shared (results, scratch); the refill below is an async-proxy
        // write into the same bytes: order the two proxies before lane 0 issues it
        fence_async_smem();
        __syncwarp();
        if (lane == 0) {
            if (stored) {
                bulk_commit();
                bulk_wait_read<0>();  // the stage (and obs tile) may be overwritten from here on
            }
            issue_load(t + SMALL_STAGES * nw, s);
        }
        __syncwarp();
        s = (s + 1 == SMALL_STAGES) ? 0 : s + 1;
    }
    if (lane == 0) bulk_wait_all<0>();  // all bulk stores globally complete before the warp retires
}

template <typename T, int N, int D, bool POLICY, int WARPS, bool PACKED, SmallVariant V>
__global__ void __launch_bounds__(WARPS * 32) hk_small_kernel(const StepParams p) {
    small_kernel_body<T, N, D, POLICY, WARPS, PACKED, V>(p);
}

}  // namespace hk
