// hk_generic.cuh — warp-per-game step kernel for any (N <= 1024, d <= 10).
//
// Mapping (DESIGN.md "K-warp"): one warp owns one game at a time.  The game's N*d words are
// double-buffered in the warp's private shared-memory slots with cp.async (LDGSTS): while game g is
// processed, game g + (number of warps) streams in (games of this class are 1-16 KB, too small for an
// efficient TMA transaction each); results leave through coalesced 16-byte stores, and an unchanged
// game of an in-place call is not stored at all.  After the liveness pass a game takes one of three
// routes: ended games (<= 1 live row) a short path of their own; games with 2-32 live rows are
// compacted and stepped with ONE compact row per lane; everything else (more live rows, multi-step
// rollouts, fused observation, fixed players, remove_repeated) runs on the padded layout, lane l
// owning rows l, l+32, ..., with the compact list of live rows feeding the dominator loop.  This is
// the kernel for BASELINE config 5 (N=64, d=5).
#pragma once
#include "hk_census.cuh"

#ifndef HK_GENERIC_MIN_CTAS
#define HK_GENERIC_MIN_CTAS 4  // resident CTAs of 8 warps the register budget is sized for (tools/time_c5.py)
#endif

namespace hk {

template <typename T>
__device__ __forceinline__ T warp_min(T v) {
    if constexpr (!Elem<T>::is_float) {
        return (T)__reduce_min_sync(0xffffffffu, (int)v);  // one REDUX instead of five shuffle + min rounds
    } else {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            T u = __shfl_xor_sync(0xffffffffu, v, o);
            v = u < v ? u : v;
        }
        return v;
    }
}

__device__ __forceinline__ float warp_maxf(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

constexpr uint32_t GENERIC_HOT_OPS = HK_OP_SHIFT | HK_OP_REPOSITION | HK_OP_NEWTON;
constexpr uint32_t GENERIC_HOT_FLAGS = HK_F_ACT_DISCRETE;

// words per row of the compact live-row list: D coordinates + the slot number, rounded up to an even
// count so that a pair of rows is a whole number of 16-byte words
__host__ __device__ constexpr int generic_compact_stride(int D) { return (D + 2) & ~1; }

// Observation features of one game as it stands (live rows from the bits of `mylive`, lane l owning rows l, l + 32, ...)
// into its row `gobs` of an obs array; `f` is the warp's feature buffer (N*d floats).  The recorded rollouts call it before
// every step.  It computes what the step's observation phase at the end of hk_generic_kernel computes; that phase keeps
// its own copy because calling this function there changes the instruction schedule of the step + features kernels.
template <typename T, int D, int RT>
__device__ __forceinline__ void generic_features(const T* x, uint32_t mylive, float* f, float* gobs, int N, int R, int lane,
                                                 uint32_t kflags, float pad) {
    constexpr int UNR = RT > 0 ? RT : 1;
    float mx = -1.0f;
    _Pragma("unroll UNR")
    for (int r = 0; r < R; ++r) {
        if (!((mylive >> r) & 1u)) continue;
        const int i = lane + 32 * r;
#pragma unroll
        for (int k = 0; k < D; ++k) mx = fmaxf(mx, Elem<T>::to_float(x[i * D + k]));
    }
    mx = warp_maxf(mx);
    if (mx == 0.0f || ((kflags & HK_F_RESCALE_EPS) && mx > 0.0f && mx <= 1e-8f)) mx = 1.0f;
    const bool resc = (kflags & HK_F_OBS_RESCALE) && (mx > 0.0f);
    _Pragma("unroll UNR")
    for (int r = 0; r < R; ++r) {
        const int i = lane + 32 * r;
        if (i >= N) continue;
        const bool lv = (mylive >> r) & 1u;
#pragma unroll
        for (int k = 0; k < D; ++k) {
            float v = Elem<T>::to_float(x[i * D + k]);
            v = (resc && lv && v != 0.0f) ? __fdiv_rn(v, mx) : v;
            f[i * D + k] = lv ? v : pad;
        }
    }
    __syncwarp();
    const bool sorted = kflags & (HK_F_OBS_SORT_COORD0 | HK_F_OBS_SORT_LEX | HK_F_OBS_SORT_LEX_FIRST);
    const bool lex = kflags & HK_F_OBS_SORT_LEX;
    const bool lexf = kflags & HK_F_OBS_SORT_LEX_FIRST;
    _Pragma("unroll UNR")
    for (int r = 0; r < R; ++r) {
        const int i = lane + 32 * r;
        if (i >= N) continue;
        float fi[D];
#pragma unroll
        for (int k = 0; k < D; ++k) fi[k] = f[i * D + k];
        int rank = i;
        if (sorted) {
            rank = 0;
            for (int j = 0; j < N; ++j) {
                bool gt = f[j * D] > fi[0];
                bool eq = f[j * D] == fi[0];
                if (lex) {
#pragma unroll
                    for (int k = 1; k < D; ++k) {
                        const float fj = f[j * D + k];
                        gt = (fj > fi[k]) || ((fj == fi[k]) && gt);
                        eq = eq && (fj == fi[k]);
                    }
                } else if (lexf) {
                    gt = f[j * D + D - 1] > fi[D - 1];
                    eq = f[j * D + D - 1] == fi[D - 1];
#pragma unroll
                    for (int k = D - 2; k >= 0; --k) {
                        const float fj = f[j * D + k];
                        gt = (fj > fi[k]) || ((fj == fi[k]) && gt);
                        eq = eq && (fj == fi[k]);
                    }
                }
                rank += (gt || (eq && j < i)) ? 1 : 0;
            }
        }
#pragma unroll
        for (int k = 0; k < D; ++k) gobs[rank * D + k] = fi[k];
    }
}

// smem per warp: two state buffers x[2][Wpad] (the next game is in flight while the current one is processed), then
// (OBS) f[Wpad] floats, then lmw[ceil(N/32)] (padded to 4 words), then the compact list of live rows,
// (N + 1) * generic_compact_stride(D) words
// RT = rows per lane known at compile time (1: N <= 32, 2: N <= 64; the r-loops unroll and their
// guards become predication) or 0 for any N (run-time loops).
// V (GenericVariant):
// CENSUS (Census, CensusHot): the instantiations that serve hk_step_census (plain in-place single steps); they are
// separate so that the census bookkeeping costs the other calls nothing (the kernel is bound by instruction issue).
// REC (Rec, ThrRec): recorded rollouts (hk_rollout_record, with OBS for the feature buffer): every game takes the padded
// route, whose step loop writes the features of the state before each step to row st of p.obs_t and the played actions
// after the shift.
// THR (Thr, ThrRec): rollouts with a value threshold (hk_rollout_threshold): the crossing step of every game, from
// its live entries on entry and after every step (one vote over the rows the warp holds), goes to p.over_step; with
// p.stop_at_threshold a game that has crossed sits out the later steps of both routes and writes its per-step outputs
// as an ended game that does not change: its done flag again, no reward, (REC) no action.
template <typename T, int D, int RT, GenericVariant V>
__global__ void __launch_bounds__(256, HK_GENERIC_MIN_CTAS) hk_generic_kernel(const StepParams p, int warps_per_cta, int slot_words) {
    // (static: plain constexpr locals are captured by the [&] lambdas below, which changes the code the compiler emits)
    static constexpr bool OBS = is_obs(V), HOT = is_hot(V), CENSUS = is_census(V), REC = is_rec(V), THR = is_thr(V);
    // One game ahead in flight per warp.  Three ahead (four buffers) measured slower at C5 (0.232 vs 0.224 ms per step,
    // tail 0.148 vs 0.138): the kernel is bound by instruction issue, not by the latency of its loads.
    constexpr int NBUF = 2;
    // HOT (Hot, CensusHot): the plain random-play step (shift + reposition + newton, discrete host ids, int32 action arrays,
    // one step, no observation) with its op and flag words known at compile time, so that the dozens of
    // run-time tests of them fold away; every other call takes the general instantiation.
    const uint32_t kops = HOT ? GENERIC_HOT_OPS : p.ops;
    const uint32_t kflags = HOT ? GENERIC_HOT_FLAGS : p.flags;
    const int kT = HOT ? 1 : p.T;
    constexpr int UNR = RT > 0 ? RT : 1;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int N = p.N;
    const int W = N * D;
    const int R = RT > 0 ? RT : ((N + 31) >> 5);
    const int Wpad = (W + 3) & ~3;
    uint32_t* slot = reinterpret_cast<uint32_t*>(smem_raw) + (size_t)warp * slot_words;
    float* f = reinterpret_cast<float*>(slot + NBUF * Wpad);
    uint32_t* lmw = slot + NBUF * Wpad + (OBS ? Wpad : 0);
    constexpr int CSTRIDE = generic_compact_stride(D);                            // words per compact row (even)
    uint32_t* comp = lmw + ((((N + 31) >> 5) + 3) & ~3);                          // (N + 1) compact rows, 16-byte aligned

    const uint32_t* gin = reinterpret_cast<const uint32_t*>(p.in);
    uint32_t* gout = reinterpret_cast<uint32_t*>(p.out);
    const bool vec_in = aligned16(p.in) && ((W & 3) == 0);
    const bool vec_out = aligned16(p.out) && ((W & 3) == 0);
    const T padv = Elem<T>::pad(p.pad);
    const int OW = W + ((REC ? p.agent_obs : p.obs_coord != nullptr) ? D : 0);
    const bool inplace = (gout == gin) && !(kflags & HK_F_STORE_ALL);
    // the short path for ended games covers plain single steps only
    const bool ended_fast_path = !REC && !THR &&
        kT == 1 && !(OBS && p.obs) && !p.host_out && !(kops & ~(HK_OP_SHIFT | HK_OP_REPOSITION | HK_OP_NEWTON)) &&
        !(kflags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER | HK_F_AGENT_FIRST | HK_F_AGENT_LAST));
    const bool compact_path = !REC &&
        !(OBS && p.obs) && !p.host_out && !(kops & HK_OP_DEDUPE) &&
        !(kflags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER | HK_F_AGENT_FIRST | HK_F_AGENT_LAST));

    const long long gw = (long long)blockIdx.x * warps_per_cta + warp;
    const long long nw = (long long)gridDim.x * warps_per_cta;

    // lane l copies the 16-byte chunks l, l+32, ... of a game: how many that is
    const int chunks = W >> 2;
    const int chunk_iters = (chunks >> 5) + (((chunks & 31) > lane) ? 1 : 0);
    auto prefetch = [&](long long g, int b) {
        uint32_t* dst = slot + b * Wpad;
        const uint32_t* src = gin + g * W;
        if (vec_in) {
            if constexpr (RT > 0) {  // at most RT*32 rows: a fixed number of 16-byte chunks per lane, guarded
                constexpr int ITERS = (RT * 32 * D / 4 + 31) / 32;
                // one shared-memory address and one global address per call, immediate offsets per chunk
                const uint32_t d16 = smem_u32(dst) + 16u * lane;
                const char* s16 = reinterpret_cast<const char*>(src) + 16 * lane;
#pragma unroll
                for (int it = 0; it < ITERS; ++it) {
                    if (it < chunk_iters)
                        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d16 + 512u * it), "l"(s16 + 512 * it)
                                     : "memory");
                }
            } else {
                for (int c = lane; c < (W >> 2); c += 32) cp_async_16(dst + 4 * c, src + 4 * c);
            }
        } else {
            for (int w = lane; w < W; w += 32) cp_async_4(dst + w, src + w);
        }
    };

    // ---- census (hk_step_census): games at rest are answered from their census byte and never loaded, and
    // (rows_k > 0) the small games that hk_rows_kernel stepped just before this launch are not touched.
    // The warp visits game gw + it * nw at iteration `it`.  Census bytes are held 32 iterations at a time (lane l:
    // iteration cbase + l; two batches, so the look-ahead never waits on a load); a ballot turns a batch into a
    // mask of the games to PLAY, and the loop jumps from one set bit to the next: a skipped game costs nothing.
    const bool use_census = CENSUS && (p.census != nullptr);
    const bool frozen_rest = census_frozen_rest(kops, kflags);
    const uint32_t rows_k = CENSUS ? (uint32_t)p.rows_k : 0u;
    auto skip_game = [&](uint32_t v) -> bool {
        return census_at_rest(v, frozen_rest) || (rows_k && v != 0 && census_live_count(v) <= rows_k);
    };
    // census mask of the game just stepped: bit i <=> row i alive (N <= 64)
    auto store_mask = [&](long long gg, uint32_t lo, uint32_t hi) {
        if (p.live_mask && lane == 0) p.live_mask[gg] = ((uint64_t)hi << 32) | lo;
    };
    // finished-game counts: lane l accumulates the games finished after steps l and l + 32 and flushes them
    // once, instead of one same-address atomic per game and step
    int dc0 = 0, dc1 = 0;
    auto count_done = [&](int st) {
        if (st < 32) dc0 += (lane == st) ? 1 : 0;
        else if (st < 64) dc1 += (lane == st - 32) ? 1 : 0;
        else if (lane == 0) atomicAdd(p.done_count + st, 1);
    };
    const long long n_it = (CENSUS && p.B > gw) ? (p.B - gw + nw - 1) / nw : 0;  // iterations of this warp
    // one batch of census bytes: the lane's byte, the play mask, and the outputs of the batch's games at rest
    // (when no hk_rows_kernel ran before: it writes them otherwise)
    auto census_batch = [&](long long it0, uint32_t& cv) -> uint32_t {
        const long long itl = it0 + lane;
        const bool exists = itl < n_it;
        const long long gg = gw + itl * nw;
        cv = (use_census && exists) ? (uint32_t)__ldg(p.census + gg) : 0u;
        if (use_census && !rows_k) {
            const bool rest = exists && census_at_rest(cv, frozen_rest);
            if (rest) {
                write_rest_outputs(p, gg, cv, rest_reward(kflags));
                if (p.done_bits) atomicOr(p.done_bits + (gg >> 5), 1u << (gg & 31));
            }
            if (p.done_count) {
                const int n = __popc(__ballot_sync(0xffffffffu, rest));
                dc0 += (lane == 0) ? n : 0;
            }
        }
        return __ballot_sync(0xffffffffu, exists && !(use_census && skip_game(cv)));
    };
    long long cbase = 0;
    uint32_t cv_cur = 0, cv_nxt = 0;
    uint32_t pm_cur = CENSUS ? census_batch(0, cv_cur) : 0u, pm_nxt = CENSUS ? census_batch(32, cv_nxt) : 0u;
    constexpr long long IT_END = -1;
    // the first iteration to play at or after `from` (which lies in [cbase, cbase + 64]), IT_END if none is left
    auto next_play = [&](long long from) -> long long {
        for (;;) {
            int o = (int)(from - cbase);
            if (o < 32) {
                const uint32_t m = pm_cur & (0xffffffffu << o);
                if (m) return cbase + (__ffs((int)m) - 1);
                o = 32;
            }
            if (o < 64) {
                const uint32_t m = pm_nxt & (0xffffffffu << (o - 32));
                if (m) return cbase + 32 + (__ffs((int)m) - 1);
            }
            if (cbase + 64 >= n_it) return IT_END;
            cbase += 32;  // nothing left in the older batch: bring in the next one
            cv_cur = cv_nxt;
            pm_cur = pm_nxt;
            pm_nxt = census_batch(cbase + 32, cv_nxt);
            from = cbase + 32;
        }
    };

    int b = 0;
    int32_t ha_nx = 3, ax_nx = 0;
    // the loop runs over game indices; -1 ends it.  Without a census the next game is simply g + nw.
    long long it = CENSUS ? next_play(0) : 0;
    long long g = CENSUS ? (it == IT_END ? -1 : gw + it * nw) : (gw < p.B ? gw : -1);
    long long g_nx = -1;
    if (g >= 0) {
        if (kops & HK_OP_SHIFT) load_actions(p, kflags, g, 0, ha_nx, ax_nx);
        prefetch(g, 0);
    }
    cp_async_commit();
    for (; g >= 0; g = g_nx, b = (b + 1 == NBUF) ? 0 : b + 1) {
        if constexpr (CENSUS) {
            it = next_play(it + 1);
            g_nx = (it == IT_END) ? -1 : gw + it * nw;
        } else {
            g_nx = (g + nw < p.B) ? g + nw : -1;
        }
        {   // the buffer that held the previous game is free: the next game to play goes there
            const int bn = (b + 1 >= NBUF) ? b + 1 - NBUF : b + 1;
            if (g_nx >= 0) prefetch(g_nx, bn);
        }
        cp_async_commit();  // one group per iteration (possibly empty) keeps the wait count uniform
        // this game's actions were requested one iteration ago (a dependent global load per game would
        // otherwise sit on the critical path of the short iterations); request the next game's now
        int32_t ha = ha_nx, ax = ax_nx;
        if ((kops & HK_OP_SHIFT) && g_nx >= 0) {
            load_actions(p, kflags, g_nx, 0, ha_nx, ax_nx);
        }
        cp_async_wait<1>();  // everything but the newest group has landed: game g is in buffer b
        __syncwarp();
        T* x = reinterpret_cast<T*>(slot + b * Wpad);

        // Did the game change?  An unchanged game of an in-place call is not written back (in a long
        // rollout most games have ended and sit at a fixed point); everything is when out != in.
        bool chg = !inplace;

        // ---- liveness ----
        uint32_t mylive = 0;  // bit r <=> row lane + 32 r is live
        int cnt = 0;
        _Pragma("unroll UNR")
        for (int r = 0; r < R; ++r) {
            const int i = lane + 32 * r;
            bool lv = false;
            if (i < N) {
                if constexpr (Elem<T>::is_float) {
#pragma unroll
                    for (int k = 0; k < D; ++k) {  // canonicalise -0.0 (a game that held one counts as changed)
                        const float v = x[i * D + k], c = v + 0.0f;
                        chg = chg || (__float_as_int(v) != __float_as_int(c));
                        x[i * D + k] = c;
                    }
                }
                lv = x[i * D] >= Elem<T>::zero();
            }
            cnt += __popc(__ballot_sync(0xffffffffu, lv));
            mylive |= lv ? (1u << r) : 0u;
        }
        int32_t over = kT + 1;  // (THR) the crossing step, kT + 1 while the game stays below the threshold
        if constexpr (THR) {
            bool e = false;
            _Pragma("unroll UNR")
            for (int r = 0; r < R; ++r) {
                const int i = lane + 32 * r;
                if (i >= N || !((mylive >> r) & 1u)) continue;
#pragma unroll
                for (int k = 0; k < D; ++k) e = e || (Elem<T>::to_float(x[i * D + k]) >= p.threshold);
            }
            if (__any_sync(0xffffffffu, e)) over = 0;
        }
        // ---- ended games, single step: a short path of their own ----
        // Most games of a long rollout have at most one live row; nothing of the machinery below
        // (ballot rounds, the step loop, the filter) applies to them.  The lone row's lane plays the
        // step, lane 0 writes the outputs (done before the step: no reward), and the state is stored
        // only if the row moved or a dead row needed normalising.
        if (cnt <= 1 && ended_fast_path) {
            bool exceed = false;
            _Pragma("unroll UNR")
            for (int r = 0; r < R; ++r) {
                const int i = lane + 32 * r;
                if (i >= N) continue;
                if ((mylive >> r) & 1u) {
                    T v[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) v[k] = x[i * D + k];
                    if (kops & HK_OP_SHIFT) {
                        const uint32_t cm = action_mask(ha, kflags);
                        bool apply = (ax >= 0) && (ax < D) && !(kflags & HK_F_FREEZE_ENDED);
                        if (kflags & HK_F_NOOP_INVALID) apply = apply && ((cm >> (ax & 31)) & 1u);
                        T s = Elem<T>::zero();
#pragma unroll
                        for (int k = 0; k < D; ++k) s = ((cm >> k) & 1u) ? s + v[k] : s;
#pragma unroll
                        for (int k = 0; k < D; ++k) v[k] = (apply && k == ax) ? s : v[k];
                    }
                    if (kops & HK_OP_REPOSITION) {  // a lone point minus its own coordinates
#pragma unroll
                        for (int k = 0; k < D; ++k) v[k] = Elem<T>::zero();
                    }
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        chg = chg || (Elem<T>::bits(v[k]) != Elem<T>::bits(x[i * D + k]));
                        x[i * D + k] = v[k];
                    }
                    if (p.exceed_flag) {
#pragma unroll
                        for (int k = 0; k < D; ++k) exceed = exceed || (Elem<T>::to_float(v[k]) >= p.threshold);
                    }
                } else if (kops) {
                    uint32_t bad = 0;
#pragma unroll
                    for (int k = 0; k < D; ++k) bad |= (uint32_t)Elem<T>::bits(x[i * D + k]) ^ (uint32_t)Elem<T>::bits(padv);
                    if (bad) {
                        chg = true;
#pragma unroll
                        for (int k = 0; k < D; ++k) x[i * D + k] = padv;
                    }
                }
            }
            if (lane == 0) {
                if (p.done) p.done[g] = 1;
                if (p.reward) p.reward[g] = rest_reward(kflags);
                if (p.num_points) p.num_points[g] = cnt;
                if (p.length) p.length[g] = 0;
                if (CENSUS && p.done_bits) atomicOr(p.done_bits + (g >> 5), 1u << (g & 31));
            }
            if (p.done_count) count_done(0);
            if (use_census) {  // (dead rows are normalised by now: kops != 0 on the census path)
                bool moving = false;  // a live row away from the origin
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    const int i = lane + 32 * r;
                    if (i < N && ((mylive >> r) & 1u)) {
#pragma unroll
                        for (int k = 0; k < D; ++k) moving = moving || (Elem<T>::bits(x[i * D + k]) != 0);
                    }
                }
                const bool org = !__any_sync(0xffffffffu, moving);
                if (lane == 0) p.census[g] = census_after_step(cnt, org);
                if (p.live_mask)
                    store_mask(g, __ballot_sync(0xffffffffu, mylive & 1u), __ballot_sync(0xffffffffu, (mylive >> 1) & 1u));
            }
            if (p.exceed_flag) {
                if (__any_sync(0xffffffffu, exceed) && lane == 0) *p.exceed_flag = 1;
            }
            __syncwarp();
            if (gout && __any_sync(0xffffffffu, chg)) {
                const uint32_t* src = slot + b * Wpad;
                uint32_t* dst = gout + g * W;
                if (vec_out) {
                    for (int c = lane; c < (W >> 2); c += 32)
                        reinterpret_cast<uint4*>(dst)[c] = reinterpret_cast<const uint4*>(src)[c];
                } else {
                    for (int w = lane; w < W; w += 32) dst[w] = src[w];
                }
            }
            __syncwarp();  // every lane is done with buffer b before the next prefetch may overwrite it
            continue;
        }
        // ---- games with 2 .. 32 live rows: one COMPACT row per lane, for one step or a whole rollout ----
        // The general path below keeps the padded layout (lane l owns rows l, l+32, ...) and pays for it
        // with ballot rounds and row loops in every op: ~1 200 warp-instructions for a three-point
        // game.  Here the live rows are compacted first (the list the filter needs anyway), lane v
        // takes compact row v and keeps it in registers for all T steps, and the survivors go back to
        // their slots at the end: ~150 + 12 per live row and step.  Rows that die stay parked at +BIG
        // in the compact list, so the list is built once per game.
        if (cnt >= 2 && cnt <= 32 && compact_path) {
            int base = 0;
            _Pragma("unroll UNR")
            for (int r = 0; r < R; ++r) {
                const bool lv = (mylive >> r) & 1u;
                const uint32_t bal = __ballot_sync(0xffffffffu, lv);
                if (lv) {
                    const int i = lane + 32 * r;
                    uint32_t* dst = comp + (base + __popc(bal & ((1u << lane) - 1u))) * CSTRIDE;
#pragma unroll
                    for (int k = 0; k < D; ++k) dst[k] = (uint32_t)Elem<T>::bits(x[i * D + k]);
                    dst[D] = (uint32_t)i;
                }
                base += __popc(bal);
            }
            __syncwarp();
            int ccnt = cnt;  // rows in the compact list (a long rollout rebuilds it as rows die)
            bool act = lane < ccnt;
            T v[D], v0[D];
#pragma unroll
            for (int k = 0; k < D; ++k) {
                v[k] = act ? Elem<T>::from_bits(comp[lane * CSTRIDE + k]) : Elem<T>::big();
                v0[k] = v[k];
            }
            int myslot = act ? (int)comp[lane * CSTRIDE + D] : 0;
            bool rebuilt = false;  // after a rebuild v0 no longer belongs to this lane's row: rows are written back regardless
            if ((ccnt & 1) && lane <= D) comp[ccnt * CSTRIDE + lane] = (uint32_t)Elem<T>::bits(Elem<T>::big());  // pad row: dominates nothing
            uint32_t live = (ccnt >= 32) ? 0xffffffffu : ((1u << ccnt) - 1u);
            int cur = cnt;
            int32_t len = kT + 1;
            int npairs = (ccnt + 1) >> 1;
            for (int st = 0; st < kT; ++st) {
                if constexpr (THR) {
                    if (p.stop_at_threshold && over <= st) {  // stopped at the threshold: the game sits out the step
                        const bool dn = cur < 2;
                        if (lane == 0) {
                            if (p.done) p.done[(long long)st * p.B + g] = dn ? 1 : 0;
                            if (p.reward) p.reward[(long long)st * p.B + g] = rest_reward(kflags);
                        }
                        if (p.done_count && dn) count_done(st);
                        continue;
                    }
                }
                if (st > 0 && cur >= 2 && 2 * cur <= ccnt) {
                    // Half of the listed rows have died: rebuild the list from the survivors so that the
                    // filter's cost keeps following the live count.  Rows that died go back to their slots
                    // as padding now; survivors move to the lanes below `cur`.
                    const bool alive_now = (live >> lane) & 1u;
                    __syncwarp();
                    if (act && !alive_now) {
#pragma unroll
                        for (int k = 0; k < D; ++k) x[myslot * D + k] = padv;
                    }
                    if (alive_now) {
                        uint32_t* dst = comp + __popc(live & ((1u << lane) - 1u)) * CSTRIDE;
#pragma unroll
                        for (int k = 0; k < D; ++k) dst[k] = (uint32_t)Elem<T>::bits(v[k]);
                        dst[D] = (uint32_t)myslot;
                    }
                    __syncwarp();
                    ccnt = cur;
                    act = lane < ccnt;
#pragma unroll
                    for (int k = 0; k < D; ++k) v[k] = act ? Elem<T>::from_bits(comp[lane * CSTRIDE + k]) : Elem<T>::big();
                    myslot = act ? (int)comp[lane * CSTRIDE + D] : 0;
                    __syncwarp();
                    if ((ccnt & 1) && lane <= D) comp[ccnt * CSTRIDE + lane] = (uint32_t)Elem<T>::bits(Elem<T>::big());
                    live = (1u << ccnt) - 1u;  // (ccnt <= 16 here)
                    npairs = (ccnt + 1) >> 1;
                    rebuilt = true;
                    chg = true;
                }
                int32_t ha_n = 3, ax_n = 0;
                if ((kops & HK_OP_SHIFT) && st + 1 < kT) load_actions(p, kflags, g, st + 1, ha_n, ax_n);
                const bool prev_done = cur < 2;
                const bool alive0 = (live >> lane) & 1u;
                if ((kops & HK_OP_SHIFT) && cur > 0) {
                    const uint32_t cm = action_mask(ha, kflags);
                    bool apply = (ax >= 0) && (ax < D);
                    if (kflags & HK_F_NOOP_INVALID) apply = apply && ((cm >> (ax & 31)) & 1u);
                    if (kflags & HK_F_FREEZE_ENDED) apply = apply && !prev_done;
                    if (apply && alive0) {
                        T s = Elem<T>::zero();
#pragma unroll
                        for (int k = 0; k < D; ++k) s = ((cm >> k) & 1u) ? s + v[k] : s;
#pragma unroll
                        for (int k = 0; k < D; ++k) v[k] = (k == ax) ? s : v[k];
                    }
                }
                if ((kops & HK_OP_REPOSITION) && cur > 0) {
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        const T mn = warp_min<T>(alive0 ? v[k] : Elem<T>::big());
                        v[k] = alive0 ? v[k] - mn : v[k];
                    }
                }
                if ((kops & HK_OP_NEWTON) && cur >= 2) {
                    __syncwarp();
                    if (act) {  // rows that have died are parked at +BIG: they dominate nothing
#pragma unroll
                        for (int k = 0; k < D; ++k)
                            comp[lane * CSTRIDE + k] = (uint32_t)Elem<T>::bits(alive0 ? v[k] : Elem<T>::big());
                    }
                    __syncwarp();
                    int32_t acc = (int32_t)0x80000000;
                    for (int pr = 0; pr < npairs; ++pr) {  // two dominators per trip, 16-byte broadcast loads
                        uint32_t w[2 * CSTRIDE];
                        const uint4* src = reinterpret_cast<const uint4*>(comp + pr * 2 * CSTRIDE);
#pragma unroll
                        for (int q = 0; q < CSTRIDE / 2; ++q) {
                            const uint4 u = src[q];
                            w[4 * q] = u.x, w[4 * q + 1] = u.y, w[4 * q + 2] = u.z, w[4 * q + 3] = u.w;
                        }
                        int32_t ta = 0, tb = 0;
#pragma unroll
                        for (int k = 0; k < D; ++k) {
                            ta |= Elem<T>::bits(v[k] - Elem<T>::from_bits(w[k]));
                            tb |= Elem<T>::bits(v[k] - Elem<T>::from_bits(w[CSTRIDE + k]));
                        }
                        // compact order is slot order: ties only kill from a lower position (also neutralises the
                        // self pair)
                        acc &= (ta - ((2 * pr >= lane) ? 1 : 0)) & (tb - ((2 * pr + 1 >= lane) ? 1 : 0));
                    }
                    live = __ballot_sync(0xffffffffu, alive0 && (acc < 0));
                }
                const bool alive = (live >> lane) & 1u;
                if constexpr (Elem<T>::is_float) {
                    if (kops & HK_OP_RESCALE) {
                        float mx = -1.0f;
#pragma unroll
                        for (int k = 0; k < D; ++k) mx = alive ? fmaxf(mx, v[k]) : mx;
                        mx = warp_maxf(mx);
                        if (mx == 0.0f || ((kflags & HK_F_RESCALE_EPS) && mx > 0.0f && mx <= 1e-8f)) mx = 1.0f;
                        if (mx > 0.0f && alive) {
#pragma unroll
                            for (int k = 0; k < D; ++k) v[k] = (v[k] != 0.0f) ? __fdiv_rn(v[k], mx) : v[k];
                        }
                    }
                }
                cur = __popc(live);
                const bool dn = cur < 2;
                if (lane == 0) {
                    if (p.done) p.done[(long long)st * p.B + g] = dn ? 1 : 0;
                    if (CENSUS && p.done_bits && dn) atomicOr(p.done_bits + (g >> 5), 1u << (g & 31));
                    if (p.reward) p.reward[(long long)st * p.B + g] = step_reward(kflags, dn, prev_done);
                }
                if (p.done_count && dn) count_done(st);
                if (dn && !prev_done) len = st + 1;
                if constexpr (THR) {
                    if (over > kT) {
                        bool e = false;
                        if (alive) {
#pragma unroll
                            for (int k = 0; k < D; ++k) e = e || (Elem<T>::to_float(v[k]) >= p.threshold);
                        }
                        if (__any_sync(0xffffffffu, e)) over = st + 1;
                    }
                }
                ha = ha_n;
                ax = ax_n;
            }
            if (use_census) {
                bool moving = false;
                if ((live >> lane) & 1u) {
#pragma unroll
                    for (int k = 0; k < D; ++k) moving = moving || (Elem<T>::bits(v[k]) != 0);
                }
                const bool org = !__any_sync(0xffffffffu, moving);
                if (lane == 0) p.census[g] = census_after_step(cur, org);
                if (p.live_mask) {
                    const bool al = (live >> lane) & 1u;
                    const uint32_t lo = __reduce_or_sync(0xffffffffu, (al && myslot < 32) ? (1u << myslot) : 0u);
                    const uint32_t hi = __reduce_or_sync(0xffffffffu, (al && myslot >= 32 && myslot < 64) ? (1u << (myslot - 32)) : 0u);
                    store_mask(g, lo, hi);
                }
            }
            // survivors and killed rows go back to their slots of the padded game
            const bool alive = (live >> lane) & 1u;
            bool exceed = false;
            if (act) {
                bool rowchg = !alive || rebuilt;
#pragma unroll
                for (int k = 0; k < D; ++k) rowchg = rowchg || (Elem<T>::bits(v[k]) != Elem<T>::bits(v0[k]));
                if (rowchg) {
                    chg = true;
#pragma unroll
                    for (int k = 0; k < D; ++k) x[myslot * D + k] = alive ? v[k] : padv;
                }
            }
            if (alive && p.exceed_flag) {
#pragma unroll
                for (int k = 0; k < D; ++k) exceed = exceed || (Elem<T>::to_float(v[k]) >= p.threshold);
            }
            if (kops) {  // dead rows that do not hold the padding value are normalised, as every reference op does
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    const int i = lane + 32 * r;
                    if (i >= N || ((mylive >> r) & 1u)) continue;
                    uint32_t bad = 0;
#pragma unroll
                    for (int k = 0; k < D; ++k) bad |= (uint32_t)Elem<T>::bits(x[i * D + k]) ^ (uint32_t)Elem<T>::bits(padv);
                    if (bad) {
                        chg = true;
#pragma unroll
                        for (int k = 0; k < D; ++k) x[i * D + k] = padv;
                    }
                }
            }
            if (lane == 0) {
                if (p.num_points) p.num_points[g] = cur;
                if (p.length) p.length[g] = len;
                if constexpr (THR) {
                    if (p.over_step) p.over_step[g] = over;
                }
            }
            if (p.exceed_flag) {
                if (__any_sync(0xffffffffu, exceed) && lane == 0) *p.exceed_flag = 1;
            }
            __syncwarp();
            if (gout && __any_sync(0xffffffffu, chg)) {
                const uint32_t* src = slot + b * Wpad;
                uint32_t* dst = gout + g * W;
                if (vec_out) {
                    for (int c = lane; c < (W >> 2); c += 32)
                        reinterpret_cast<uint4*>(dst)[c] = reinterpret_cast<const uint4*>(src)[c];
                } else {
                    for (int w = lane; w < W; w += 32) dst[w] = src[w];
                }
            }
            __syncwarp();  // every lane is done with buffer b before the next prefetch may overwrite it
            continue;
        }
        int32_t len = (cnt < 2) ? 0 : kT + 1;
        for (int st = 0; st < kT; ++st) {
            float* gobs_t = nullptr;
            if constexpr (REC) {
                if (p.obs_t) {
                    gobs_t = p.obs_t + ((long long)st * p.B + g) * OW;
                    generic_features<T, D, RT>(x, mylive, f, gobs_t, N, R, lane, kflags, p.pad);
                }
            }
            if constexpr (THR) {
                if (p.stop_at_threshold && over <= st) {  // stopped at the threshold: the game sits out the step
                    const bool dn = cnt < 2;
                    if (lane == 0) {
                        if (p.done) p.done[(long long)st * p.B + g] = dn ? 1 : 0;
                        if (p.reward) p.reward[(long long)st * p.B + g] = rest_reward(kflags);
                        if constexpr (REC) {
                            const long long o = (long long)st * p.B + g;
                            if (p.host_mask_t) p.host_mask_t[o] = 0;
                            if (p.axis_played_t) p.axis_played_t[o] = -1;
                        }
                    }
                    if constexpr (REC) {
                        if (gobs_t && p.agent_obs && lane < D) gobs_t[W + lane] = 0.0f;
                    }
                    if (p.done_count && dn) count_done(st);
                    __syncwarp();
                    continue;
                }
            }
            int32_t ha_n = 3, ax_n = 0;
            if ((kops & HK_OP_SHIFT) && st + 1 < kT) {
                load_actions(p, kflags, g, st + 1, ha_n, ax_n);
            }
            const bool prev_done = cnt < 2;

            // ---- shift ----
            if ((kops & HK_OP_SHIFT) && cnt == 0 && p.host_out && lane == 0) p.host_out[g] = 0;
            uint32_t played_cm = 0, played_ax = 0;  // (REC) what the shift used, 0 without one
            if constexpr (REC) {
                if ((kops & HK_OP_SHIFT) && cnt == 0) {  // nothing moves; the players answer as on any other game
                    const uint32_t cm = (kflags & HK_F_HOST_ALL_COORD) ? ((1u << D) - 1u)
                                        : (kflags & HK_F_HOST_ZEILLINGER) ? decode_host_action(0) : action_mask(ha, kflags);
                    played_cm = (kflags & (HK_F_HOST_ALL_COORD | HK_F_HOST_ZEILLINGER)) ? 0u : cm;
                    played_ax = (uint32_t)agent_policy_axis(cm, ax, kflags, D);
                }
            }
            if ((kops & HK_OP_SHIFT) && cnt > 0) {
                uint32_t cm;
                if (kflags & HK_F_HOST_ALL_COORD) {
                    cm = (1u << D) - 1u;
                } else if (kflags & HK_F_HOST_ZEILLINGER) {
                    // Zeillinger's host, lane-parallel: every lane scans the pairs (i, j) of its own rows i,
                    // then a lexicographic (L, S, flat index) minimum is reduced over the warp
                    _Pragma("unroll UNR")
                    for (int r = 0; r < R; ++r) {
                        const uint32_t bal = __ballot_sync(0xffffffffu, (mylive >> r) & 1u);
                        if (lane == 0) lmw[r] = bal;
                    }
                    __syncwarp();
                    ZeilBest zb;
                    zb.L = __int_as_float(0x7f800000);
                    zb.S = zb.L;
                    zb.i = -1;
                    zb.j = -1;
                    _Pragma("unroll UNR")
                    for (int r = 0; r < R; ++r) {
                        if (!((mylive >> r) & 1u)) continue;
                        const int i = lane + 32 * r;
                        float vi[D];
#pragma unroll
                        for (int k = 0; k < D; ++k) vi[k] = Elem<T>::to_float(x[i * D + k]);
                        for (int r2 = 0; r2 < R; ++r2) {
                            uint32_t m = lmw[r2];
                            while (m) {
                                const int j = 32 * r2 + __ffs((int)m) - 1;
                                m &= m - 1;
                                float vj[D];
#pragma unroll
                                for (int k = 0; k < D; ++k) vj[k] = Elem<T>::to_float(x[j * D + k]);
                                zeillinger_consider<D>(zb, vi, vj, i, j);
                            }
                        }
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) {
                        const float L2 = __shfl_xor_sync(0xffffffffu, zb.L, o);
                        const float S2 = __shfl_xor_sync(0xffffffffu, zb.S, o);
                        const int i2 = __shfl_xor_sync(0xffffffffu, zb.i, o);
                        const int j2 = __shfl_xor_sync(0xffffffffu, zb.j, o);
                        const long long f1 = (long long)zb.i * N + zb.j, f2 = (long long)i2 * N + j2;
                        const bool take = (i2 >= 0) && ((zb.i < 0) || (L2 < zb.L) || (L2 == zb.L && (S2 < zb.S || (S2 == zb.S && f2 < f1))));
                        zb.L = take ? L2 : zb.L;
                        zb.S = take ? S2 : zb.S;
                        zb.i = take ? i2 : zb.i;
                        zb.j = take ? j2 : zb.j;
                    }
                    const bool found = zb.i >= 0;
                    float vi[D], vj[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        vi[k] = found ? Elem<T>::to_float(x[zb.i * D + k]) : 0.0f;
                        vj[k] = found ? Elem<T>::to_float(x[zb.j * D + k]) : 0.0f;
                    }
                    cm = zeillinger_mask_from_diff<D>(vi, vj, found);
                    __syncwarp();
                } else {
                    cm = action_mask(ha, kflags);
                }
                ax = agent_policy_axis(cm, ax, kflags, D);
                if constexpr (REC) {
                    played_cm = cm;
                    played_ax = (uint32_t)ax;
                }
                bool apply = (ax >= 0) && (ax < D);
                if (p.host_out) {  // hk_host_policy: report the host's choice, move nothing
                    if (lane == 0) p.host_out[g] = (int32_t)cm;
                    apply = false;
                }
                if (kflags & HK_F_NOOP_INVALID) apply = apply && ((cm >> (ax & 31)) & 1u);
                if (kflags & HK_F_FREEZE_ENDED) apply = apply && !prev_done;
                if (apply) {
                    _Pragma("unroll UNR")
                    for (int r = 0; r < R; ++r) {
                        if (!((mylive >> r) & 1u)) continue;
                        const int i = lane + 32 * r;
                        T s = Elem<T>::zero();
#pragma unroll
                        for (int k = 0; k < D; ++k) s = ((cm >> k) & 1u) ? s + x[i * D + k] : s;
                        chg = chg || (x[i * D + ax] != s);
                        x[i * D + ax] = s;
                    }
                }
            }
            if constexpr (REC) {
                if (lane == 0) {
                    const long long o = (long long)st * p.B + g;
                    if (p.host_mask_t) p.host_mask_t[o] = (int32_t)played_cm;
                    if (p.axis_played_t) p.axis_played_t[o] = (int32_t)played_ax;
                }
                if (gobs_t && p.agent_obs && lane < D) gobs_t[W + lane] = (float)((played_cm >> lane) & 1u);
            }
            // ---- reposition ----
            if ((kops & HK_OP_REPOSITION) && cnt == 1) {
                // a lone point minus its own coordinates: the origin (most games of a long rollout are here)
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    if (!((mylive >> r) & 1u)) continue;
                    const int i = lane + 32 * r;
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        chg = chg || (x[i * D + k] != Elem<T>::zero());
                        x[i * D + k] = Elem<T>::zero();
                    }
                }
            } else if ((kops & HK_OP_REPOSITION) && cnt > 1) {
                T mn[D];
#pragma unroll
                for (int k = 0; k < D; ++k) mn[k] = Elem<T>::big();
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    if (!((mylive >> r) & 1u)) continue;
                    const int i = lane + 32 * r;
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        const T v = x[i * D + k];
                        mn[k] = v < mn[k] ? v : mn[k];
                    }
                }
#pragma unroll
                for (int k = 0; k < D; ++k) {
                    mn[k] = warp_min<T>(mn[k]);
                    chg = chg || (mn[k] != Elem<T>::zero());
                }
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    if (!((mylive >> r) & 1u)) continue;
                    const int i = lane + 32 * r;
#pragma unroll
                    for (int k = 0; k < D; ++k) x[i * D + k] -= mn[k];
                }
            }
            // ---- dedupe alone (remove_repeated _fn.py:192-213) ----
            if ((kops & HK_OP_DEDUPE) && cnt >= 2) {
                // A row that died in an earlier step of a rollout still holds its old values in the slot (dead rows
                // are padded on the way out): whether row j is live comes from the warp's live masks, not its data.
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    const uint32_t bal = __ballot_sync(0xffffffffu, (mylive >> r) & 1u);
                    if (lane == 0) lmw[r] = bal;
                }
                __syncwarp();
                uint32_t kill = 0;
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    if (!((mylive >> r) & 1u)) continue;
                    const int i = lane + 32 * r;
                    bool rep = false;
                    for (int j = 0; j < i; ++j) {
                        bool eq = (lmw[j >> 5] >> (j & 31)) & 1u;
#pragma unroll
                        for (int k = 0; k < D; ++k) eq = eq && (x[i * D + k] == x[j * D + k]);
                        rep = rep || eq;
                    }
                    kill |= rep ? (1u << r) : 0u;
                }
                __syncwarp();
                chg = chg || (kill != 0);
                mylive &= ~kill;
            }
            // ---- newton: dedupe + dominance, reading the pre-removal state ----
            if ((kops & HK_OP_NEWTON) && cnt >= 2) {
                // The live rows are first copied, in slot order, into a COMPACT list in shared memory (row k at
                // k*CSTRIDE: D coordinates, then the slot number), so that the dominator loop walks it linearly
                // with 16-byte broadcast loads, two dominators per trip, instead of decoding ballot words into row
                // addresses on every trip (that bookkeeping and the scalar loads were half of the loop's
                // instructions).  An odd count is padded with a copy of the last row: AND-accumulation is idempotent.
                int base = 0;
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    const bool lv = (mylive >> r) & 1u;
                    const uint32_t bal = __ballot_sync(0xffffffffu, lv);
                    if (lv) {
                        const int i = lane + 32 * r;
                        uint32_t* dst = comp + (base + __popc(bal & ((1u << lane) - 1u))) * CSTRIDE;
#pragma unroll
                        for (int k = 0; k < D; ++k) dst[k] = (uint32_t)Elem<T>::bits(x[i * D + k]);
                        dst[D] = (uint32_t)i;
                    }
                    base += __popc(bal);
                }
                __syncwarp();
                if ((base & 1) && lane <= D) comp[base * CSTRIDE + lane] = comp[(base - 1) * CSTRIDE + lane];
                __syncwarp();
                const int npairs = (base + 1) >> 1;
                uint32_t kill = 0;
                auto load_pair = [&](int pr, T (&xa)[D], T (&xb)[D], int& ja, int& jb) {
                    uint32_t w[2 * CSTRIDE];
                    const uint4* src = reinterpret_cast<const uint4*>(comp + pr * 2 * CSTRIDE);
#pragma unroll
                    for (int q = 0; q < CSTRIDE / 2; ++q) {
                        const uint4 v = src[q];
                        w[4 * q] = v.x, w[4 * q + 1] = v.y, w[4 * q + 2] = v.z, w[4 * q + 3] = v.w;
                    }
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        xa[k] = Elem<T>::from_bits(w[k]);
                        xb[k] = Elem<T>::from_bits(w[CSTRIDE + k]);
                    }
                    ja = (int)w[D];
                    jb = (int)w[CSTRIDE + D];
                };
                if (R <= 2) {
                    // both rows of the lane ride on the same broadcast of the dominator pair
                    const int i0 = lane, i1 = lane + 32;
                    const bool l0 = mylive & 1u, l1 = (mylive >> 1) & 1u;
                    T a0[D], a1[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        a0[k] = l0 ? x[i0 * D + k] : Elem<T>::big();
                        a1[k] = l1 ? x[i1 * D + k] : Elem<T>::big();
                    }
                    int32_t acc0 = (int32_t)0x80000000, acc1 = (int32_t)0x80000000;
                    for (int pr = 0; pr < npairs; ++pr) {
                        T xa[D], xb[D];
                        int ja, jb;
                        load_pair(pr, xa, xb, ja, jb);
                        int32_t t0a = Elem<T>::bits(a0[0] - xa[0]), t1a = Elem<T>::bits(a1[0] - xa[0]);
                        int32_t t0b = Elem<T>::bits(a0[0] - xb[0]), t1b = Elem<T>::bits(a1[0] - xb[0]);
#pragma unroll
                        for (int k = 1; k < D; ++k) {
                            t0a |= Elem<T>::bits(a0[k] - xa[k]);
                            t1a |= Elem<T>::bits(a1[k] - xa[k]);
                            t0b |= Elem<T>::bits(a0[k] - xb[k]);
                            t1b |= Elem<T>::bits(a1[k] - xb[k]);
                        }
                        // ties only kill from a lower slot; this also neutralises the self pair
                        acc0 &= (t0a - ((ja >= i0) ? 1 : 0)) & (t0b - ((jb >= i0) ? 1 : 0));
                        acc1 &= (t1a - ((ja >= i1) ? 1 : 0)) & (t1b - ((jb >= i1) ? 1 : 0));
                    }
                    kill = ((acc0 >= 0) ? 1u : 0u) | ((acc1 >= 0) ? 2u : 0u);
                } else {
                    _Pragma("unroll UNR")
                    for (int r = 0; r < R; ++r) {
                        const int i = lane + 32 * r;
                        const bool lv = (mylive >> r) & 1u;
                        T xi[D];
#pragma unroll
                        for (int k = 0; k < D; ++k) xi[k] = lv ? x[i * D + k] : Elem<T>::big();
                        int32_t acc = (int32_t)0x80000000;
                        for (int pr = 0; pr < npairs; ++pr) {
                            T xa[D], xb[D];
                            int ja, jb;
                            load_pair(pr, xa, xb, ja, jb);
                            int32_t ta = Elem<T>::bits(xi[0] - xa[0]), tb = Elem<T>::bits(xi[0] - xb[0]);
#pragma unroll
                            for (int k = 1; k < D; ++k) {
                                ta |= Elem<T>::bits(xi[k] - xa[k]);
                                tb |= Elem<T>::bits(xi[k] - xb[k]);
                            }
                            acc &= (ta - ((ja >= i) ? 1 : 0)) & (tb - ((jb >= i) ? 1 : 0));
                        }
                        kill |= (acc >= 0) ? (1u << r) : 0u;
                    }
                }
                __syncwarp();
                chg = chg || (kill != 0);
                mylive &= ~kill;
            }
            // ---- rescale (float state) ----
            if constexpr (Elem<T>::is_float) {
                if (kops & HK_OP_RESCALE) {
                    float mx = -1.0f;
                    _Pragma("unroll UNR")
                    for (int r = 0; r < R; ++r) {
                        if (!((mylive >> r) & 1u)) continue;
                        const int i = lane + 32 * r;
#pragma unroll
                        for (int k = 0; k < D; ++k) mx = fmaxf(mx, x[i * D + k]);
                    }
                    mx = warp_maxf(mx);
                    if (mx == 0.0f || ((kflags & HK_F_RESCALE_EPS) && mx > 0.0f && mx <= 1e-8f)) mx = 1.0f;
                    if (mx > 0.0f) {
                        _Pragma("unroll UNR")
                        for (int r = 0; r < R; ++r) {
                            if (!((mylive >> r) & 1u)) continue;
                            const int i = lane + 32 * r;
#pragma unroll
                            for (int k = 0; k < D; ++k) {
                                const float v = x[i * D + k];  // 0 / mx = 0: keep zeros (common after reposition) out of the divider
                                const float q = (v != 0.0f) ? __fdiv_rn(v, mx) : v;
                                chg = chg || (q != v);
                                x[i * D + k] = q;
                            }
                        }
                    }
                }
            }
            // ---- per-step outputs ----
            cnt = 0;
            _Pragma("unroll UNR")
            for (int r = 0; r < R; ++r) cnt += __popc(__ballot_sync(0xffffffffu, (mylive >> r) & 1u));
            const bool dn = cnt < 2;
            if (lane == 0) {
                if (p.done) p.done[(long long)st * p.B + g] = dn ? 1 : 0;
                if (CENSUS && p.done_bits && dn) atomicOr(p.done_bits + (g >> 5), 1u << (g & 31));
                if (p.reward) p.reward[(long long)st * p.B + g] = step_reward(kflags, dn, prev_done);
            }
            if (p.done_count && dn) count_done(st);
            if (dn && !prev_done) len = st + 1;
            if constexpr (THR) {
                if (over > kT) {
                    bool e = false;
                    _Pragma("unroll UNR")
                    for (int r = 0; r < R; ++r) {
                        const int i = lane + 32 * r;
                        if (i >= N || !((mylive >> r) & 1u)) continue;
#pragma unroll
                        for (int k = 0; k < D; ++k) e = e || (Elem<T>::to_float(x[i * D + k]) >= p.threshold);
                    }
                    if (__any_sync(0xffffffffu, e)) over = st + 1;
                }
            }
            ha = ha_n;
            ax = ax_n;
            __syncwarp();
        }
        if (use_census) {
            bool moving = false;
            if (cnt <= 1) {
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    const int i = lane + 32 * r;
                    if (i < N && ((mylive >> r) & 1u)) {
#pragma unroll
                        for (int k = 0; k < D; ++k) moving = moving || (Elem<T>::bits(x[i * D + k]) != 0);
                    }
                }
            }
            const bool org = !__any_sync(0xffffffffu, moving);
            if (lane == 0) p.census[g] = census_after_step(cnt, org);
            if (p.live_mask)
                store_mask(g, __ballot_sync(0xffffffffu, mylive & 1u), __ballot_sync(0xffffffffu, (mylive >> 1) & 1u));
        }
        // ---- outputs ----
        bool exceed = false;
        _Pragma("unroll UNR")
        for (int r = 0; r < R; ++r) {
            const int i = lane + 32 * r;
            const bool lv = (mylive >> r) & 1u;
            if (i < N) {
                if (lv) {
                    if (p.exceed_flag) {
#pragma unroll
                        for (int k = 0; k < D; ++k) exceed |= Elem<T>::to_float(x[i * D + k]) >= p.threshold;
                    }
                } else if (kops) {  // every reference op rewrites dead rows with the padding value: usually they hold it
                    uint32_t bad = 0;
#pragma unroll
                    for (int k = 0; k < D; ++k) bad |= (uint32_t)Elem<T>::bits(x[i * D + k]) ^ (uint32_t)Elem<T>::bits(padv);
                    if (bad) {
                        chg = true;
#pragma unroll
                        for (int k = 0; k < D; ++k) x[i * D + k] = padv;
                    }
                }
            }
        }
        if (lane == 0) {
            if (p.num_points) p.num_points[g] = cnt;
            if (p.length) p.length[g] = len;
            if constexpr (THR) {
                if (p.over_step) p.over_step[g] = over;
            }
        }
        if (p.exceed_flag) {
            if (__any_sync(0xffffffffu, exceed) && lane == 0) *p.exceed_flag = 1;
        }
        __syncwarp();
        if (gout && __any_sync(0xffffffffu, chg)) {
            const uint32_t* src = slot + b * Wpad;
            uint32_t* dst = gout + g * W;
            if (vec_out) {
                for (int c = lane; c < (W >> 2); c += 32)
                    reinterpret_cast<uint4*>(dst)[c] = reinterpret_cast<const uint4*>(src)[c];
            } else {
                for (int w = lane; w < W; w += 32) dst[w] = src[w];
            }
        }
        // ---- observation features ----
        if constexpr (OBS) {
            if (p.obs) {
                float mx = -1.0f;
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    if (!((mylive >> r) & 1u)) continue;
                    const int i = lane + 32 * r;
#pragma unroll
                    for (int k = 0; k < D; ++k) mx = fmaxf(mx, Elem<T>::to_float(x[i * D + k]));
                }
                mx = warp_maxf(mx);
                if (mx == 0.0f || ((kflags & HK_F_RESCALE_EPS) && mx > 0.0f && mx <= 1e-8f)) mx = 1.0f;
                const bool resc = (kflags & HK_F_OBS_RESCALE) && (mx > 0.0f);
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    const int i = lane + 32 * r;
                    if (i >= N) continue;
                    const bool lv = (mylive >> r) & 1u;
#pragma unroll
                    for (int k = 0; k < D; ++k) {
                        float v = Elem<T>::to_float(x[i * D + k]);
                        v = (resc && lv && v != 0.0f) ? __fdiv_rn(v, mx) : v;
                        f[i * D + k] = lv ? v : p.pad;
                    }
                }
                __syncwarp();
                float* gobs = p.obs + g * (long long)OW;
                const bool sorted = kflags & (HK_F_OBS_SORT_COORD0 | HK_F_OBS_SORT_LEX | HK_F_OBS_SORT_LEX_FIRST);
                const bool lex = kflags & HK_F_OBS_SORT_LEX;
                const bool lexf = kflags & HK_F_OBS_SORT_LEX_FIRST;
                _Pragma("unroll UNR")
                for (int r = 0; r < R; ++r) {
                    const int i = lane + 32 * r;
                    if (i >= N) continue;
                    float fi[D];
#pragma unroll
                    for (int k = 0; k < D; ++k) fi[k] = f[i * D + k];
                    int rank = i;
                    if (sorted) {
                        rank = 0;
                        for (int j = 0; j < N; ++j) {
                            bool gt = f[j * D] > fi[0];
                            bool eq = f[j * D] == fi[0];
                            if (lex) {
#pragma unroll
                                for (int k = 1; k < D; ++k) {
                                    const float fj = f[j * D + k];
                                    gt = (fj > fi[k]) || ((fj == fi[k]) && gt);
                                    eq = eq && (fj == fi[k]);
                                }
                            } else if (lexf) {
                                gt = f[j * D + D - 1] > fi[D - 1];
                                eq = f[j * D + D - 1] == fi[D - 1];
#pragma unroll
                                for (int k = D - 2; k >= 0; --k) {
                                    const float fj = f[j * D + k];
                                    gt = (fj > fi[k]) || ((fj == fi[k]) && gt);
                                    eq = eq && (fj == fi[k]);
                                }
                            }
                            rank += (gt || (eq && j < i)) ? 1 : 0;
                        }
                    }
#pragma unroll
                    for (int k = 0; k < D; ++k) gobs[rank * D + k] = fi[k];
                }
                if (p.obs_coord && lane < D) {
                    const uint32_t ocm = action_mask(load_action(p.obs_coord, g, kflags), kflags);
                    gobs[W + lane] = (float)((ocm >> lane) & 1u);
                }
            }
        }
        __syncwarp();  // every lane is done with buffer b before the next prefetch may overwrite it
    }
    cp_async_wait<0>();
    if (p.done_count) {
        if (dc0) atomicAdd(p.done_count + lane, dc0);
        if (dc1) atomicAdd(p.done_count + 32 + lane, dc1);
    }
}

}  // namespace hk
