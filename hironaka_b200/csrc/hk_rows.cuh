// hk_rows.cuh — census-scheduled thread-per-game step for the SMALL games of a large padded shape.
//
// The warp-per-game kernel (hk_generic.cuh) spends a whole warp and ~300 warp-instructions on a game, however
// few of its N rows are alive.  In a rollout at (64,5) most games are down to a handful of rows after three or
// four steps (mean 7.4 live rows after 4 random-play steps, 3.2 after 8): one LANE per game is then the right
// mapping, but a padded game is 1 280 bytes, far too much to stage 32 of them per warp.  With the census the
// kernel does not need the padded game at all: the census byte gives the live count and the census mask (one
// 64-bit word per game, written by whichever kernel stepped the game last) says WHICH rows are alive, so a lane
// gathers just its game's live rows (d words each) straight into a compact shared-memory area, steps them in
// registers with the thread-per-game code of hk_small.cuh (tiers of 2, 4 and 8 rows), and writes back only the
// rows that changed or died.  At (64,5) that is ~100-200 bytes of traffic and ~30 warp-instructions per game
// instead of 2 560 bytes and ~300.
//
// One step of a large shape with a census is two launches (hk_capi.cu): this kernel takes the games whose known
// live count is at most ROWS_MAX_K (and answers the games at rest from their census byte), the warp-per-game
// kernel then takes the rest and skips what was done here.
#pragma once
#include "hk_census.cuh"
#include "hk_small.cuh"

namespace hk {

constexpr int ROWS_MAX_K = ROWS_K;        // games with at most this many live rows are stepped here
constexpr int ROWS_ROUND_GAMES = 1024;  // games a warp schedules together

template <int D, int WARPS, int STAGES>
struct RowsLayout {
    static constexpr int LANE_WORDS = ROWS_MAX_K * D + 1 - ((ROWS_MAX_K * D) & 1);  // odd stride: conflict-free lanes
    static constexpr int STAGE_WORDS = 32 * LANE_WORDS;
    static constexpr int CLS_WORDS = ROWS_ROUND_GAMES / 4;
    static constexpr int ORDER_WORDS = ROWS_ROUND_GAMES / 2;
    static constexpr int WARP_WORDS = STAGES * STAGE_WORDS + CLS_WORDS + ORDER_WORDS;
    static constexpr size_t SMEM_BYTES = (size_t)WARPS * WARP_WORDS * 4;
};

// K compact rows of one game per lane: gather order = slot order, so the lowest-slot-wins rule of the dedupe holds
template <typename T, int D, int K>
__device__ __forceinline__ void rows_step(const StepParams& p, const uint32_t* area, uint32_t* g_state, long long g,
                                          uint64_t mask, int cnt, bool valid, int32_t ha, int32_t ax, int& new_cnt,
                                          uint64_t& new_mask, bool& origin, bool& exceed) {
    T y[K * D];
    uint32_t clm = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const bool lv = valid && k < cnt;
        clm |= lv ? (1u << k) : 0u;
#pragma unroll
        for (int c = 0; c < D; ++c) y[k * D + c] = lv ? Elem<T>::from_bits(area[k * D + c]) : Elem<T>::zero();
    }
    const uint32_t clm0 = clm;
    clm = game_step<T, K, D, 0, false>(y, clm, p.ops, p.flags, ha, ax);
    new_cnt = __popc(clm);
    if (p.exceed_flag) exceed = exceeds<T, K, D>(y, clm, p.threshold);
    // back to the slots: a row that died becomes padding, a row that moved is rewritten, the others are left alone
    const T padv = Elem<T>::pad(p.pad);
    uint64_t m = mask, nm = mask;
    uint32_t nz = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        if ((clm0 >> k) & 1u) {
            const int slot = __ffsll((long long)m) - 1;
            m &= m - 1;
            const bool alive = (clm >> k) & 1u;
            bool moved = false;
#pragma unroll
            for (int c = 0; c < D; ++c) {
                moved = moved || ((uint32_t)Elem<T>::bits(y[k * D + c]) != area[k * D + c]);
                nz |= alive ? (uint32_t)Elem<T>::bits(y[k * D + c]) : 0u;
            }
            if (!alive) nm &= ~(1ull << slot);
            if (!alive || moved) {
                uint32_t* dst = g_state + slot * D;
#pragma unroll
                for (int c = 0; c < D; ++c) dst[c] = (uint32_t)Elem<T>::bits(alive ? y[k * D + c] : padv);
            }
        }
    }
    new_mask = nm;
    origin = (nz == 0);
}

template <typename T, int D, int WARPS, int STAGES>
__global__ void __launch_bounds__(WARPS * 32) hk_rows_kernel(const StepParams p) {
    using L = RowsLayout<D, WARPS, STAGES>;
    constexpr int LW = L::LANE_WORDS;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t* wbase = reinterpret_cast<uint32_t*>(smem_raw) + (size_t)warp * L::WARP_WORDS;
    uint32_t* stages = wbase;
    uint8_t* clsb = reinterpret_cast<uint8_t*>(wbase + STAGES * L::STAGE_WORDS);
    uint16_t* order = reinterpret_cast<uint16_t*>(wbase + STAGES * L::STAGE_WORDS + L::CLS_WORDS);

    const long long B = p.B;
    const int W = p.N * D;
    const long long gw = (long long)blockIdx.x * WARPS + warp;
    const long long nw = (long long)gridDim.x * WARPS;
    uint32_t* gst = reinterpret_cast<uint32_t*>(p.out);
    const uint32_t lt = (1u << lane) - 1u;
    const bool frozen_rest = census_frozen_rest(p.ops, p.flags);
    const float rest_r = rest_reward(p.flags);
    int done_total = 0;

    // a warp owns a contiguous run of games, scheduled in rounds of RG games (a multiple of 32, at most
    // ROWS_ROUND_GAMES; smaller when the batch is small, so that every warp of the grid has a round)
    long long per = (B + nw - 1) / nw;
    per = (per + 31) & ~31ll;
    const int RG = (int)(per > ROWS_ROUND_GAMES ? ROWS_ROUND_GAMES : (per < 32 ? 32 : per));
    const long long rounds = (B + RG - 1) / RG;
    const long long rpw = (rounds + nw - 1) / nw;
    for (long long rd = gw * rpw; rd < (gw + 1) * rpw && rd < rounds; ++rd) {
        const long long g0 = rd * RG;
        const int ng = (int)((B - g0 < RG) ? (B - g0) : RG);
        // ---- the round's census bytes into shared memory ----
        {
            const uint8_t* cb = p.census + g0;
            if ((reinterpret_cast<uintptr_t>(cb) & 3u) == 0) {
                for (int o = lane * 4; o < ng; o += 128) {
                    if (o + 4 <= ng) cp_async_4(clsb + o, cb + o);
                    else {
                        for (int q = 0; q < 4; ++q) clsb[o + q] = (o + q < ng) ? __ldg(cb + o + q) : (uint8_t)0;
                    }
                }
                cp_async_commit();
                cp_async_wait<0>();
            } else {
                for (int o = lane; o < ng; o += 32) clsb[o] = __ldg(cb + o);
            }
            __syncwarp();
        }
        // ---- games at rest: outputs from the census byte; small games in play: classes 1..3 by live count ----
        uint32_t classes = 0;
        for (int o = lane; o < ((ng + 31) & ~31); o += 32) {
            const bool valid = o < ng;
            const uint32_t v = valid ? (uint32_t)clsb[o] : 0u;
            const bool rest = valid && census_at_rest(v, frozen_rest);
            const long long g = g0 + o;
            if (rest) write_rest_outputs(p, g, v, rest_r);
            const uint32_t restmask = __ballot_sync(0xffffffffu, rest);
            done_total += __popc(restmask);
            // the tile's word of the done mask: games at rest now; games that finish in this step are ORed in later
            // (by this kernel or by the warp-per-game launch that follows)
            if (p.done_bits && lane == 0) p.done_bits[g >> 5] = restmask;
            const int cnt = (int)census_live_count(v);
            const int c = (!valid || rest || v == 0 || cnt > ROWS_MAX_K) ? 0 : (cnt <= 2 ? 1 : (cnt <= 4 ? 2 : 3));
            if (valid) clsb[o] = (uint8_t)(c ? (c | (cnt << 2)) : 0);  // class in the low 2 bits, live count above
            classes |= 1u << c;
        }
        classes = __reduce_or_sync(0xffffffffu, classes) & ~1u;
        __syncwarp();
        if (classes == 0) continue;
        int total = 0;
        for (int q = 1; q <= 3; ++q) {
            if (!((classes >> q) & 1u)) continue;
            for (int o = lane; o < ((ng + 31) & ~31); o += 32) {
                const bool m = (o < ng) && ((clsb[o] & 3u) == (uint32_t)q);
                const uint32_t bal = __ballot_sync(0xffffffffu, m);
                if (m) order[total + __popc(bal & lt)] = (uint16_t)o;
                total += __popc(bal);
            }
        }
        __syncwarp();
        const int nchunks = (total + 31) >> 5;

        struct Pick {
            long long g;
            uint64_t mask;
            int cnt;
            bool valid;
        };
        auto pick = [&](int v) -> Pick {
            Pick k;
            const int idx = v * 32 + lane;
            k.valid = idx < total;
            const int o = k.valid ? (int)order[idx] : 0;
            k.g = g0 + o;
            k.cnt = k.valid ? (int)(clsb[o] >> 2) : 0;
            k.mask = k.valid ? __ldg(reinterpret_cast<const unsigned long long*>(p.live_mask) + k.g) : 0ull;
            return k;
        };
        // each lane gathers the live rows of its own game, D words per row, into its compact area
        auto gather = [&](const Pick& k, uint32_t* stage) {
            uint32_t* area = stage + lane * LW;
            const uint32_t* src = gst + k.g * W;
            uint64_t m = k.mask;
#pragma unroll
            for (int r = 0; r < ROWS_MAX_K; ++r) {
                if (r < k.cnt) {
                    const int slot = __ffsll((long long)m) - 1;
                    m &= m - 1;
#pragma unroll
                    for (int c = 0; c < D; ++c) cp_async_4(area + r * D + c, src + slot * D + c);
                }
            }
            cp_async_commit();
        };

        Pick cur = pick(0), nxt;
        nxt.g = 0, nxt.mask = 0, nxt.cnt = 0, nxt.valid = false;
        gather(cur, stages);
        for (int v = 0; v < nchunks; ++v) {
            uint32_t* stage = stages + (STAGES == 1 ? 0 : (v & 1)) * L::STAGE_WORDS;
            int32_t ha = 3, ax = 0;
            if ((p.ops & HK_OP_SHIFT) && cur.valid) load_actions(p, p.flags, cur.g, 0, ha, ax);
            if (STAGES >= 2 && v + 1 < nchunks) {
                nxt = pick(v + 1);
                gather(nxt, stages + ((v + 1) & 1) * L::STAGE_WORDS);
                cp_async_wait<1>();
            } else {
                cp_async_wait<0>();
            }
            __syncwarp();
            const int cmax = __reduce_max_sync(0xffffffffu, cur.cnt);
            const uint32_t* area = stage + lane * LW;
            int ncnt = 0;
            uint64_t nmask = 0;
            bool origin = false, exceed = false;
            const bool prev_done = cur.cnt < 2;
            if (cmax <= 2)
                rows_step<T, D, 2>(p, area, gst + cur.g * W, cur.g, cur.mask, cur.cnt, cur.valid, ha, ax, ncnt, nmask, origin, exceed);
            else if (cmax <= 4)
                rows_step<T, D, 4>(p, area, gst + cur.g * W, cur.g, cur.mask, cur.cnt, cur.valid, ha, ax, ncnt, nmask, origin, exceed);
            else
                rows_step<T, D, ROWS_MAX_K>(p, area, gst + cur.g * W, cur.g, cur.mask, cur.cnt, cur.valid, ha, ax, ncnt, nmask, origin, exceed);
            const bool dn = ncnt < 2;
            if (cur.valid) {
                if (p.done) p.done[cur.g] = dn ? 1 : 0;
                if (p.reward) p.reward[cur.g] = step_reward(p.flags, dn, prev_done);
                if (p.num_points) p.num_points[cur.g] = ncnt;
                if (p.done_bits && dn) atomicOr(p.done_bits + (cur.g >> 5), 1u << (cur.g & 31));
                p.census[cur.g] = census_after_step(ncnt, origin);
                if (nmask != cur.mask) p.live_mask[cur.g] = nmask;
            }
            done_total += __popc(__ballot_sync(0xffffffffu, cur.valid && dn));
            if (p.exceed_flag) {
                if (__any_sync(0xffffffffu, exceed && cur.valid) && lane == 0) *p.exceed_flag = 1;
            }
            __syncwarp();
            if (STAGES == 1 && v + 1 < nchunks) {
                nxt = pick(v + 1);
                gather(nxt, stages);
            }
            cur = nxt;
        }
    }
    if (p.done_count && done_total && lane == 0) atomicAdd(p.done_count, done_total);
}

}  // namespace hk
