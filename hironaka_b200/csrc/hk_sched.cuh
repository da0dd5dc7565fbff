// hk_sched.cuh — census-scheduled thread-per-game step kernel (in-place single steps of small games).
//
// The tile-ring kernel (hk_small.cuh) reads every game every step and lets a tile's BUSIEST game pick the
// tier for all 32.  In a rollout that wastes most of the work: a game that has ended sits at a fixed point
// (a lone point at the origin: 52 % of the games after 5 random-play steps at (20,3), 95 % after 10), and the
// live counts inside a tile are heavy-tailed (mean 6 rows, tile maximum 11 at the root).  This kernel keeps
// a CENSUS — one byte per game, written by the previous step — and schedules by it:
//   * games at rest are not loaded at all: their done = 1 / reward = 0 come from the census byte;
//   * the other games of a warp's tiles are ordered by live count (counting sort over six tier classes)
//     and cut into chunks of 32, so that a chunk's tier fits all of its games;
//   * each chunk is gathered game by game: where a game is a whole number of 16-byte words ((20,3): 240 B)
//     every lane issues ONE TMA bulk copy (cp.async.bulk, SASS UBLKCP) for its own game onto the stage's
//     mbarrier, and a changed game goes back with one bulk store per lane; the other shapes ((10,3), (5,3),
//     unaligned pointers) are copied with cp.async in 8/4-byte pieces, 15 lanes per game.  The chunk is
//     processed by the same per-game code as the tile-ring kernel (small_process_tile).
// Work and DRAM traffic follow the number of games still in play instead of the batch size.
//
// The census byte is defined in hk_census.cuh.
#pragma once
#include "hk_census.cuh"
#include "hk_small.cuh"

namespace hk {

constexpr int SCHED_ROUND_TILES = 32;  // tiles (of 32 games) a warp schedules together
#ifndef SCHED_PASS_UNROLL
#define SCHED_PASS_UNROLL 2
#endif
constexpr int kSchedPassUnroll = SCHED_PASS_UNROLL;
#ifndef SCHED_NATURAL_NUM
#define SCHED_NATURAL_NUM 1  // a round is stepped tile by tile in natural order while at least NUM / DEN of
#define SCHED_NATURAL_DEN 2  // its games are in play (tools/time_census.py)
#endif
// the class sort packs its counts in 10-bit fields: a sorted round has fewer games in play than games (< 1024) only
// while the ratio is at most one (above one, rounds wholly in play would be sorted too)
static_assert(SCHED_NATURAL_NUM <= SCHED_NATURAL_DEN, "a sorted round must have fewer than 1024 games in play");

template <int N, int D, int WARPS, int STAGES, bool OBS = false>
struct SchedLayout {
    static constexpr int W = N * D;
    static constexpr int STAGE_WORDS = 32 * W;
    static constexpr int OBS_WORDS = OBS ? 32 * (W + D) : 0;  // the observation rows of one chunk
    // per warp: STAGES game stages, the class bytes of a round (one per game), the sorted order (u16 per game)
    static constexpr int CLS_WORDS = SCHED_ROUND_TILES * 32 / 4;
    static constexpr int ORDER_WORDS = SCHED_ROUND_TILES * 32 / 2;
    static constexpr int WARP_WORDS = STAGES * STAGE_WORDS + CLS_WORDS + ORDER_WORDS + OBS_WORDS;
    static constexpr int BAR_BYTES = 256;  // mbarriers first (WARPS * STAGES of them), then the warps' areas
    static_assert(WARPS * STAGES * 8 <= BAR_BYTES, "mbarrier area too small");
    static constexpr size_t SMEM_BYTES = BAR_BYTES + (size_t)WARPS * WARP_WORDS * 4;
};

// Byte-SIMD helpers of the census pass: a 32-bit word holds the census bytes of four consecutive games.
// bit 7 of each byte of the result: that byte of x (<= 0x7f) is >= t (t <= 0x7f; no borrow crosses a byte)
__device__ __forceinline__ uint32_t bytes_ge7(uint32_t x7, uint32_t t) {
    return ((x7 | 0x80808080u) - t * 0x01010101u) & 0x80808080u;
}
// bits 0..3: which bytes of x are non-zero
__device__ __forceinline__ uint32_t nonzero_bytes4(uint32_t x) {
    const uint32_t hi = (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
    return ((hi >> 7) * 0x01020408u) >> 24;  // bits 0, 8, 16, 24 -> 24, 25, 26, 27 (no two partial products collide)
}

// Class codes of four census bytes (the class array's format): class 0 = at rest or no such game; 1..6 = the tier
// class of a game in play (6 for an unknown byte, 1 for "ended, not at rest under this launch's ops" and for 1-2
// live rows, else 1 + [v > 2] + [v > 4] + [v > 8] + [v > 12] + [v > 16]); 0x80 = at rest; 0x40 = its live count.
// vmask keeps the bytes of games that exist; rest7 returns the at-rest flags (bit 7 of each byte): census_at_rest of
// each byte, four at a time.
__device__ __forceinline__ uint32_t census_codes4(uint32_t w, uint32_t vmask, bool frozen_rest, uint32_t& rest7) {
    constexpr uint32_t BYTES4 = 0x01010101u;                   // times a byte value: that value in each byte
    constexpr uint32_t ENDED4 = CENSUS_ENDED * BYTES4;         // the ended bit of each byte
    constexpr uint32_t LOW4 = (~CENSUS_ENDED & 0xffu) * BYTES4;  // the bits below it: a live count in play
    static_assert(CENSUS_AT_ORIGIN << 6 == CENSUS_ENDED, "the at-origin bit is shifted onto the ended bit");
    w &= vmask;
    const uint32_t ended = w & ENDED4;
    rest7 = ended & ((w << 6) | (frozen_rest ? ENDED4 : 0u)) & vmask;  // ended and (at origin or frozen)
    const uint32_t x7 = w & LOW4;
    uint32_t c = 0x01010101u + (bytes_ge7(x7, 3) >> 7) + (bytes_ge7(x7, 5) >> 7) + (bytes_ge7(x7, 9) >> 7) +
                 (bytes_ge7(x7, 13) >> 7) + (bytes_ge7(x7, 17) >> 7);
    const uint32_t unknown = ~(bytes_ge7(x7, 1) | ended) & ENDED4;  // a zero byte
    c += (unknown >> 7) * 5u;
    const uint32_t endedff = (ended >> 7) * 0xffu;
    c = (c & ~endedff) | (ended >> 7);
    c &= vmask & ~((rest7 >> 7) * 0xffu);
    return c | rest7 | ((w & BYTES4) << 6);  // bit 0 of each byte (the live count of an ended game) at 0x40
}

// Per-lane counts of the classes 1..6 of four class codes, packed in 10-bit fields: classes 1-3 in lo, 4-6 in hi.
__device__ __forceinline__ void class_counts4(uint32_t code, uint32_t& lo, uint32_t& hi) {
    const uint32_t x7 = code & 0x07070707u;
    const int g1 = __popc(bytes_ge7(x7, 1)), g2 = __popc(bytes_ge7(x7, 2)), g3 = __popc(bytes_ge7(x7, 3));
    const int g4 = __popc(bytes_ge7(x7, 4)), g5 = __popc(bytes_ge7(x7, 5)), g6 = __popc(bytes_ge7(x7, 6));
    lo = (uint32_t)(g1 - g2) | ((uint32_t)(g2 - g3) << 10) | ((uint32_t)(g3 - g4) << 20);
    hi = (uint32_t)(g4 - g5) | ((uint32_t)(g5 - g6) << 10) | ((uint32_t)g6 << 20);
}

// OBS: the instantiation that also builds the observation features of the new state (p.obs, sorted modes only):
// a game at rest has a CONSTANT observation — its lone point, at the origin, sorts first, the rest is padding — so
// it is written from the census byte like the other outputs, and only the games in play run the feature code.
template <typename T, int N, int D, int WARPS, int STAGES, bool OBS = false, int MINB = 1>
__global__ void __launch_bounds__(WARPS * 32, MINB) hk_sched_kernel(const StepParams p) {
    using L = SchedLayout<N, D, WARPS, STAGES, OBS>;
    constexpr int W = L::W;
    constexpr int CHW = (W % 4 == 0) ? 4 : ((W % 2 == 0) ? 2 : 1);  // words per copy piece
    constexpr int LPG = W / CHW;                                     // lanes per game
    static_assert(LPG <= 32, "a game is copied by at most one warp instruction");
    constexpr int GPI = 32 / LPG;                                    // games per copy instruction
    constexpr int COPY_ITERS = (32 + GPI - 1) / GPI;
    extern __shared__ __align__(128) uint8_t smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw) + warp * STAGES;
    uint32_t* wbase = reinterpret_cast<uint32_t*>(smem_raw + L::BAR_BYTES) + (size_t)warp * L::WARP_WORDS;
    uint32_t* stages = wbase;
    uint8_t* clsb = reinterpret_cast<uint8_t*>(wbase + STAGES * L::STAGE_WORDS);
    uint16_t* order = reinterpret_cast<uint16_t*>(wbase + STAGES * L::STAGE_WORDS + L::CLS_WORDS);
    float* obs_tile = reinterpret_cast<float*>(wbase + STAGES * L::STAGE_WORDS + L::CLS_WORDS + L::ORDER_WORDS);
    const int OW = W + (p.obs_coord ? D : 0);
    const bool obs_bulk = OBS && aligned16(p.obs) && ((OW & 3) == 0);

    const long long B = p.B;
    const long long ntiles = (B + 31) >> 5;
    const long long gw = (long long)blockIdx.x * WARPS + warp;
    const long long nw = (long long)gridDim.x * WARPS;
    uint32_t* gst = reinterpret_cast<uint32_t*>(p.out);  // in place: p.out == p.in
    const bool piece_ok = ((reinterpret_cast<uintptr_t>(p.out)) & (CHW * 4 - 1)) == 0;
    // one TMA bulk copy per game when a game is a whole number of 16-byte words and the state is 16-byte aligned
    const bool bulk = ((W * 4) % 16 == 0) && aligned16(p.out);
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < STAGES; ++s) mbar_init(&bar[s], 1);
        mbar_fence_init();
    }
    __syncwarp();
    uint32_t phase_bits = 0;  // bit s = parity to wait for on stage s
    const uint32_t lt = (1u << lane) - 1u;
    const bool frozen_rest = census_frozen_rest(p.ops, p.flags);
    const float rest_r = rest_reward(p.flags);
    // piece lane -> (game slot within the instruction, piece within the game)
    const int sub = lane / LPG, piece = lane - sub * LPG;
    int settled_total = 0;  // per lane: games at rest
    // outputs of the games at rest as one vector store per lane (four games) where the pointer allows it
    const bool done4 = p.done && ((reinterpret_cast<uintptr_t>(p.done) & 3u) == 0);
    const bool reward16 = p.reward && aligned16(p.reward);
    const bool npoints16 = p.num_points && aligned16(p.num_points);

    // A warp owns a CONTIGUOUS run of tiles (its games share DRAM pages when they are gathered one by one),
    // scheduled in rounds of SCHED_ROUND_TILES.
    const long long tpw = (ntiles + nw - 1) / nw;
    const long long t_begin = gw * tpw;
    const long long t_end = (t_begin + tpw < ntiles) ? (t_begin + tpw) : ntiles;
    auto tile_of = [&](long long j) -> long long { return t_begin + j; };  // the warp's j-th tile
    uint32_t* clsw = reinterpret_cast<uint32_t*>(clsb);
    for (long long j0 = 0; tile_of(j0) < t_end; j0 += SCHED_ROUND_TILES) {
        // ---- census of this round's tiles: outputs of the games at rest, class bytes of the others ----
        const int nk = (int)((t_end - t_begin - j0 < SCHED_ROUND_TILES) ? (t_end - t_begin - j0) : SCHED_ROUND_TILES);
        const int ngroups = (nk + 3) >> 2;  // groups of four tiles: lane l holds the census bytes of games 4l .. 4l+3
        const long long first = tile_of(j0) << 5;  // the round's first game
        const int cbytes = (int)((B - first < (long long)nk * 32) ? (B - first) : (long long)nk * 32);  // its games
        // The round's census words are staged in the class array, one per lane and group, all requests in flight at
        // once: cp.async where the census is 4-byte aligned, words assembled from byte loads otherwise (and for the
        // word that crosses B).  Bytes past B read as 0.
        {
            const uint8_t* cbase = p.census + first;
            const bool caligned = (reinterpret_cast<uintptr_t>(cbase) & 3u) == 0;
            for (int o = lane * 4; o < nk * 32; o += 128) {
                if (caligned && o + 4 <= cbytes) {
                    cp_async_4(clsb + o, cbase + o);
                } else {
                    uint32_t wv = 0;
                    for (int q = 0; q < 4; ++q) wv |= (o + q < cbytes) ? (uint32_t)__ldg(cbase + o + q) << (8 * q) : 0u;
                    clsw[o >> 2] = wv;
                }
            }
            cp_async_commit();
            cp_async_wait<0>();
            __syncwarp();
        }
        // pass 1, four games per lane: class codes of the round (one 32-bit word per lane and group, the byte order of
        // the class array: byte k * 32 + i is game i of tile k), what is in play; without the fused observation also
        // the outputs of the games at rest (with it they are a second pass, below, that knows which tiles are about to
        // be stepped whole).  Late in a rollout this loop IS the step: a warp walks its tiles and finds a handful of
        // games in play.  Kept rolled: the kernel's hot loops compete for the instruction cache.
        uint32_t tilemask = 0;
        int inplay = 0;
        for (int G = 0; G < ngroups; ++G) {
            const int o = G * 128 + lane * 4;  // the lane's first game, within the round
            const int left = cbytes - o;
            const uint32_t vmask = left >= 4 ? 0xffffffffu : (left > 0 ? (1u << (8 * left)) - 1u : 0u);
            const uint32_t w = clsw[G * 32 + lane];
            uint32_t rest7;
            const uint32_t code = census_codes4(w, vmask, frozen_rest, rest7);
            clsw[G * 32 + lane] = code;
            const uint32_t cls = code & 0x07070707u;
            // tile t of the group is lanes 8t .. 8t+7: byte t of the ballot
            tilemask |= nonzero_bytes4(__ballot_sync(0xffffffffu, cls != 0)) << (4 * G);
            inplay += __popc(bytes_ge7(cls, 1));
            settled_total += __popc(rest7);
            if constexpr (!OBS) {
                if (rest7) {
                    // Four games in one store, those in play included: the chunk loop writes their outputs later, from
                    // this warp, after the __syncwarp that ends this pass (it orders these stores before those).
                    const long long g0 = first + o;
                    const bool whole = left >= 4;
                    const uint32_t live = w & 0x01010101u;
                    if (whole && done4) *reinterpret_cast<uint32_t*>(p.done + g0) = rest7 >> 7;
                    if (whole && reward16) *reinterpret_cast<float4*>(p.reward + g0) = make_float4(rest_r, rest_r, rest_r, rest_r);
                    if (whole && npoints16) *reinterpret_cast<int4*>(p.num_points + g0) = make_int4((int)(live & 1u), (int)((live >> 8) & 1u), (int)((live >> 16) & 1u), (int)(live >> 24));
                    for (uint32_t m = rest7; m; m &= m - 1) {  // otherwise one store per game at rest
                        const int b = (__ffs((int)m) - 1) >> 3;
                        if (p.done && !(whole && done4)) p.done[g0 + b] = 1;
                        if (p.reward && !(whole && reward16)) p.reward[g0 + b] = rest_r;
                        if (p.num_points && !(whole && npoints16)) p.num_points[g0 + b] = (int32_t)((live >> (8 * b)) & 1u);
                    }
                }
                if (p.done_bits) {
                    // the tile's word of the done mask: the games at rest now (the games that finish in this step are
                    // ORed in by the chunk loop); eight lanes' nibbles, one lane per tile stores it
                    uint32_t bits = nonzero_bytes4(rest7) << (4 * (lane & 7));
                    bits |= __shfl_xor_sync(0xffffffffu, bits, 1);
                    bits |= __shfl_xor_sync(0xffffffffu, bits, 2);
                    bits |= __shfl_xor_sync(0xffffffffu, bits, 4);
                    const int k = G * 4 + (lane >> 3);
                    if ((lane & 7) == 0 && k < nk) p.done_bits[tile_of(j0 + k)] = bits;
                }
            }
        }
        inplay = __reduce_add_sync(0xffffffffu, inplay);
        const int ngames = cbytes;
        // While most games are still in play the tiles are stepped whole, in natural order: one bulk copy per
        // tile and coalesced actions / outputs beat the per-game gather, and there is little to skip.  Later the
        // games in play are sorted by class and gathered one by one.
        // (with the fused observation the per-game stores of the sorted order cost more: natural order down to a quarter)
        const bool natural = OBS ? (inplay * 4 >= ngames) : (inplay * SCHED_NATURAL_DEN >= ngames * SCHED_NATURAL_NUM);
        __syncwarp();
        // ---- counting sort of the games in play by class: order[] lists them (tile slot * 32 + lane) ----
        int total = 0;
        if (!natural && inplay <= 32) {  // one chunk whatever the order: a single compaction pass
#pragma unroll kSchedPassUnroll
            for (int k = 0; k < nk; ++k) {
                if (!((tilemask >> k) & 1u)) continue;
                const bool m = (clsb[k * 32 + lane] & 7u) != 0u;
                const uint32_t bal = __ballot_sync(0xffffffffu, m);
                if (m) order[total + __popc(bal & lt)] = (uint16_t)(k * 32 + lane);
                total += __popc(bal);
            }
        } else if (!natural) {
            // One counting sort over the class words, in game order inside a class (group, lane, byte).  Counts are
            // packed three classes to a word in 10-bit fields: a sorted round has fewer than 1024 games in play.
            // First the round's count of each class, then its start in order[] ...
            uint32_t tlo = 0, thi = 0;
            for (int G = 0; G < ngroups; ++G) {
                if (!((tilemask >> (4 * G)) & 0xfu)) continue;
                uint32_t lo, hi;
                class_counts4(clsw[G * 32 + lane], lo, hi);
                tlo += lo;
                thi += hi;
            }
            tlo = __reduce_add_sync(0xffffffffu, tlo);
            thi = __reduce_add_sync(0xffffffffu, thi);
            const uint32_t s123 = ((tlo * 0x00100401u) >> 20) & 0x3ffu;  // games of classes 1..3
            uint32_t plo = ((tlo << 10) + (tlo << 20)) & 0x3ffffc00u;    // starts of classes 1, 2, 3
            uint32_t phi = s123 * 0x00100401u + (((thi << 10) + (thi << 20)) & 0x3ffffc00u);  // of 4, 5, 6
            // ... then group by group: a warp scan of the lanes' packed counts gives each lane its place
            for (int G = 0; G < ngroups; ++G) {
                if (!((tilemask >> (4 * G)) & 0xfu)) continue;
                const uint32_t code = clsw[G * 32 + lane];
                uint32_t lo, hi;
                class_counts4(code, lo, hi);
                uint32_t ilo = lo, ihi = hi;  // inclusive scan over the lanes
#pragma unroll
                for (int s = 1; s < 32; s <<= 1) {
                    const uint32_t a = __shfl_up_sync(0xffffffffu, ilo, s), b = __shfl_up_sync(0xffffffffu, ihi, s);
                    if (lane >= s) {
                        ilo += a;
                        ihi += b;
                    }
                }
                uint32_t qlo = plo + ilo - lo, qhi = phi + ihi - hi;  // this lane's next slot of each class
                plo += __shfl_sync(0xffffffffu, ilo, 31);
                phi += __shfl_sync(0xffffffffu, ihi, 31);
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const int c = (code >> (8 * b)) & 7;
                    if (c == 0) continue;
                    const int sh = 10 * (c > 3 ? c - 4 : c - 1);
                    uint32_t& q = (c > 3) ? qhi : qlo;
                    order[(q >> sh) & 0x3ffu] = (uint16_t)(G * 128 + lane * 4 + b);
                    q += 1u << sh;
                }
            }
            total = inplay;
        }
        __syncwarp();
        const int nchunks = natural ? __popc(tilemask) : ((total + 31) >> 5);
        uint32_t tiles_left = tilemask;  // natural order: the tiles still to be requested

        // lane's game of chunk v (natural order: the next tile with a game in play; its games at rest ride along
        // in the tile copy but are not stepped: their outputs were written above)
        auto chunk_game = [&](int v, long long& g, bool& valid) {
            if (natural) {
                const int k = __ffs((int)tiles_left) - 1;
                tiles_left &= tiles_left - 1;
                g = (tile_of(j0 + k) << 5) + lane;
                valid = (g < B) && ((clsb[k * 32 + lane] & 7u) != 0);
                return;
            }
            const int idx = v * 32 + lane;
            valid = idx < total;
            const int lid = valid ? (int)order[idx] : 0;
            g = (tile_of(j0 + (lid >> 5)) << 5) + (lid & 31);
        };
        // gather the chunk's games into a stage: game slot s at s * W words
        auto gather = [&](long long g, bool valid, uint32_t* stage, int sidx) {
            if (natural) {  // the whole tile: games g - lane .. of which (B - first) may be fewer than 32
                const long long first = g - lane;
                const int cnt = (int)((B - first < 32) ? (B - first) : 32);
                if (bulk) {
                    bulk_wait_read<0>();
                    // the lanes wrote this stage with st.shared (results, scratch) and it may not have been stored: order
                    // those generic-proxy writes before the async-proxy write of the refill
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        mbar_expect_tx(&bar[sidx], (uint32_t)cnt * (uint32_t)(W * 4));
                        bulk_load(stage, gst + first * W, (uint32_t)cnt * (uint32_t)(W * 4), &bar[sidx]);
                    }
                    return;
                }
                if (piece_ok) {
                    for (int w = lane * CHW; w < cnt * W; w += 32 * CHW) {
                        if constexpr (CHW == 4) cp_async_16(stage + w, gst + first * W + w);
                        else if constexpr (CHW == 2) cp_async_8(stage + w, gst + first * W + w);
                        else cp_async_4(stage + w, gst + first * W + w);
                    }
                } else {
                    for (int w = lane; w < cnt * W; w += 32) cp_async_4(stage + w, gst + first * W + w);
                }
                cp_async_commit();
                return;
            }
            if (bulk) {
                // the lane's own earlier bulk store from this stage must have finished READING it
                bulk_wait_read<0>();
                fence_async_smem();  // (as above: earlier st.shared writes of this stage before the async-proxy refill)
                const int nvalid = __popc(__ballot_sync(0xffffffffu, valid));
                if (lane == 0) mbar_expect_tx(&bar[sidx], (uint32_t)nvalid * (uint32_t)(W * 4));
                __syncwarp();
                if (valid) bulk_load(stage + lane * W, gst + g * W, (uint32_t)(W * 4), &bar[sidx]);
                return;
            }
            if (piece_ok) {
#pragma unroll
                for (int it = 0; it < COPY_ITERS; ++it) {
                    const int s = it * GPI + sub;
                    const long long gs = __shfl_sync(0xffffffffu, g, s & 31);
                    const bool vs = __shfl_sync(0xffffffffu, valid ? 1 : 0, s & 31) != 0;
                    if (sub < GPI && s < 32 && vs) {
                        uint32_t* dst = stage + s * W + piece * CHW;
                        const uint32_t* src = gst + gs * W + piece * CHW;
                        if constexpr (CHW == 4) cp_async_16(dst, src);
                        else if constexpr (CHW == 2) cp_async_8(dst, src);
                        else cp_async_4(dst, src);
                    }
                }
            } else {  // state pointer aligned to 4 bytes only: word copies
                for (int s = 0; s < 32; ++s) {
                    const long long gs = __shfl_sync(0xffffffffu, g, s);
                    const bool vs = __shfl_sync(0xffffffffu, valid ? 1 : 0, s) != 0;
                    if (vs) {
                        for (int w = lane; w < W; w += 32) cp_async_4(stage + s * W + w, gst + gs * W + w);
                    }
                }
            }
            cp_async_commit();
        };

        // the first chunk is requested BEFORE the outputs of the games at rest are written: pass 2 runs in the shadow of
        // that load's DRAM latency (late in a rollout a warp has one short chunk: the load was the longest wait of the step)
        long long g_cur = 0, g_nxt = 0;
        bool v_cur = false, v_nxt = false;
        if (inplay) {
            chunk_game(0, g_cur, v_cur);
            gather(g_cur, v_cur, stages, 0);
        }
        // pass 2 (fused observation only): the outputs of the games at rest, from their census bytes
        for (int k = 0; OBS && k < nk; ++k) {
            const long long g = (tile_of(j0 + k) << 5) + lane;
            const uint32_t code = clsb[k * 32 + lane];
            const bool rest = code & 0x80u;
            const uint32_t v = (code >> 6) & 1u;  // live count of a game at rest
            if (rest) write_rest_outputs(p, g, v, rest_r);
            const uint32_t restmask = __ballot_sync(0xffffffffu, rest);
            if constexpr (OBS) {
                // (warp-uniform) the constant observation of every game at rest of this tile — unless the tile is about to
                // be stepped whole in natural order: its observation rows are then stored as one block, these included
                if (p.obs && restmask && !(natural && ((tilemask >> k) & 1u))) {
                    // staged in the observation tile like a chunk's rows, then ONE bulk store for a tile that is
                    // at rest as a whole (the common case late in a rollout), one per game otherwise
                    float* orow = obs_tile + lane * OW;
                    bulk_wait_read<0>();  // earlier observation stores have read the tile
                    __syncwarp();
                    if (rest) {
                        const float z = (v & 1u) ? 0.0f : p.pad;  // the lone point, at the origin, sorts first
                        const uint32_t ocm = p.obs_coord ? action_mask(load_action(p.obs_coord, g, p.flags), p.flags) : 0u;
                        if ((OW & 3) == 0 && D <= 4 && !p.obs_coord) {
                            float4* o4 = reinterpret_cast<float4*>(orow);
                            const float4 padv4 = make_float4(p.pad, p.pad, p.pad, p.pad);
                            o4[0] = make_float4(z, D > 1 ? z : p.pad, D > 2 ? z : p.pad, D > 3 ? z : p.pad);
#pragma unroll
                            for (int q = 1; q < W / 4; ++q) o4[q] = padv4;
                        } else {
                            for (int w = 0; w < OW; ++w)
                                orow[w] = (w < D) ? z : (w < W ? p.pad : (float)((ocm >> (w - W)) & 1u));
                        }
                    }
                    const long long first = g - lane;
                    const int cnt = (int)((B - first < 32) ? (B - first) : 32);
                    const uint32_t allmask = (cnt == 32) ? 0xffffffffu : ((1u << cnt) - 1u);
                    if (obs_bulk) {
                        fence_async_smem();
                        __syncwarp();
                        if (restmask == allmask) {
                            if (lane == 0) bulk_store(p.obs + first * OW, obs_tile, (uint32_t)(cnt * OW) * 4u);
                        } else if (rest) {
                            bulk_store(p.obs + g * OW, orow, (uint32_t)OW * 4u);
                        }
                        bulk_commit();
                    } else {
                        __syncwarp();
                        uint32_t m = restmask;
                        while (m) {
                            const int r = __ffs((int)m) - 1;
                            m &= m - 1;
                            warp_copy_words(reinterpret_cast<uint32_t*>(p.obs + (first + r) * OW),
                                            reinterpret_cast<uint32_t*>(obs_tile + r * OW), OW, lane);
                        }
                    }
                    __syncwarp();
                }
            }
            // the tile's word of the done mask: the games at rest now, the games that finish in this step later
            if (p.done_bits && lane == 0) p.done_bits[tile_of(j0 + k)] = restmask;
        }
        __syncwarp();
        if (inplay == 0) continue;
        for (int v = 0; v < nchunks; ++v) {
            const int sidx = (STAGES == 1) ? 0 : (v & 1);
            uint32_t* stage = stages + sidx * L::STAGE_WORDS;
            LaneState ls;
            ls.g = g_cur;
            ls.valid = v_cur;
            ls.shift = (p.ops & HK_OP_SHIFT) && ls.valid;
            ls.ha = 3;
            ls.ax = 0;
            ls.origin = false;
            if (ls.shift) load_actions(p, p.flags, ls.g, 0, ls.ha, ls.ax);
            // (measured and not kept: with one stage, a prefetch of the next tile into L2 here, as in hk_small.cuh)
            if (bulk) {  // this chunk's games have landed (they were requested one chunk ago)
                mbar_wait(&bar[sidx], (phase_bits >> sidx) & 1u);
                phase_bits ^= (1u << sidx);
            }
            if constexpr (STAGES >= 2) {
                // the next chunk streams into the other stage while this one is processed (its bulk stores of
                // the chunk before have had the wait above to drain)
                if (v + 1 < nchunks) {
                    chunk_game(v + 1, g_nxt, v_nxt);
                    gather(g_nxt, v_nxt, stages + ((v + 1) & 1) * L::STAGE_WORDS, (v + 1) & 1);
                    if (!bulk) cp_async_wait<1>();
                } else {
                    if (!bulk) cp_async_wait<0>();
                }
            } else {
                if (!bulk) cp_async_wait<0>();
            }
            __syncwarp();
            uint32_t* row = stage + lane * W;
            bool exceed = false;
            bool chg = false;  // in place: only changed games go back
            bool released = false;  // the stage has been handed back (and refilled) in the middle of the step
            if constexpr (!OBS && STAGES == 1 && !Elem<T>::is_float) {
                // packed tiers, direct route (hk_small.cuh): once the rows are gathered the stage is refilled — the next
                // chunk's load runs behind this chunk's arithmetic — and the changed rows go straight to global memory
                auto release = [&]() {
                    released = true;
                    __syncwarp();
                    if (v + 1 < nchunks) {
                        chunk_game(v + 1, g_nxt, v_nxt);
                        gather(g_nxt, v_nxt, stages, 0);
                    }
                };
                small_process_tile<T, N, D, false, true, decltype(release)>(p, ls, row, exceed, chg, gst + ls.g * W,
                                                                            release);
            } else {
                small_process_tile<T, N, D, false>(p, ls, row, exceed, chg);
            }
            if (ls.valid) {
                if (p.num_points) p.num_points[ls.g] = ls.cnt;
                if (p.done_bits && ls.cnt < 2) atomicOr(p.done_bits + (ls.g >> 5), 1u << (ls.g & 31));
                p.census[ls.g] = census_after_step(ls.cnt, ls.origin);
            }
            if (p.exceed_flag) {
                if (__any_sync(0xffffffffu, exceed && ls.valid) && lane == 0) *p.exceed_flag = 1;
            }
            if constexpr (OBS) {
                if (p.obs) {  // ---- observation features of the new state (in the lane's row area), as in K-small ----
                    const bool ingrid = ls.g < B;  // (natural order: the games at rest of the tile ride along)
                    float* orow = obs_tile + lane * OW;
                    bulk_wait_read<0>();  // the previous chunk's observation stores have read the tile
                    __syncwarp();
                    lane_features<T, N, D>(p, row, orow, OW, lane, ingrid);
                    append_obs_coord<D>(p, ls.g, ingrid, orow, W);
                    if (natural) {  // the tile's observations are contiguous
                        const long long first = ls.g - lane;
                        const int cnt = (int)((B - first < 32) ? (B - first) : 32);
                        if (obs_bulk) {
                            fence_async_smem();
                            __syncwarp();
                            if (lane == 0) bulk_store(p.obs + first * OW, obs_tile, (uint32_t)(cnt * OW) * 4u);
                            bulk_commit();
                        } else {
                            __syncwarp();
                            warp_copy_words(reinterpret_cast<uint32_t*>(p.obs + first * OW), reinterpret_cast<uint32_t*>(obs_tile),
                                            cnt * OW, lane);
                        }
                    } else if (obs_bulk) {  // one bulk store per game
                        fence_async_smem();
                        __syncwarp();
                        if (ls.valid) bulk_store(p.obs + ls.g * OW, orow, (uint32_t)OW * 4u);
                        bulk_commit();
                    } else {
                        __syncwarp();
                        for (int s2 = 0; s2 < 32; ++s2) {
                            const long long gs = __shfl_sync(0xffffffffu, ls.g, s2);
                            const bool vs = __shfl_sync(0xffffffffu, ls.valid ? 1 : 0, s2) != 0;
                            if (vs) warp_copy_words(reinterpret_cast<uint32_t*>(p.obs + gs * OW),
                                                    reinterpret_cast<uint32_t*>(obs_tile + s2 * OW), OW, lane);
                        }
                    }
                    __syncwarp();
                }
            }
            // ---- write-back of the changed games, GPI games per instruction ----
            uint32_t dirty = __ballot_sync(0xffffffffu, ls.valid && chg);
            __syncwarp();
            if (natural && __popc(dirty) > HK_SPARSE_STORE_MAX) {  // many changed games: the tile goes back whole
                const long long first = ls.g - lane;
                const int cnt = (int)((B - first < 32) ? (B - first) : 32);
                if (bulk) {
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0) bulk_store(gst + first * W, stage, (uint32_t)cnt * (uint32_t)(W * 4));
                    bulk_commit();
                } else {
                    warp_copy_words(gst + first * W, stage, cnt * W, lane);
                }
            } else if (bulk) {
                if (dirty) {
                    fence_async_smem();  // the lanes' st.shared results before the async-proxy reads of the stores
                    __syncwarp();
                    if (ls.valid && chg) bulk_store(gst + ls.g * W, row, (uint32_t)(W * 4));
                    bulk_commit();
                }
            } else if (piece_ok) {
                while (dirty) {
                    int s = -1;
                    uint32_t m = dirty;
#pragma unroll
                    for (int q = 0; q < GPI; ++q) {  // the q-th dirty game goes to the lanes with sub == q
                        const int b = m ? (__ffs((int)m) - 1) : -1;
                        m &= m - 1;
                        if (q == sub) s = b;
                    }
                    dirty = m;
                    const long long gs = __shfl_sync(0xffffffffu, ls.g, s < 0 ? 0 : s);
                    if (sub < GPI && s >= 0) {
                        const uint32_t* src = stage + s * W + piece * CHW;
                        uint32_t* dst = gst + gs * W + piece * CHW;
                        if constexpr (CHW == 4) *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
                        else if constexpr (CHW == 2) *reinterpret_cast<uint2*>(dst) = *reinterpret_cast<const uint2*>(src);
                        else *dst = *src;
                    }
                }
            } else {
                while (dirty) {
                    const int s = __ffs((int)dirty) - 1;
                    dirty &= dirty - 1;
                    const long long gs = __shfl_sync(0xffffffffu, ls.g, s);
                    warp_copy_words(gst + gs * W, stage + s * W, W, lane);
                }
            }
            __syncwarp();  // every lane is done with this stage before a later gather overwrites it
            if constexpr (STAGES == 1) {
                if (v + 1 < nchunks && !released) {
                    chunk_game(v + 1, g_nxt, v_nxt);
                    gather(g_nxt, v_nxt, stages, 0);
                }
            }
            g_cur = g_nxt;
            v_cur = v_nxt;
        }
    }
    if (bulk || obs_bulk) bulk_wait_all<0>();  // this lane's bulk stores are globally complete before the warp retires
    if (p.done_count) {
        settled_total = __reduce_add_sync(0xffffffffu, settled_total);
        if (settled_total && lane == 0) atomicAdd(p.done_count, settled_total);
    }
}

}  // namespace hk
