// hk_census.cuh — the census of hk_step_census: one byte per game, kept next to the state by the step that last
// touched the game and read by the next, so that games at rest are answered without loading them.
//
//   0                                      unknown: the game is read and counted
//   1 .. CENSUS_MAX_COUNT                  live rows of a game in play (counts above the maximum are stored as it)
//   CENSUS_ENDED | 2·at_origin | count     ended game (count <= 1 live rows, dead rows normalised); at_origin: no
//                                          row, or the lone row at the origin, so that no op moves it
//
// Large padded shapes (rows_shape, not is_small_shape) continue after the bytes, 8-byte aligned, with one 64-bit live
// mask per game (bit i <=> row i alive).  The NumPy decoders of the tests state the same format independently.
#pragma once
#include "hk_launch.cuh"

namespace hk {

constexpr uint32_t CENSUS_ENDED = 0x80u;
constexpr uint32_t CENSUS_AT_ORIGIN = 2u;
constexpr uint32_t CENSUS_MAX_COUNT = 127u;

// at rest under a launch: nothing moves an origin / empty game; a frozen ended game also rests when neither
// reposition nor rescale would move its lone point
__device__ __forceinline__ bool census_frozen_rest(uint32_t ops, uint32_t flags) {
    return (flags & HK_F_FREEZE_ENDED) && !(ops & (HK_OP_REPOSITION | HK_OP_RESCALE));
}

// the game is at rest under this launch's ops: its outputs come from the byte and it is not stepped
__device__ __forceinline__ bool census_at_rest(uint32_t byte, const bool& frozen_rest) {
    return (byte & CENSUS_ENDED) && ((byte & CENSUS_AT_ORIGIN) || frozen_rest);
}

// live count a known (non-zero) byte stands for
__device__ __forceinline__ uint32_t census_live_count(uint32_t byte) { return (byte & CENSUS_ENDED) ? (byte & 1u) : byte; }

// the byte of a game after a step left it with live_count rows (at_origin matters only once it has ended)
__device__ __forceinline__ uint8_t census_after_step(int live_count, const bool& at_origin) {
    return (uint8_t)((live_count <= 1) ? (CENSUS_ENDED | (at_origin ? CENSUS_AT_ORIGIN : 0u) | (uint32_t)live_count)
                                       : (uint32_t)(live_count > (int)CENSUS_MAX_COUNT ? (int)CENSUS_MAX_COUNT : live_count));
}

// byte offset of the live masks of a large padded shape
__host__ __device__ constexpr long long census_mask_offset(long long B) { return (B + 7) & ~7ll; }

__host__ __device__ constexpr long long census_bytes(long long B, int N, int d) {
    return (is_small_shape(N, d) || !rows_shape(N, d)) ? B : census_mask_offset(B) + 8 * B;
}

}  // namespace hk
