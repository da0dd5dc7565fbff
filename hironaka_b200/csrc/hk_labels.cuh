// hk_labels.cuh — value labels from the game-value search (hk_search_value_labels): every state hk_search_value
// solved with a value of at least one, read from its history after the level loop and hk_value_finish_kernel.  The
// kernels only read what the kernels of hk_minimax.cuh leave; none of those kernels changes.
//
// Two facts make the history a table of exact labels:
//   - an entry of level l solved in round R has value R - l, whatever its root's status: once a state is solved its
//     subtree stops growing, so no state below it is solved in a later round, and a state solved in round R has no
//     ancestor solved before R.  Ended states are the entries with R == l; the labels are the solved entries with R > l.
//   - the optimal host moves of a solved state are exactly its groups whose children are all solved: such a group has
//     Q = (its last child's round) - l <= R - l, the value; a group with an unsolved child c has value(c) >= R - l, since
//     c's subtree was built through level R.  A group's children are all solved exactly when h_rem at its first child is
//     0: the solve kernel takes one from it per solved child.
// The level of an entry is the number of parent hops up to its root (h_parent[h] < h).  Levels follow each other in
// the history, so a tile whose first and last entries have the same level lies in that level: two walks per tile, and
// only entries of the few tiles across a level boundary walk for themselves.
//
// Four passes over the `used` entries of the history, the count -> scan -> write pattern of the searches:
//   level   one thread per SEARCH_THREADS tile: the tile's level, or -1 across a boundary.
//   count   one thread per entry: the labels of each tile.
//   scan    two levels: one block per SEARCH_SCAN_THREADS tiles scans them in place and writes the block's sum, then one
//           block scans the block sums and writes the total.  (Up to 2^31 entries make 2^23 tiles: too many for one
//           block to walk.)
//   write   one warp per tile with labels before max_labels: a label at position < max_labels writes its level, value,
//           path and root (walking up) and its optimal set (the first child by binary search on the non-decreasing
//           h_parent).  Labels are in history order: level non-decreasing and, within a level, root non-decreasing,
//           since frontiers are in root order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "hk_minimax.cuh"
#include "hk_search.cuh"

namespace hk {

struct LabelParams {
    long long used;                  // entries of the search's history: [0, used)
    long long* tile_sum;             // [ceil(used / SEARCH_THREADS)] labels per tile, then the prefix in its scan block
    long long* block_sum;            // [ceil(tiles / SEARCH_SCAN_THREADS)] labels per scan block, then the prefix
    long long* total;                // [1] the number of labels
    int32_t* tile_level;             // [tiles] the level of every entry of the tile, -1 across a level boundary
    long long max_labels;            // labels written: those at positions < max_labels
    int max_depth;                   // row length of mask and axis
    int32_t* root;                   // [max_labels]
    int32_t* level;                  // [max_labels]
    int32_t* value;                  // [max_labels]
    unsigned long long* optimal;     // [max_labels] bit g: the group of action id g is fully solved
    int32_t* mask;                   // [max_labels, max_depth] the path from the root; 0 past the label's level
    int32_t* axis;                   // [max_labels, max_depth]; -1 past the label's level
};

// the level of entry h: the parent hops up to its root
__device__ __forceinline__ int label_level(const ValueParams& p, long long h) {
    int l = 0;
    for (int32_t a = p.h_parent[h]; a >= 0; a = p.h_parent[a]) ++l;
    return l;
}

// one thread per tile: the level of every entry of the tile, or -1 when it straddles a level boundary.  Levels follow
// each other in the history, so one walk from the tile's first entry and one from its last decide it.
__global__ void hk_label_level_kernel(const ValueParams p, const LabelParams q, long long tiles) {
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < tiles; t += (long long)gridDim.x * blockDim.x) {
        const long long first = t * SEARCH_THREADS;
        const long long last = first + SEARCH_THREADS - 1 < q.used ? first + SEARCH_THREADS - 1 : q.used - 1;
        const int a = label_level(p, first);
        q.tile_level[t] = a == label_level(p, last) ? a : -1;
    }
}

// whether entry h is a label, and its level when it is; `tile` is its tile's tile_level
__device__ __forceinline__ bool label_at(const ValueParams& p, long long h, int tile, int* level) {
    const int32_t s = p.h_solved[h];
    if (s <= 0) return false;  // unsolved, or an ended root (round 0, level 0)
    *level = tile >= 0 ? tile : label_level(p, h);
    return s > *level;
}

__global__ void __launch_bounds__(SEARCH_THREADS) hk_label_count_kernel(const ValueParams p, const LabelParams q) {
    const long long h = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
    const int tile = q.tile_level[blockIdx.x];
    int l;
    const int n = __syncthreads_count(h < q.used && label_at(p, h, tile, &l));
    if (threadIdx.x == 0) q.tile_sum[blockIdx.x] = n;
}

// one block per SEARCH_SCAN_THREADS tiles: the exclusive prefix of each tile within its block, and the block's sum
__global__ void __launch_bounds__(SEARCH_SCAN_THREADS) hk_label_scan_tiles_kernel(const LabelParams q, long long tiles) {
    __shared__ long long ws[32];
    const long long t = (long long)blockIdx.x * SEARCH_SCAN_THREADS + threadIdx.x;
    const long long v = t < tiles ? q.tile_sum[t] : 0;
    long long tot;
    const long long ex = search_block_scan(v, ws, &tot);
    if (t < tiles) q.tile_sum[t] = ex;
    if (threadIdx.x == 0) q.block_sum[blockIdx.x] = tot;
}

// one block: the exclusive prefix of the block sums, and the total
__global__ void __launch_bounds__(SEARCH_SCAN_THREADS) hk_label_scan_blocks_kernel(const LabelParams q, long long blocks) {
    __shared__ long long ws[32];
    long long carry = 0;
    for (long long start = 0; start < blocks; start += SEARCH_SCAN_THREADS) {
        const long long j = start + threadIdx.x;
        const long long v = j < blocks ? q.block_sum[j] : 0;
        long long tot;
        const long long ex = search_block_scan(v, ws, &tot);
        if (j < blocks) q.block_sum[j] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) *q.total = carry;
}

// label k: entry h of level l
__device__ __forceinline__ void label_write(const ValueParams& p, const LabelParams& q, long long h, int l, long long k) {
    q.level[k] = l;
    q.value[k] = p.h_solved[h] - l;
    // the path: the move that made each state on the way up, from position l - 1 down to 0
    int32_t* mask = q.mask + k * q.max_depth;
    int32_t* axis = q.axis + k * q.max_depth;
    long long e = h;
    for (int t = l - 1; t >= 0; --t) {
        const int S = p.h_mask[e];
        unsigned m = (unsigned)S;
        for (int j = p.h_rank[e]; j > 0; --j) m &= m - 1;
        mask[t] = S;
        axis[t] = __ffs((int)m) - 1;
        e = p.h_parent[e];
    }
    q.root[k] = (int32_t)e;
    for (int t = l; t < q.max_depth; ++t) {
        mask[t] = 0;
        axis[t] = -1;
    }
    // the first child of h: the lower bound of h in the non-decreasing h_parent; then each group's first child
    long long lo = h + 1, hi = q.used;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (p.h_parent[mid] < h) lo = mid + 1;
        else hi = mid;
    }
    unsigned long long opt = 0;
    if (lo + p.children <= q.used && p.h_parent[lo] == h) {  // otherwise an empty set rather than a read past the history
        int g = 0;
        for (int j = 0; j < p.children; j += __popc(p.pair[j] & 63), ++g)
            if (p.h_rem[lo + j] == 0) opt |= 1ull << g;
    }
    q.optimal[k] = opt;
}

// one warp per tile with labels before max_labels, 32 entries at a time
__global__ void __launch_bounds__(SEARCH_THREADS) hk_label_write_kernel(const ValueParams p, const LabelParams q,
                                                                        long long tiles) {
    const long long t = (long long)blockIdx.x * (SEARCH_THREADS / 32) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (t >= tiles) return;
    long long k = q.block_sum[t / SEARCH_SCAN_THREADS] + q.tile_sum[t];
    const long long next = t + 1 < tiles ? q.block_sum[(t + 1) / SEARCH_SCAN_THREADS] + q.tile_sum[t + 1] : *q.total;
    if (k == next || k >= q.max_labels) return;  // no label in the tile, or all past the truncation
    const int tile = q.tile_level[t];
    const long long end = (t + 1) * SEARCH_THREADS < q.used ? (t + 1) * SEARCH_THREADS : q.used;
    for (long long h0 = t * SEARCH_THREADS; h0 < end && k < q.max_labels; h0 += 32) {
        const long long h = h0 + lane;
        int l = 0;
        const bool is = h < end && label_at(p, h, tile, &l);
        const unsigned bits = __ballot_sync(0xffffffffu, is);
        const long long pos = k + __popc(bits & ((1u << lane) - 1));
        k += __popc(bits);
        if (is && pos < q.max_labels) label_write(p, q, h, l, pos);
    }
}

}  // namespace hk
