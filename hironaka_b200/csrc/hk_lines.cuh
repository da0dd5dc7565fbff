// hk_lines.cuh — lines of play from the game-tree searches (hk_search_depth_line, hk_search_value_line): the kernels
// that keep a small history during hk_search_depth's level loop and walk it at the end, and the walk down
// hk_search_value's history.  They only read what the search kernels of hk_search.cuh and hk_minimax.cuh leave; none of
// those kernels changes.
//
// Depth line.  Every node of every level has an entry in a history the batch shares: the parent's entry (-1 for a
// root), and the set and axis the parent played to make it.  The set takes 16 bits, since the depth search takes d up to
// HK_MAX_DIM.  Level L fills [hist_base, hist_base + M), the roots are entries 0..B-1, as in hk_search_value.  Per level:
//   deep    one thread per frontier node: the first node of each root stores its entry in deep[root].  A frontier is in
//           lexicographic order of the axis sequences that lead to it (children are made in increasing axis order and
//           stay in parent order), so after the last level a root reaches, deep[root] ends the smallest of its deepest
//           lines.
//   history one thread per node, after hk_search_scatter_kernel: the node's children get their entries, at the
//           positions the scatter used (the scanned tile prefix, the prefix of the counts in the tile, the root's shift).
//   the history cut: the level loop passes min(capacity, history room) to hk_search_decide_kernel as the capacity.  When
//           the room is the smaller, hk_line_save_kernel keeps each root's children before the decide kernel zeroes
//           them, and hk_line_relabel_kernel gives the roots that decide kernel cut the status hk_search_value's rules
//           give: CAPACITY if the candidates up to the root pass `capacity`, HISTORY otherwise.
// At the end one thread per root walks up from deep[root] and writes the moves from the last to the first.
//
// Value line.  One thread per resolved root walks down hk_search_value's history.  h_parent is non-decreasing over the
// history (children are placed in parent order, levels follow each other), so a state's children, one block of
// d*2^(d-1) - d entries grouped by S in increasing order, are found by binary search.  Every state of the line is
// solved in the root's round R: the host plays the first group whose children are all solved by R, the agent the
// lowest-rank child solved in R.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/hironaka_b200.h"
#include "hk_minimax.cuh"
#include "hk_search.cuh"

namespace hk {

struct LineParams {
    long long hist_base;    // history entry of this frontier's first node
    long long hist_used;    // entries of levels 0..level; the next level's first entry
    int32_t* h_parent;      // [history] parent's entry, -1 for a root
    uint16_t* h_set;        // [history] the set the parent played
    uint8_t* h_axis;        // [history] the axis the parent played
    int32_t* deep;          // [B] entry of the first node of the root's deepest level so far
    long long* root_ch;     // [B] children of the root at this level (hk_line_save_kernel)
    long long capacity;     // the caller's frontier capacity (the decide kernel may get less)
};

__global__ void __launch_bounds__(SEARCH_THREADS) hk_line_deep_kernel(const SearchParams p, const LineParams l) {
    const long long i = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
    if (i >= p.M) return;
    const int r = search_root(p, i);
    if (i == 0 || search_root(p, i - 1) != r) l.deep[r] = (int32_t)(l.hist_base + i);
}

__global__ void __launch_bounds__(SEARCH_THREADS) hk_line_history_kernel(const SearchParams p, const LineParams l) {
    __shared__ int warp_tot[SEARCH_THREADS / 32];
    const long long i = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int c = 0, r = 0;
    if (i < p.M) {
        c = p.count[i];
        r = search_root(p, i);
    }
    // the raw position of this node's first child, as hk_search_scatter_kernel computes it
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (c == 0) return;
    const long long shift = p.root_shift[r];
    if (shift == SEARCH_DROPPED) return;
    int before = 0;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    const long long pos = p.tile_sum[blockIdx.x] + before + incl - c + shift;
    const int32_t parent = (int32_t)(l.hist_base + i);
    for (int j = 0; j < c; ++j) {
        const long long h = l.hist_used + pos + j;
        l.h_parent[h] = parent;
        l.h_set[h] = (uint16_t)p.child_mask[pos + j];
        l.h_axis[h] = (uint8_t)p.child_axis[pos + j];
    }
}

// before hk_search_decide_kernel, which zeroes root_children: the children of every root in play
__global__ void hk_line_save_kernel(const SearchParams p, const LineParams l) {
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < p.n_active; j += (long long)gridDim.x * blockDim.x) {
        const int r = p.active[j];
        l.root_ch[r] = (long long)p.root_children[r];
    }
}

// after hk_search_decide_kernel ran with the history room as its capacity: the candidates (kept roots and roots it cut
// with CAPACITY) in root order; a cut root stays CAPACITY only if the candidates up to it pass the caller's capacity
__global__ void __launch_bounds__(SEARCH_SCAN_THREADS) hk_line_relabel_kernel(const SearchParams p, const LineParams l) {
    __shared__ long long ws[32];
    long long carry = 0;
    for (long long start = 0; start < p.n_active; start += SEARCH_SCAN_THREADS) {
        const long long j = start + threadIdx.x;
        const bool in = j < p.n_active;
        const int r = in ? p.active[j] : 0;
        const bool cut = in && p.status[r] == HK_SEARCH_CAPACITY;
        const bool cand = cut || (in && p.root_shift[r] != SEARCH_DROPPED);
        const long long ch = cand ? l.root_ch[r] : 0;
        long long tot;
        const long long end = carry + search_block_scan(ch, ws, &tot) + ch;
        carry += tot;
        if (cut && end <= l.capacity) p.status[r] = HK_SEARCH_HISTORY;
    }
}

// one thread per root: the moves from deep[root] up to the root, written from position depth - 1 down to 0; mask 0 and
// axis -1 past the line's end
__global__ void hk_line_depth_walk_kernel(const int32_t* depth, const LineParams l, int32_t* line_mask,
                                          int32_t* line_axis, long long B, int max_depth) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < B; r += (long long)gridDim.x * blockDim.x) {
        int32_t* mask = line_mask + r * max_depth;
        int32_t* axis = line_axis + r * max_depth;
        const int n = depth[r];
        for (int t = n; t < max_depth; ++t) {
            mask[t] = 0;
            axis[t] = -1;
        }
        int32_t h = l.deep[r];
        for (int t = n - 1; t >= 0; --t) {
            mask[t] = l.h_set[h];
            axis[t] = l.h_axis[h];
            h = l.h_parent[h];
        }
    }
}

// one thread per root: the optimal line of a resolved root (hk_search_value's history of `used` entries, after
// hk_value_finish_kernel); an empty line for any other root.  A state on the line always has a group first won in the
// root's round, with a child solved in that round; should the history ever say otherwise, the line is left empty
// rather than read past it.
__global__ void hk_line_value_walk_kernel(const ValueParams p, long long used, int32_t* line_mask, int32_t* line_axis,
                                          int max_depth) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < p.B; r += (long long)gridDim.x * blockDim.x) {
        int32_t* mask = line_mask + r * max_depth;
        int32_t* axis = line_axis + r * max_depth;
        const int32_t round = p.h_solved[r];
        int n = p.status[r] == HK_SEARCH_RESOLVED && round != VALUE_UNSOLVED ? round : 0;
        long long h = r;
        for (int t = 0; t < n; ++t) {
            // the first child of h: the lower bound of h in the non-decreasing h_parent
            long long lo = p.B, hi = used;
            while (lo < hi) {
                const long long mid = (lo + hi) >> 1;
                if (p.h_parent[mid] < h) lo = mid + 1;
                else hi = mid;
            }
            // the first group whose children are all solved by `round`, then its lowest-rank child solved in `round`
            long long pick = -1;
            for (int j = 0; j < p.children && pick < 0 && lo + p.children <= used && p.h_parent[lo] == h;) {
                const int S = p.pair[j] & 63, size = __popc(S);
                bool won = true;
                for (int k = 0; k < size; ++k) {
                    const int32_t s = p.h_solved[lo + j + k];
                    won &= s != VALUE_UNSOLVED && s <= round;
                }
                if (won)
                    for (int k = 0; k < size && pick < 0; ++k)
                        if (p.h_solved[lo + j + k] == round) pick = lo + j + k;
                j += size;
            }
            if (pick < 0) {
                n = 0;
                break;
            }
            const int e = p.pair[pick - lo];
            mask[t] = e & 63;
            axis[t] = (e >> 6) & 7;
            h = pick;
        }
        for (int t = n; t < max_depth; ++t) {
            mask[t] = 0;
            axis[t] = -1;
        }
    }
}

}  // namespace hk
