// hk_minimax.cuh — the kernels of the game-value search (hk_search_value): the fewest moves the best host needs to end
// the game, whatever the agent replies, found level by level.
//
// A frontier is as in hk_search.cuh: int32 states [M, N, d], each with its root, the nodes of a root contiguous and the
// roots in increasing order.  Every node of every level also has an entry in the history, which the whole batch shares
// and which level L fills at [hist_base, hist_base + M).  The roots are entries 0..B-1.  An entry holds the parent's
// entry (-1 for a root), the coordinate set S of the node's group (the children of the parent for one S), the node's
// rank in its group (the group's first child is entry h - rank), the unsolved children of the group (kept at the
// group's first child) and the round in which the node was solved (VALUE_UNSOLVED before).
//
// One level is four launches and then hk_step in place on the children:
//   solve   one thread per node: an ended node (<= 1 live row) is solved in this round, and its thread walks up.  It
//           takes one from its group's count with atomicSub; the thread that empties a group has won it for the
//           parent: it lowers the root's best set with atomicMin when the parent is a root, and solves the parent with
//           atomicCAS.  The thread whose CAS succeeds walks on from the parent.  So each newly solved node is handled
//           once, by one thread: the work follows the nodes that change, not the history.  It also records each
//           node's kind (ended, open, open with a live entry past the int32 bound) for the count kernel.
//   count   one thread per node: d*2^(d-1) - d children (one per (S, axis), S over the sets with |S| >= 2 in
//           increasing order, the axes of S in increasing order) for an open node none of whose ancestors is solved
//           (the parent chain is walked), 0 otherwise; the per-root and per-tile sums of hk_search_count_kernel.
//   decide  one block: the cuts of hk_search_decide_kernel over the roots in play, in root order, after the solved
//           roots leave: int32 bound, node budget, frontier capacity, then the history.
//   scatter one warp per node writes its children's (S, axis), history entries and rows.
// Which thread solves a node depends on timing; which nodes are solved, in which round, and the minimum over the won
// sets do not (integer counts, CAS from one value to the round, min).  Positions come from prefix sums in node order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/hironaka_b200.h"
#include "hk_search.cuh"

namespace hk {

constexpr int VALUE_MAX_CHILDREN = 186;           // d = 6: the sum of |S| over the 57 sets with |S| >= 2
constexpr int32_t VALUE_UNSOLVED = -1;            // solved round of a node not solved yet
constexpr int32_t VALUE_NO_SET = 0x7fffffff;      // a root's best set before one of its groups is won

// kind of a frontier node, written by the solve kernel
constexpr uint8_t VALUE_ENDED = 0;
constexpr uint8_t VALUE_OPEN = 1;
constexpr uint8_t VALUE_OPEN_BIG = 2;  // open, with a live entry >= floor(2^30 / d)

struct ValueParams {
    const int32_t* state;      // [M, N, d] frontier of this level
    const int32_t* node_root;  // [M] root of each node; nullptr at level 0 (node i is root i)
    long long M, B;
    int N, d;
    int level;                 // depth of this frontier, and the round the solve kernel runs
    int expand;                // 0 at level max_depth: nodes are not expanded, open ones stop their root
    int32_t bound;             // floor(2^30 / d)
    int children;              // children of an expanded node
    long long max_nodes, capacity, history;
    long long hist_base;       // history entry of this frontier's first node
    long long hist_used;       // entries of levels 0..level; the next level's first entry
    uint16_t pair[VALUE_MAX_CHILDREN];  // child j plays S = pair & 63 and axis (pair >> 6) & 7, rank pair >> 9 in S
    uint8_t* kind;             // [M] VALUE_ENDED / VALUE_OPEN / VALUE_OPEN_BIG
    uint8_t* count;            // [M] children of each node
    long long* tile_sum;       // [ceil(M / SEARCH_THREADS)] children per tile; the decide kernel scans it in place
    unsigned long long* root_children;  // [B] children per root at this level (zeroed again by the decide kernel)
    int32_t* root_flag;        // [B] SEARCH_FLAG_* (zeroed again by the decide kernel)
    long long* root_shift;     // [B] next-frontier position of a child = raw prefix + shift, or SEARCH_DROPPED
    const int32_t* active;     // [n_active] the roots with nodes in this frontier, in increasing order
    int32_t* active_next;      // the roots with nodes in the next frontier
    long long n_active;
    long long* counters;       // [2] out: children in the next frontier, roots in play at the next level
    int32_t* value;            // [B] results
    int32_t* best_mask;        // [B] VALUE_NO_SET, lowered by the solve kernel; hk_value_finish_kernel sets the result
    long long* nodes;
    int8_t* status;
    // history [history]
    int32_t* h_parent;
    int32_t* h_solved;
    int32_t* h_rem;
    uint8_t* h_mask;
    uint8_t* h_rank;
    // next frontier (scatter)
    int32_t* child_state;      // [capacity, N, d]
    int32_t* child_root;       // [capacity]
    int32_t* child_mask;       // [capacity] S
    int32_t* child_axis;       // [capacity] the axis this child plays
};

__global__ void hk_value_init_kernel(const ValueParams p, int32_t* active) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < p.B; r += (long long)gridDim.x * blockDim.x) {
        p.value[r] = 0;
        p.best_mask[r] = VALUE_NO_SET;
        p.nodes[r] = 1;
        p.status[r] = HK_SEARCH_RESOLVED;
        p.h_parent[r] = -1;
        p.h_solved[r] = VALUE_UNSOLVED;
        active[r] = (int32_t)r;
    }
}

// best_mask: the smallest won set of a resolved root, 0 for a root that had already ended, -1 for a root not resolved
__global__ void hk_value_finish_kernel(const ValueParams p) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < p.B; r += (long long)gridDim.x * blockDim.x) {
        const int32_t b = p.best_mask[r];
        p.best_mask[r] = p.h_solved[r] == VALUE_UNSOLVED ? -1 : b == VALUE_NO_SET ? 0 : b;
    }
}

__device__ __forceinline__ int value_root(const ValueParams& p, long long i) {
    return p.node_root ? p.node_root[i] : (int)i;
}

__global__ void __launch_bounds__(SEARCH_THREADS) hk_value_solve_kernel(const ValueParams p) {
    const long long i = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
    if (i >= p.M) return;
    const int32_t* x = p.state + i * p.N * p.d;
    int live = 0;
    bool big = false;
    for (int row = 0; row < p.N; ++row) {
        const int32_t* q = x + row * p.d;
        if (q[0] < 0) continue;
        ++live;
        for (int k = 0; k < p.d; ++k) big |= q[k] >= p.bound;
    }
    if (live > 1) {
        p.kind[i] = big ? VALUE_OPEN_BIG : VALUE_OPEN;
        return;
    }
    p.kind[i] = VALUE_ENDED;
    // no node below this level exists yet, so nothing else writes this node's round
    long long h = p.hist_base + i;
    p.h_solved[h] = p.level;
    for (;;) {
        const int32_t par = p.h_parent[h];
        if (par < 0) break;
        if (atomicSub(&p.h_rem[h - p.h_rank[h]], 1) != 1) break;  // the group still has an unsolved child
        if (par < p.B) atomicMin(&p.best_mask[par], (int32_t)p.h_mask[h]);
        if (atomicCAS(&p.h_solved[par], VALUE_UNSOLVED, p.level) != VALUE_UNSOLVED) break;  // won before in this round
        h = par;
    }
}

__global__ void __launch_bounds__(SEARCH_THREADS) hk_value_count_kernel(const ValueParams p) {
    const long long i = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int r = -1, c = 0, flag = 0;
    if (i < p.M) {
        r = value_root(p, i);
        const uint8_t k = p.kind[i];
        bool pruned = k == VALUE_ENDED;
        for (int32_t a = p.h_parent[p.hist_base + i]; a >= 0 && !pruned; a = p.h_parent[a]) pruned = p.h_solved[a] != VALUE_UNSOLVED;
        if (!pruned) {
            if (!p.expand) flag = SEARCH_FLAG_OPEN;
            else {
                c = p.children;
                if (k == VALUE_OPEN_BIG) flag = SEARCH_FLAG_BOUND;
            }
        }
        p.count[i] = (uint8_t)c;
    }
    // the sums of hk_search_count_kernel (which keeps its own copy, and so its machine code)
    const unsigned grp = __match_any_sync(0xffffffffu, r);
    const int sum = __reduce_add_sync(grp, c);
    const int any = __reduce_or_sync(grp, flag);
    if (r >= 0 && lane == __ffs((int)grp) - 1) {
        if (sum) atomicAdd(&p.root_children[r], (unsigned long long)sum);
        if (any) atomicOr(&p.root_flag[r], any);
    }
    __shared__ int red[SEARCH_THREADS / 32];
    const int wsum = __reduce_add_sync(0xffffffffu, c);
    if (lane == 0) red[threadIdx.x >> 5] = wsum;
    __syncthreads();
    if (threadIdx.x == 0) {
        long long t = 0;
#pragma unroll
        for (int w = 0; w < SEARCH_THREADS / 32; ++w) t += red[w];
        p.tile_sum[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(SEARCH_SCAN_THREADS) hk_value_decide_kernel(const ValueParams p) {
    __shared__ long long ws[32];
    __shared__ unsigned long long kept_total;
    if (threadIdx.x == 0) kept_total = 0;
    search_scan_tiles(p.tile_sum, p.M, ws);
    // the roots in play, in increasing order: solved roots leave; cuts int32 bound -> node budget -> capacity -> history
    long long raw_carry = 0, kept_carry = 0, next_carry = 0;
    for (long long start = 0; start < p.n_active; start += SEARCH_SCAN_THREADS) {
        const long long j = start + threadIdx.x;
        const bool in = j < p.n_active;
        const int r = in ? p.active[j] : 0;
        long long ch = 0;
        int flag = 0;
        if (in) {
            ch = (long long)p.root_children[r];
            flag = p.root_flag[r];
            p.root_children[r] = 0;
            p.root_flag[r] = 0;
        }
        int8_t st = HK_SEARCH_RESOLVED;
        bool cand = false;
        if (in) {
            p.value[r] = p.level;  // this round is done: the value, or the level the true value lies beyond
            // a solved root has no children: the root itself is a solved ancestor of every node of its frontier
            if (p.h_solved[r] != VALUE_UNSOLVED) {
            } else if (flag & SEARCH_FLAG_OPEN) st = HK_SEARCH_MAX_DEPTH;
            else if (ch > 0) {
                if (flag & SEARCH_FLAG_BOUND) st = HK_SEARCH_INT32_BOUND;
                else if (p.nodes[r] + ch > p.max_nodes) st = HK_SEARCH_MAX_NODES;
                else cand = true;
            }
        }
        long long tot;
        const long long raw_ex = search_block_scan(ch, ws, &tot);
        const long long raw_off = raw_carry + raw_ex;
        raw_carry += tot;
        // the candidates that fit form a prefix in root order: dropping from the highest index down stops there
        const long long kept_ex = search_block_scan(cand ? ch : 0, ws, &tot);
        const long long kept_end = kept_carry + kept_ex + ch;
        kept_carry += tot;
        const bool keep = cand && kept_end <= p.capacity && p.hist_used + kept_end <= p.history;
        if (cand && !keep) st = kept_end > p.capacity ? HK_SEARCH_CAPACITY : HK_SEARCH_HISTORY;
        const long long next_ex = search_block_scan(keep ? 1 : 0, ws, &tot);
        if (in) {
            if (st) p.status[r] = st;
            if (keep) {
                atomicAdd(&kept_total, (unsigned long long)ch);
                p.nodes[r] += ch;
                p.active_next[next_carry + next_ex] = r;
                p.root_shift[r] = kept_end - ch - raw_off;
            } else {
                p.root_shift[r] = SEARCH_DROPPED;
            }
        }
        next_carry += tot;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        p.counters[0] = (long long)kept_total;
        p.counters[1] = next_carry;
    }
}

__global__ void __launch_bounds__(SEARCH_THREADS) hk_value_scatter_kernel(const ValueParams p) {
    __shared__ long long ws_pos[SEARCH_THREADS];
    __shared__ int32_t ws_root[SEARCH_THREADS];
    __shared__ int warp_tot[SEARCH_THREADS / 32];
    __shared__ uint16_t pair[VALUE_MAX_CHILDREN];
    for (int j = threadIdx.x; j < p.children; j += SEARCH_THREADS) pair[j] = p.pair[j];
    const long long base = (long long)blockIdx.x * SEARCH_THREADS;
    const long long i = base + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int c = 0, r = 0;
    if (i < p.M) {
        c = p.count[i];
        r = value_root(p, i);
    }
    // raw position of this node's first child: tile offset + prefix of the counts inside the tile (as
    // hk_search_scatter_kernel)
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    int before = 0;
    for (int w = 0; w < warp; ++w) before += warp_tot[w];
    long long pos = -1;
    if (c > 0) {
        const long long shift = p.root_shift[r];
        if (shift != SEARCH_DROPPED) pos = p.tile_sum[blockIdx.x] + before + incl - c + shift;
    }
    ws_pos[threadIdx.x] = pos;
    ws_root[threadIdx.x] = r;
    __syncthreads();
    // one warp per node: the children's pairs and history entries, then the rows, the parent read once for all
    const int words = p.N * p.d;
    const int C = p.children;
    for (int k = warp; k < SEARCH_THREADS; k += SEARCH_THREADS / 32) {
        const long long dst0 = ws_pos[k];
        if (dst0 < 0) continue;
        const int32_t parent = (int32_t)(p.hist_base + base + k);
        const int32_t root = ws_root[k];
        for (int j = lane; j < C; j += 32) {
            const int e = pair[j];
            const int S = e & 63, rank = e >> 9;
            const long long q = dst0 + j, h = p.hist_used + q;
            p.child_root[q] = root;
            p.child_mask[q] = S;
            p.child_axis[q] = (e >> 6) & 7;
            p.h_parent[h] = parent;
            p.h_solved[h] = VALUE_UNSOLVED;
            p.h_mask[h] = (uint8_t)S;
            p.h_rank[h] = (uint8_t)rank;
            if (rank == 0) p.h_rem[h] = __popc(S);
        }
        const int32_t* src = p.state + (base + k) * words;
        for (int w = lane; w < words; w += 32) {
            const int32_t v = src[w];
            for (int j = 0; j < C; ++j) p.child_state[(dst0 + j) * words + w] = v;
        }
    }
}

}  // namespace hk
