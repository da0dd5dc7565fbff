// hk_search.cuh — the bookkeeping kernels of the level-by-level game-tree search (hk_search_depth).
//
// One level of the search takes a frontier of nodes (int32 states [M, N, d], each with the index of its root; the
// nodes of a root are contiguous and the roots appear in increasing order) and the host's coordinate set of every
// node (hk_host_policy), and writes the next frontier: one child per axis of the set, in increasing axis order, as a
// copy of the parent with the (set, axis) that hk_step then plays on it in place.  Three launches, the
// count -> one-block scan -> scatter pattern of hk_experience.cuh:
//   count   one thread per node: 0 children for an ended node (<= 1 live row, hk_step's done rule), popcount(set)
//           otherwise; per-root sums of the counts and flags (int32 bound, open node at the depth limit) by
//           warp-aggregated atomics (integer sums: the same whatever the order), per-tile sums of the counts.
//   decide  one block: the exclusive scan of the tile sums, then over the roots still in play, in root order, the
//           cuts (int32 bound, node budget, frontier capacity: in that order) and the per-root bookkeeping.  The roots
//           that go on form the next level's root list; the number of children and of such roots is what the host
//           reads back.
//   scatter one thread per node places its children; one warp per node copies the parent's rows once per child.
// Nothing here depends on the launch geometry: positions come from prefix sums in node order, and the capacity cut
// drops roots from the highest index down.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace hk {

constexpr int SEARCH_THREADS = 256;  // nodes per tile of the count and scatter kernels
constexpr int SEARCH_SCAN_THREADS = 1024;

// per-root flags raised by the count kernel
constexpr int SEARCH_FLAG_BOUND = 1;  // a node to expand has a live entry >= floor(2^30 / d)
constexpr int SEARCH_FLAG_OPEN = 2;   // a node at the depth limit has not ended

constexpr long long SEARCH_DROPPED = -(1ll << 62);  // root_shift of a root whose children are not added

struct SearchParams {
    const int32_t* state;      // [M, N, d] frontier of this level
    const int32_t* node_root;  // [M] root of each node; nullptr at level 0 (node i is root i)
    const int32_t* policy;     // [M] host's coordinate set of each node (read when expand != 0)
    long long M;
    int N, d;
    int level;                 // depth of this frontier
    int expand;                // 0 at level max_depth: nodes are not expanded, open ones stop their root
    int32_t bound;             // floor(2^30 / d)
    long long max_nodes, capacity;
    uint8_t* count;            // [M] children of each node
    long long* tile_sum;       // [ceil(M / SEARCH_THREADS)] children per tile; the decide kernel scans it in place
    unsigned long long* root_children;  // [B] children per root at this level (zeroed again by the decide kernel)
    int32_t* root_flag;        // [B] SEARCH_FLAG_* (zeroed again by the decide kernel)
    long long* root_shift;     // [B] next-frontier position of a child = raw prefix + shift, or SEARCH_DROPPED
    const int32_t* active;     // [n_active] the roots with nodes in this frontier, in increasing order
    int32_t* active_next;      // the roots with nodes in the next frontier
    long long n_active;
    long long* counters;       // [2] out: children in the next frontier, roots in play at the next level
    int32_t* depth;            // [B] results
    long long* nodes;
    int8_t* status;
    // next frontier (scatter)
    int32_t* child_state;      // [capacity, N, d]
    int32_t* child_root;       // [capacity]
    int32_t* child_mask;       // [capacity] the parent's coordinate set
    int32_t* child_axis;       // [capacity] the axis this child plays
};

__global__ void hk_search_init_kernel(int32_t* depth, long long* nodes, int8_t* status, int32_t* active, long long B) {
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < B; r += (long long)gridDim.x * blockDim.x) {
        depth[r] = 0;
        nodes[r] = 1;
        status[r] = 0;
        active[r] = (int32_t)r;
    }
}

__device__ __forceinline__ int search_root(const SearchParams& p, long long i) {
    return p.node_root ? p.node_root[i] : (int)i;
}

__global__ void __launch_bounds__(SEARCH_THREADS) hk_search_count_kernel(const SearchParams p) {
    const long long i = (long long)blockIdx.x * SEARCH_THREADS + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int r = -1, c = 0, flag = 0;
    if (i < p.M) {
        r = search_root(p, i);
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
            if (!p.expand) flag = SEARCH_FLAG_OPEN;
            else {
                c = __popc((unsigned)p.policy[i]);
                if (big) flag = SEARCH_FLAG_BOUND;
            }
        }
        p.count[i] = (uint8_t)c;
    }
    // the nodes of a root are contiguous: one atomic per root and warp
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

// exclusive scan of one value per thread over a block of SEARCH_SCAN_THREADS threads; *total gets the block's sum.
// Every thread of the block calls it; `ws` is 32 words of shared memory.
__device__ __forceinline__ long long search_block_scan(long long v, long long* ws, long long* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long u = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += u;
    }
    if (lane == 31) ws[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        long long w = ws[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += u;
        }
        ws[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const long long excl = (warp ? ws[warp - 1] : 0) + incl - v;
    *total = ws[31];
    __syncthreads();  // ws is reused by the next call
    return excl;
}

// exclusive scan in place of the tile sums of a frontier of M nodes: the raw position (before any cut) of each tile's
// first child.  Every thread of a SEARCH_SCAN_THREADS block calls it.
__device__ __forceinline__ void search_scan_tiles(long long* tile_sum, long long M, long long* ws) {
    const long long tiles = (M + SEARCH_THREADS - 1) / SEARCH_THREADS;
    long long carry = 0;
    for (long long start = 0; start < tiles; start += SEARCH_SCAN_THREADS) {
        const long long t = start + threadIdx.x;
        const long long v = t < tiles ? tile_sum[t] : 0;
        long long tot;
        const long long ex = search_block_scan(v, ws, &tot);
        if (t < tiles) tile_sum[t] = carry + ex;
        carry += tot;
    }
}

__global__ void __launch_bounds__(SEARCH_SCAN_THREADS) hk_search_decide_kernel(const SearchParams p) {
    __shared__ long long ws[32];
    __shared__ unsigned long long kept_total;
    if (threadIdx.x == 0) kept_total = 0;
    // 1. the raw position of each tile's first child
    search_scan_tiles(p.tile_sum, p.M, ws);
    // 2. the roots in play, in increasing order: cuts int32 bound -> node budget -> capacity
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
        int8_t st = 0;
        bool cand = false;
        if (in) {
            if (flag & SEARCH_FLAG_OPEN) st = 1;
            else if (ch > 0) {
                if (flag & SEARCH_FLAG_BOUND) st = 4;
                else if (p.nodes[r] + ch > p.max_nodes) st = 2;
                else cand = true;
            }
        }
        long long tot;
        const long long raw_ex = search_block_scan(ch, ws, &tot);
        const long long raw_off = raw_carry + raw_ex;
        raw_carry += tot;
        // the candidates that fit form a prefix in root order: dropping from the highest index down stops there
        const long long kept_ex = search_block_scan(cand ? ch : 0, ws, &tot);
        const long long kept_off = kept_carry + kept_ex;
        kept_carry += tot;
        const bool keep = cand && kept_off + ch <= p.capacity;
        if (cand && !keep) st = 3;
        const long long next_ex = search_block_scan(keep ? 1 : 0, ws, &tot);
        if (in) {
            if (st) p.status[r] = st;
            if (keep) {
                atomicAdd(&kept_total, (unsigned long long)ch);
                p.nodes[r] += ch;
                p.depth[r] = p.level + 1;
                p.active_next[next_carry + next_ex] = r;
                p.root_shift[r] = kept_off - raw_off;
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

__global__ void __launch_bounds__(SEARCH_THREADS) hk_search_scatter_kernel(const SearchParams p) {
    __shared__ long long ws_pos[SEARCH_THREADS];
    __shared__ int32_t ws_c[SEARCH_THREADS];
    __shared__ int warp_tot[SEARCH_THREADS / 32];
    const long long base = (long long)blockIdx.x * SEARCH_THREADS;
    const long long i = base + threadIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int c = 0, r = 0;
    if (i < p.M) {
        c = p.count[i];
        r = search_root(p, i);
    }
    // raw position of this node's first child: tile offset + prefix of the counts inside the tile
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
    if (pos >= 0) {
        const uint32_t set = (uint32_t)p.policy[i];
        uint32_t m = set;
        for (int j = 0; j < c; ++j) {
            const int a = __ffs((int)m) - 1;
            m &= m - 1;
            p.child_root[pos + j] = r;
            p.child_mask[pos + j] = (int32_t)set;
            p.child_axis[pos + j] = a;
        }
    }
    ws_pos[threadIdx.x] = pos;
    ws_c[threadIdx.x] = c;
    __syncthreads();
    // the rows: one warp per node, coalesced, the parent read once for all its children
    const int words = p.N * p.d;
    for (int k = warp; k < SEARCH_THREADS; k += SEARCH_THREADS / 32) {
        const long long dst0 = ws_pos[k];
        if (dst0 < 0) continue;
        const int cc = ws_c[k];
        const int32_t* src = p.state + (base + k) * words;
        for (int w = lane; w < words; w += 32) {
            const int32_t v = src[w];
            for (int j = 0; j < cc; ++j) p.child_state[(dst0 + j) * words + w] = v;
        }
    }
}

}  // namespace hk
