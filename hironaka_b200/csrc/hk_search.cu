// hk_search.cu — hk_search_workspace_bytes and hk_search_depth, hk_search_value_workspace_bytes and hk_search_value,
// their line forms hk_search_depth_line_workspace_bytes, hk_search_depth_line and hk_search_value_line, and the value
// labels hk_search_value_labels_workspace_bytes and hk_search_value_labels (include/hironaka_b200.h): the level loops
// of the game-tree searches.  Every level of hk_search_depth runs hk_host_policy on the frontier and the three
// bookkeeping kernels of hk_search.cuh; every level of hk_search_value runs the four kernels of hk_minimax.cuh.  Both then run hk_step in place on the children, through the same C-ABI entry
// point a caller would use, so the children are bit for bit what hk_step makes of them on either kernel family.  The
// line forms run the same loops plus the kernels of hk_lines.cuh, the value labels hk_search_value's loop plus the
// kernels of hk_labels.cuh.
#include <cuda_runtime.h>

#include <cstring>

#include "../../include/hironaka_b200.h"
#include "hk_labels.cuh"
#include "hk_lines.cuh"
#include "hk_minimax.cuh"
#include "hk_search.cuh"

namespace {

size_t align_up(size_t v) { return (v + 255) & ~(size_t)255; }

// the caller's workspace, cut into 256-byte aligned pieces (the order of hk_search_workspace_bytes)
struct SearchWorkspace {
    int32_t* frontier[2];  // [capacity, N, d] each
    int32_t* node_root[2]; // [capacity]
    int32_t* child_mask;   // [capacity]
    int32_t* child_axis;   // [capacity]
    int32_t* policy;       // [max(B, capacity)]
    uint8_t* count;        // [max(B, capacity)]
    long long* tile_sum;   // [ceil(max(B, capacity) / SEARCH_THREADS)]
    unsigned long long* root_children;  // [B]
    int32_t* root_flag;    // [B]
    long long* root_shift; // [B]
    int32_t* active[2];    // [B] each
    long long* counters;   // [2]
};

size_t carve(SearchWorkspace* w, char* base, long long B, int N, int d, long long capacity) {
    const long long P = B > capacity ? B : capacity;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* ptr = base ? base + off : nullptr;
        off += align_up(bytes);
        return ptr;
    };
    for (int k = 0; k < 2; ++k) w->frontier[k] = (int32_t*)take((size_t)capacity * N * d * 4);
    for (int k = 0; k < 2; ++k) w->node_root[k] = (int32_t*)take((size_t)capacity * 4);
    w->child_mask = (int32_t*)take((size_t)capacity * 4);
    w->child_axis = (int32_t*)take((size_t)capacity * 4);
    w->policy = (int32_t*)take((size_t)P * 4);
    w->count = (uint8_t*)take((size_t)P);
    w->tile_sum = (long long*)take((size_t)((P + hk::SEARCH_THREADS - 1) / hk::SEARCH_THREADS) * 8);
    w->root_children = (unsigned long long*)take((size_t)B * 8);
    w->root_flag = (int32_t*)take((size_t)B * 4);
    w->root_shift = (long long*)take((size_t)B * 8);
    for (int k = 0; k < 2; ++k) w->active[k] = (int32_t*)take((size_t)B * 4);
    w->counters = (long long*)take(16);
    return off;
}

// the workspace of hk_search_value (the order of hk_search_value_workspace_bytes)
struct ValueWorkspace {
    int32_t* frontier[2];  // [capacity, N, d] each
    int32_t* node_root[2]; // [capacity]
    int32_t* child_mask;   // [capacity]
    int32_t* child_axis;   // [capacity]
    uint8_t* kind;         // [max(B, capacity)]
    uint8_t* count;        // [max(B, capacity)]
    long long* tile_sum;   // [ceil(max(B, capacity) / SEARCH_THREADS)]
    unsigned long long* root_children;  // [B]
    int32_t* root_flag;    // [B]
    long long* root_shift; // [B]
    int32_t* active[2];    // [B] each
    long long* counters;   // [2]
    int32_t* h_parent;     // [history] each
    int32_t* h_solved;
    int32_t* h_rem;
    uint8_t* h_mask;
    uint8_t* h_rank;
};

size_t carve_value(ValueWorkspace* w, char* base, long long B, int N, int d, long long capacity, long long history) {
    const long long P = B > capacity ? B : capacity;
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* ptr = base ? base + off : nullptr;
        off += align_up(bytes);
        return ptr;
    };
    for (int k = 0; k < 2; ++k) w->frontier[k] = (int32_t*)take((size_t)capacity * N * d * 4);
    for (int k = 0; k < 2; ++k) w->node_root[k] = (int32_t*)take((size_t)capacity * 4);
    w->child_mask = (int32_t*)take((size_t)capacity * 4);
    w->child_axis = (int32_t*)take((size_t)capacity * 4);
    w->kind = (uint8_t*)take((size_t)P);
    w->count = (uint8_t*)take((size_t)P);
    w->tile_sum = (long long*)take((size_t)((P + hk::SEARCH_THREADS - 1) / hk::SEARCH_THREADS) * 8);
    w->root_children = (unsigned long long*)take((size_t)B * 8);
    w->root_flag = (int32_t*)take((size_t)B * 4);
    w->root_shift = (long long*)take((size_t)B * 8);
    for (int k = 0; k < 2; ++k) w->active[k] = (int32_t*)take((size_t)B * 4);
    w->counters = (long long*)take(16);
    w->h_parent = (int32_t*)take((size_t)history * 4);
    w->h_solved = (int32_t*)take((size_t)history * 4);
    w->h_rem = (int32_t*)take((size_t)history * 4);
    w->h_mask = (uint8_t*)take((size_t)history);
    w->h_rank = (uint8_t*)take((size_t)history);
    return off;
}

// the workspace of hk_search_value_labels: hk_search_value's, then the label scan (the order of
// hk_search_value_labels_workspace_bytes)
struct LabelWorkspace {
    ValueWorkspace v;
    long long* tile_sum;   // [ceil(history / SEARCH_THREADS)]
    long long* block_sum;  // [ceil(tiles / SEARCH_SCAN_THREADS)]
    long long* total;      // [1]
    int32_t* tile_level;   // [ceil(history / SEARCH_THREADS)]
};

size_t carve_labels(LabelWorkspace* w, char* base, long long B, int N, int d, long long capacity, long long history) {
    size_t off = carve_value(&w->v, base, B, N, d, capacity, history);
    auto take = [&](size_t bytes) {
        char* ptr = base ? base + off : nullptr;
        off += align_up(bytes);
        return ptr;
    };
    const long long tiles = (history + hk::SEARCH_THREADS - 1) / hk::SEARCH_THREADS;
    w->tile_sum = (long long*)take((size_t)tiles * 8);
    w->block_sum = (long long*)take((size_t)((tiles + hk::SEARCH_SCAN_THREADS - 1) / hk::SEARCH_SCAN_THREADS) * 8);
    w->total = (long long*)take(8);
    w->tile_level = (int32_t*)take((size_t)tiles * 4);
    return off;
}

// the outputs of hk_search_value_labels
struct LabelOutputs {
    long long max_labels;
    int64_t* count;  // host
    int32_t* root;
    int32_t* level;
    int32_t* value;
    uint64_t* optimal;
    int32_t* mask;
    int32_t* axis;
};

bool value_args_ok(long long B, int N, int d, long long capacity, long long history) {
    return B >= 0 && N >= 1 && d >= 2 && d <= 6 && capacity >= 1 && history >= 1 && history >= B &&
           history <= 0x7fffffffll;
}

// the workspace of hk_search_depth_line: hk_search_depth's, then the line history (the order of
// hk_search_depth_line_workspace_bytes)
struct DepthLineWorkspace {
    SearchWorkspace s;
    int32_t* h_parent;  // [history]
    uint16_t* h_set;    // [history]
    uint8_t* h_axis;    // [history]
    int32_t* deep;      // [B]
    long long* root_ch; // [B]
};

size_t carve_depth_line(DepthLineWorkspace* w, char* base, long long B, int N, int d, long long capacity,
                        long long history) {
    size_t off = carve(&w->s, base, B, N, d, capacity);
    auto take = [&](size_t bytes) {
        char* ptr = base ? base + off : nullptr;
        off += align_up(bytes);
        return ptr;
    };
    w->h_parent = (int32_t*)take((size_t)history * 4);
    w->h_set = (uint16_t*)take((size_t)history * 2);
    w->h_axis = (uint8_t*)take((size_t)history);
    w->deep = (int32_t*)take((size_t)B * 4);
    w->root_ch = (long long*)take((size_t)B * 8);
    return off;
}

bool depth_line_args_ok(long long B, int N, int d, long long capacity, long long history) {
    return B >= 0 && N >= 1 && d >= 1 && capacity >= 1 && history >= 1 && history >= B && history <= 0x7fffffffll;
}

// what the depth line adds to hk_search_depth's level loop; nullptr for hk_search_depth itself
struct DepthLine {
    DepthLineWorkspace w;
    long long history;
    int32_t* line_mask;  // [B, max_depth]
    int32_t* line_axis;  // [B, max_depth]
};

int run_search_depth(const void* roots, int32_t* depth, int64_t* nodes, int8_t* status, int64_t B, int32_t N,
                     int32_t d, uint32_t ops, uint32_t flags, int32_t max_depth, int64_t max_nodes, int64_t capacity,
                     const SearchWorkspace& w, DepthLine* line, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(w.root_children, 0, (size_t)B * 8, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(w.root_flag, 0, (size_t)B * 4, st);
    if (e == cudaSuccess && line) e = cudaMemsetAsync(line->w.h_parent, 0xff, (size_t)B * 4, st);  // roots: parent -1
    if (e != cudaSuccess) return (int)e;
    const long long root_blocks = (B + 255) / 256;
    const unsigned root_grid = (unsigned)(root_blocks > 4096 ? 4096 : root_blocks);
    hk::hk_search_init_kernel<<<root_grid, 256, 0, st>>>(depth, (long long*)nodes, status, w.active[0], B);

    hk::SearchParams p;
    memset(&p, 0, sizeof(p));
    p.N = N;
    p.d = d;
    p.bound = (int32_t)((1 << 30) / d);
    p.max_nodes = max_nodes;
    p.capacity = capacity;
    p.policy = w.policy;
    p.count = w.count;
    p.tile_sum = w.tile_sum;
    p.root_children = w.root_children;
    p.root_flag = w.root_flag;
    p.root_shift = w.root_shift;
    p.counters = w.counters;
    p.depth = depth;
    p.nodes = (long long*)nodes;
    p.status = status;
    p.child_mask = w.child_mask;
    p.child_axis = w.child_axis;
    hk::LineParams l;
    memset(&l, 0, sizeof(l));
    if (line) {
        l.h_parent = line->w.h_parent;
        l.h_set = line->w.h_set;
        l.h_axis = line->w.h_axis;
        l.deep = line->w.deep;
        l.root_ch = line->w.root_ch;
        l.capacity = capacity;
    }

    const int32_t* state = (const int32_t*)roots;
    const int32_t* node_root = nullptr;  // level 0: node i is root i
    long long M = B, n_active = B, hist_base = 0;
    for (int level = 0;; ++level) {
        const int next = level & 1;  // frontier, node-root list and root list the next level is written to
        p.state = state;
        p.node_root = node_root;
        p.M = M;
        p.level = level;
        p.expand = level < max_depth;
        p.active = w.active[level & 1];
        p.active_next = w.active[(level + 1) & 1];
        p.n_active = n_active;
        p.child_state = w.frontier[next];
        p.child_root = w.node_root[next];
        if (p.expand) {
            int rc = hk_host_policy(state, w.policy, M, N, d, HK_DTYPE_I32, flags, -1.0f, stream);
            if (rc != HK_OK) return rc;
        }
        const unsigned tiles = (unsigned)((M + hk::SEARCH_THREADS - 1) / hk::SEARCH_THREADS);
        bool history_cut = false;  // the history room, not the capacity, bounds this level
        if (line) {
            l.hist_base = hist_base;
            l.hist_used = hist_base + M;
            const long long room = line->history - l.hist_used;
            history_cut = p.expand && room < capacity;
            p.capacity = history_cut ? room : capacity;
            hk::hk_line_deep_kernel<<<tiles, hk::SEARCH_THREADS, 0, st>>>(p, l);
        }
        hk::hk_search_count_kernel<<<tiles, hk::SEARCH_THREADS, 0, st>>>(p);
        if (history_cut) {
            const long long blocks = (n_active + 255) / 256;
            hk::hk_line_save_kernel<<<(unsigned)(blocks > 4096 ? 4096 : blocks), 256, 0, st>>>(p, l);
        }
        hk::hk_search_decide_kernel<<<1, hk::SEARCH_SCAN_THREADS, 0, st>>>(p);
        if (history_cut) hk::hk_line_relabel_kernel<<<1, hk::SEARCH_SCAN_THREADS, 0, st>>>(p, l);
        long long counters[2];
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(counters, w.counters, sizeof(counters), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return (int)e;
        if (!p.expand || counters[0] == 0) break;
        hk::hk_search_scatter_kernel<<<tiles, hk::SEARCH_THREADS, 0, st>>>(p);
        if (line) hk::hk_line_history_kernel<<<tiles, hk::SEARCH_THREADS, 0, st>>>(p, l);
        e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
        int rc = hk_step(w.frontier[next], w.frontier[next], w.child_mask, w.child_axis, nullptr, nullptr, nullptr, nullptr,
                         nullptr, nullptr, counters[0], N, d, HK_DTYPE_I32, ops, 0, -1.0f, 1e8f, stream);
        if (rc != HK_OK) return rc;
        state = w.frontier[next];
        node_root = w.node_root[next];
        hist_base += M;
        M = counters[0];
        n_active = counters[1];
    }
    if (line) {
        hk::hk_line_depth_walk_kernel<<<root_grid, 256, 0, st>>>(depth, l, line->line_mask, line->line_axis, B, max_depth);
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        return (int)e;
    }
    return (int)cudaGetLastError();
}

// the checks hk_search_depth and hk_search_depth_line share; HK_OK when the arguments pass
int depth_args_error(int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t ops, uint32_t flags, int32_t max_depth,
                     int64_t max_nodes, int64_t capacity) {
    if (B < 0 || N < 1 || d < 1 || (dtype != HK_DTYPE_I32 && dtype != HK_DTYPE_F32)) return HK_ERR_BAD_ARG;
    if (hk_kernel_class(N, d) < 0) return HK_ERR_UNSUPPORTED;
    if (dtype != HK_DTYPE_I32) return HK_ERR_UNSUPPORTED;  // float32 state is not searched
    if (flags != HK_F_HOST_ZEILLINGER && flags != HK_F_HOST_ALL_COORD) return HK_ERR_BAD_ARG;
    if ((ops & (HK_OP_SHIFT | HK_OP_NEWTON)) != (HK_OP_SHIFT | HK_OP_NEWTON) ||
        (ops & ~(HK_OP_SHIFT | HK_OP_NEWTON | HK_OP_REPOSITION)))
        return HK_ERR_BAD_ARG;
    if (max_depth < 1 || max_nodes < 1 || capacity < 1) return HK_ERR_BAD_ARG;
    return HK_OK;
}

}  // namespace

extern "C" {

int64_t hk_search_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity) {
    if (B < 0 || N < 1 || d < 1 || capacity < 1) return 0;
    SearchWorkspace w;
    return (int64_t)(carve(&w, nullptr, B, N, d, capacity) + 256);  // + 256: room to align the caller's pointer
}

int hk_search_depth(const void* roots, int32_t* depth, int64_t* nodes, int8_t* status, int64_t B, int32_t N, int32_t d,
                    int32_t dtype, uint32_t ops, uint32_t flags, int32_t max_depth, int64_t max_nodes, int64_t capacity,
                    void* workspace, void* stream) {
    const int bad = depth_args_error(B, N, d, dtype, ops, flags, max_depth, max_nodes, capacity);
    if (bad != HK_OK) return bad;
    if (B == 0) return HK_OK;
    if (!roots || !depth || !nodes || !status || !workspace) return HK_ERR_BAD_ARG;
    if (((uintptr_t)roots) & 3u) return HK_ERR_ALIGN;
    SearchWorkspace w;
    carve(&w, (char*)align_up((size_t)(uintptr_t)workspace), B, N, d, capacity);
    return run_search_depth(roots, depth, nodes, status, B, N, d, ops, flags, max_depth, max_nodes, capacity, w, nullptr,
                            stream);
}

int64_t hk_search_depth_line_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity, int64_t history) {
    if (!depth_line_args_ok(B, N, d, capacity, history)) return 0;
    DepthLineWorkspace w;
    return (int64_t)(carve_depth_line(&w, nullptr, B, N, d, capacity, history) + 256);  // + 256: room to align
}

int hk_search_depth_line(const void* roots, int32_t* depth, int64_t* nodes, int8_t* status, int32_t* line_mask,
                         int32_t* line_axis, int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t ops,
                         uint32_t flags, int32_t max_depth, int64_t max_nodes, int64_t capacity, int64_t history,
                         void* workspace, void* stream) {
    const int bad = depth_args_error(B, N, d, dtype, ops, flags, max_depth, max_nodes, capacity);
    if (bad != HK_OK) return bad;
    if (!depth_line_args_ok(B, N, d, capacity, history)) return HK_ERR_BAD_ARG;
    if (B == 0) return HK_OK;
    if (!roots || !depth || !nodes || !status || !line_mask || !line_axis || !workspace) return HK_ERR_BAD_ARG;
    if (((uintptr_t)roots) & 3u) return HK_ERR_ALIGN;
    DepthLine line;
    carve_depth_line(&line.w, (char*)align_up((size_t)(uintptr_t)workspace), B, N, d, capacity, history);
    line.history = history;
    line.line_mask = line_mask;
    line.line_axis = line_axis;
    return run_search_depth(roots, depth, nodes, status, B, N, d, ops, flags, max_depth, max_nodes, capacity, line.w.s,
                            &line, stream);
}

int64_t hk_search_value_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity, int64_t history) {
    if (!value_args_ok(B, N, d, capacity, history)) return 0;
    ValueWorkspace w;
    return (int64_t)(carve_value(&w, nullptr, B, N, d, capacity, history) + 256);  // + 256: room to align the pointer
}

// hk_search_value, hk_search_value_line when `line` is set (the line outputs are then required), and
// hk_search_value_labels when `labels` is set (the workspace is then hk_search_value_labels_workspace_bytes')
static int run_search_value(const void* roots, int32_t* value, int32_t* best_mask, int64_t* nodes, int8_t* status,
                            bool line, int32_t* line_mask, int32_t* line_axis, const LabelOutputs* labels, int64_t B,
                            int32_t N, int32_t d, int32_t dtype, uint32_t ops, int32_t max_depth, int64_t max_nodes,
                            int64_t capacity, int64_t history, void* workspace, void* stream) {
    if (B < 0 || N < 1 || d < 1 || (dtype != HK_DTYPE_I32 && dtype != HK_DTYPE_F32)) return HK_ERR_BAD_ARG;
    if (hk_kernel_class(N, d) < 0 || d < 2 || d > 6) return HK_ERR_UNSUPPORTED;  // <= 186 children: a uint8 count
    if (dtype != HK_DTYPE_I32) return HK_ERR_UNSUPPORTED;  // float32 state is not searched
    if ((ops & (HK_OP_SHIFT | HK_OP_NEWTON)) != (HK_OP_SHIFT | HK_OP_NEWTON) ||
        (ops & ~(HK_OP_SHIFT | HK_OP_NEWTON | HK_OP_REPOSITION)))
        return HK_ERR_BAD_ARG;
    if (max_depth < 1 || max_nodes < 1 || !value_args_ok(B, N, d, capacity, history)) return HK_ERR_BAD_ARG;
    if (labels) {
        if (labels->max_labels < 0 || !labels->count) return HK_ERR_BAD_ARG;
        if (labels->max_labels > 0 && (!labels->root || !labels->level || !labels->value || !labels->optimal ||
                                       !labels->mask || !labels->axis))
            return HK_ERR_BAD_ARG;
        *labels->count = 0;
    }
    if (B == 0) return HK_OK;
    if (!roots || !value || !best_mask || !nodes || !status || !workspace) return HK_ERR_BAD_ARG;
    if (line && (!line_mask || !line_axis)) return HK_ERR_BAD_ARG;
    if (((uintptr_t)roots) & 3u) return HK_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)stream;
    ValueWorkspace w;
    carve_value(&w, (char*)align_up((size_t)(uintptr_t)workspace), B, N, d, capacity, history);

    static_assert(sizeof(hk::ValueParams) <= 4096, "ValueParams is passed by value to every kernel");
    hk::ValueParams p;
    memset(&p, 0, sizeof(p));
    p.B = B;
    p.N = N;
    p.d = d;
    p.bound = (int32_t)((1 << 30) / d);
    p.max_nodes = max_nodes;
    p.capacity = capacity;
    p.history = history;
    // the children of an expanded node: S over the sets with |S| >= 2 in increasing order, the axes of S in order
    for (int S = 0; S < (1 << d); ++S) {
        if (__builtin_popcount((unsigned)S) < 2) continue;
        int rank = 0;
        for (int a = 0; a < d; ++a)
            if (S >> a & 1) p.pair[p.children++] = (uint16_t)(S | a << 6 | rank++ << 9);
    }
    p.kind = w.kind;
    p.count = w.count;
    p.tile_sum = w.tile_sum;
    p.root_children = w.root_children;
    p.root_flag = w.root_flag;
    p.root_shift = w.root_shift;
    p.counters = w.counters;
    p.value = value;
    p.best_mask = best_mask;
    p.nodes = (long long*)nodes;
    p.status = status;
    p.h_parent = w.h_parent;
    p.h_solved = w.h_solved;
    p.h_rem = w.h_rem;
    p.h_mask = w.h_mask;
    p.h_rank = w.h_rank;
    p.child_mask = w.child_mask;
    p.child_axis = w.child_axis;

    cudaError_t e = cudaMemsetAsync(w.root_children, 0, (size_t)B * 8, st);
    if (e == cudaSuccess) e = cudaMemsetAsync(w.root_flag, 0, (size_t)B * 4, st);
    if (e != cudaSuccess) return (int)e;
    const long long root_blocks = (B + 255) / 256;
    const unsigned root_grid = (unsigned)(root_blocks > 4096 ? 4096 : root_blocks);
    hk::hk_value_init_kernel<<<root_grid, 256, 0, st>>>(p, w.active[0]);

    const int32_t* state = (const int32_t*)roots;
    const int32_t* node_root = nullptr;  // level 0: node i is root i
    long long M = B, n_active = B, hist_base = 0;
    for (int level = 0;; ++level) {
        const int next = level & 1;  // frontier, node-root list and root list the next level is written to
        p.state = state;
        p.node_root = node_root;
        p.M = M;
        p.level = level;
        p.expand = level < max_depth;
        p.hist_base = hist_base;
        p.hist_used = hist_base + M;
        p.active = w.active[level & 1];
        p.active_next = w.active[(level + 1) & 1];
        p.n_active = n_active;
        p.child_state = w.frontier[next];
        p.child_root = w.node_root[next];
        const unsigned tiles = (unsigned)((M + hk::SEARCH_THREADS - 1) / hk::SEARCH_THREADS);
        hk::hk_value_solve_kernel<<<tiles, hk::SEARCH_THREADS, 0, st>>>(p);
        hk::hk_value_count_kernel<<<tiles, hk::SEARCH_THREADS, 0, st>>>(p);
        hk::hk_value_decide_kernel<<<1, hk::SEARCH_SCAN_THREADS, 0, st>>>(p);
        long long counters[2];
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(counters, w.counters, sizeof(counters), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return (int)e;
        if (!p.expand || counters[0] == 0) break;
        hk::hk_value_scatter_kernel<<<tiles, hk::SEARCH_THREADS, 0, st>>>(p);
        e = cudaGetLastError();
        if (e != cudaSuccess) return (int)e;
        int rc = hk_step(w.frontier[next], w.frontier[next], w.child_mask, w.child_axis, nullptr, nullptr, nullptr, nullptr,
                         nullptr, nullptr, counters[0], N, d, HK_DTYPE_I32, ops, 0, -1.0f, 1e8f, stream);
        if (rc != HK_OK) return rc;
        state = w.frontier[next];
        node_root = w.node_root[next];
        hist_base += M;
        M = counters[0];
        n_active = counters[1];
    }
    hk::hk_value_finish_kernel<<<root_grid, 256, 0, st>>>(p);
    if (line) hk::hk_line_value_walk_kernel<<<root_grid, 256, 0, st>>>(p, p.hist_used, line_mask, line_axis, max_depth);
    if (labels) {
        LabelWorkspace lw;
        carve_labels(&lw, (char*)align_up((size_t)(uintptr_t)workspace), B, N, d, capacity, history);
        hk::LabelParams q;
        memset(&q, 0, sizeof(q));
        q.used = p.hist_used;
        q.tile_sum = lw.tile_sum;
        q.block_sum = lw.block_sum;
        q.total = lw.total;
        q.tile_level = lw.tile_level;
        q.max_labels = labels->max_labels;
        q.max_depth = max_depth;
        q.root = labels->root;
        q.level = labels->level;
        q.value = labels->value;
        q.optimal = (unsigned long long*)labels->optimal;
        q.mask = labels->mask;
        q.axis = labels->axis;
        const long long tiles = (q.used + hk::SEARCH_THREADS - 1) / hk::SEARCH_THREADS;
        const long long blocks = (tiles + hk::SEARCH_SCAN_THREADS - 1) / hk::SEARCH_SCAN_THREADS;
        const unsigned tile_grid = (unsigned)((tiles + 255) / 256);
        hk::hk_label_level_kernel<<<tile_grid, 256, 0, st>>>(p, q, tiles);
        hk::hk_label_count_kernel<<<(unsigned)tiles, hk::SEARCH_THREADS, 0, st>>>(p, q);
        hk::hk_label_scan_tiles_kernel<<<(unsigned)blocks, hk::SEARCH_SCAN_THREADS, 0, st>>>(q, tiles);
        hk::hk_label_scan_blocks_kernel<<<1, hk::SEARCH_SCAN_THREADS, 0, st>>>(q, blocks);
        if (q.max_labels > 0) {
            const long long warps = hk::SEARCH_THREADS / 32;  // one warp per tile
            const unsigned grid = (unsigned)((tiles + warps - 1) / warps);
            hk::hk_label_write_kernel<<<grid, hk::SEARCH_THREADS, 0, st>>>(p, q, tiles);
        }
        long long total = 0;
        e = cudaGetLastError();
        if (e == cudaSuccess) e = cudaMemcpyAsync(&total, lw.total, sizeof(total), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e == cudaSuccess) *labels->count = total;
        return (int)e;
    }
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    return (int)e;
}

int hk_search_value(const void* roots, int32_t* value, int32_t* best_mask, int64_t* nodes, int8_t* status, int64_t B,
                    int32_t N, int32_t d, int32_t dtype, uint32_t ops, int32_t max_depth, int64_t max_nodes,
                    int64_t capacity, int64_t history, void* workspace, void* stream) {
    return run_search_value(roots, value, best_mask, nodes, status, false, nullptr, nullptr, nullptr, B, N, d, dtype,
                            ops, max_depth, max_nodes, capacity, history, workspace, stream);
}

int hk_search_value_line(const void* roots, int32_t* value, int32_t* best_mask, int64_t* nodes, int8_t* status,
                         int32_t* line_mask, int32_t* line_axis, int64_t B, int32_t N, int32_t d, int32_t dtype,
                         uint32_t ops, int32_t max_depth, int64_t max_nodes, int64_t capacity, int64_t history,
                         void* workspace, void* stream) {
    return run_search_value(roots, value, best_mask, nodes, status, true, line_mask, line_axis, nullptr, B, N, d, dtype,
                            ops, max_depth, max_nodes, capacity, history, workspace, stream);
}

int64_t hk_search_value_labels_workspace_bytes(int64_t B, int32_t N, int32_t d, int64_t capacity, int64_t history) {
    if (!value_args_ok(B, N, d, capacity, history)) return 0;
    LabelWorkspace w;
    return (int64_t)(carve_labels(&w, nullptr, B, N, d, capacity, history) + 256);  // + 256: room to align the pointer
}

int hk_search_value_labels(const void* roots, int32_t* value, int32_t* best_mask, int64_t* nodes, int8_t* status,
                           int64_t max_labels, int64_t* label_count, int32_t* label_root, int32_t* label_level,
                           int32_t* label_value, uint64_t* label_optimal, int32_t* label_mask, int32_t* label_axis,
                           int64_t B, int32_t N, int32_t d, int32_t dtype, uint32_t ops, int32_t max_depth,
                           int64_t max_nodes, int64_t capacity, int64_t history, void* workspace, void* stream) {
    const LabelOutputs labels{max_labels, label_count, label_root, label_level, label_value, label_optimal, label_mask,
                              label_axis};
    return run_search_value(roots, value, best_mask, nodes, status, false, nullptr, nullptr, &labels, B, N, d, dtype,
                            ops, max_depth, max_nodes, capacity, history, workspace, stream);
}

}  // extern "C"
