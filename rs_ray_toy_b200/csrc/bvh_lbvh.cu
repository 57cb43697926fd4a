// Device LBVH builder (RRT_BUILD_DEVICE_LBVH): Morton keys -> radix sort -> binary radix tree -> bottom-up
// boxes -> collapse small subtrees into leaves -> Node32 / Node64 written in place, all on the GPU; the host
// only receives the primitive order (to lay the primitive records out leaf by leaf).  See lbvh_core.h for what
// it replaces in the reference and for the per-element code (shared with the host probe).
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <thread>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <vector>

#include "bvh_lbvh.hpp"
#include "lbvh_core.h"
#include "reduce.cuh"

namespace rrt {

using namespace lbvh;

namespace {

#define LB_CUDA(call)                                                           \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) {                                                \
            if (err) *err = std::string(#call) + ": " + cudaGetErrorString(e_); \
            return RRT_ERR_CUDA;                                                \
        }                                                                       \
    } while (0)

struct CentroidFrame {
    float lo[3], inv_ext[3];
};

__global__ void __launch_bounds__(256) keys_kernel(uint32_t n, const BoxF* __restrict__ boxes, CentroidFrame f,
                                                    uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keys[i] = morton63(boxes[i], f.lo, f.inv_ext);
    vals[i] = i;
}

__global__ void __launch_bounds__(256) hierarchy_kernel(uint32_t n, const uint64_t* __restrict__ keys,
                                                         RadixNode* __restrict__ nodes, int32_t* __restrict__ parent_of_node,
                                                         int32_t* __restrict__ parent_of_leaf) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    const RadixNode r = radix_node(keys, (int64_t)n, (int64_t)i);
    nodes[i] = r;
    if (r.left < 0) parent_of_leaf[~r.left] = (int32_t)i; else parent_of_node[r.left] = (int32_t)i;
    if (r.right < 0) parent_of_leaf[~r.right] = (int32_t)i; else parent_of_node[r.right] = (int32_t)i;
    if (i == 0) parent_of_node[0] = -1;
}

// One thread per primitive (sorted position): gathers its box, then climbs; the second thread to reach a
// node owns it (its sibling's box is complete and visible after the fence).
__global__ void __launch_bounds__(256) refit_kernel(uint32_t n, const BoxF* __restrict__ boxes, const uint32_t* __restrict__ order,
                                                     const RadixNode* __restrict__ nodes, const int32_t* __restrict__ parent_of_node,
                                                     const int32_t* __restrict__ parent_of_leaf, BoxF* __restrict__ leaf_box,
                                                     BoxF* __restrict__ node_box, uint32_t* __restrict__ visits) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    leaf_box[p] = boxes[order[p]];
    __threadfence();
    int32_t node = parent_of_leaf[p];
    while (node >= 0) {
        if (atomicAdd(visits + node, 1u) == 0u) return;  // first arrival: the sibling subtree is not done yet
        __threadfence();
        const RadixNode r = nodes[node];
        const volatile BoxF* lb = r.left < 0 ? leaf_box + ~r.left : node_box + r.left;
        const volatile BoxF* rb = r.right < 0 ? leaf_box + ~r.right : node_box + r.right;
        BoxF a, b;
        for (int k = 0; k < 3; ++k) {
            a.lo[k] = lb->lo[k]; a.hi[k] = lb->hi[k];
            b.lo[k] = rb->lo[k]; b.hi[k] = rb->hi[k];
        }
        node_box[node] = box_union(a, b);
        __threadfence();
        node = parent_of_node[node];
    }
}

__global__ void __launch_bounds__(256) flag_kernel(uint32_t n_internal, const RadixNode* __restrict__ nodes, uint32_t max_leaf,
                                                    uint32_t* __restrict__ keep) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_internal) return;
    keep[i] = (nodes[i].last - nodes[i].first + 1u > max_leaf) ? 1u : 0u;
}

// ---- exclusive prefix sum of uint32 (any length): 1024-element blocks, block sums scanned recursively -------------------
constexpr int kScanTile = 1024;
__global__ void __launch_bounds__(kScanTile) scan_tiles_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n,
                                                                uint32_t* __restrict__ tile_sums) {
    __shared__ uint32_t warp_sums[32];
    const uint32_t i = blockIdx.x * kScanTile + threadIdx.x;
    const uint32_t v = i < n ? in[i] : 0u;
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, off);
        if ((int)lane >= off) x += y;
    }
    if (lane == 31) warp_sums[warp] = x;
    __syncthreads();
    if (warp == 0) {
        uint32_t w = warp_sums[lane];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, w, off);
            if ((int)lane >= off) w += y;
        }
        warp_sums[lane] = w;
    }
    __syncthreads();
    const uint32_t incl = x + (warp > 0 ? warp_sums[warp - 1] : 0u);
    if (i < n) out[i] = incl - v;
    if (tile_sums != nullptr && threadIdx.x == kScanTile - 1) tile_sums[blockIdx.x] = incl;
}
__global__ void __launch_bounds__(kScanTile) scan_add_kernel(uint32_t* __restrict__ out, uint32_t n, const uint32_t* __restrict__ tile_offsets) {
    const uint32_t i = blockIdx.x * kScanTile + threadIdx.x;
    if (i < n) out[i] += tile_offsets[blockIdx.x];
}
// scratch: at least scan_scratch_words(n) uint32
size_t scan_scratch_words(size_t n) {
    size_t total = 0;
    while (n > (size_t)kScanTile) {
        n = (n + kScanTile - 1) / kScanTile;
        total += n;
    }
    return total + 1;
}
void exclusive_scan_u32(const uint32_t* d_in, uint32_t* d_out, uint32_t n, uint32_t* d_scratch, cudaStream_t s) {
    if (n == 0) return;
    const uint32_t tiles = (n + kScanTile - 1) / kScanTile;
    if (tiles == 1) {
        scan_tiles_kernel<<<1, kScanTile, 0, s>>>(d_in, d_out, n, nullptr);
        return;
    }
    scan_tiles_kernel<<<tiles, kScanTile, 0, s>>>(d_in, d_out, n, d_scratch);
    exclusive_scan_u32(d_scratch, d_scratch, tiles, d_scratch + tiles, s);  // in place: a tile reads before it writes
    scan_add_kernel<<<tiles, kScanTile, 0, s>>>(d_out, n, d_scratch);
}

// ---- stable LSD radix sort of (63-bit key, uint32 value) pairs, 8 bits per pass ---------------------------------------------
// A pass: (1) per-tile digit histograms, stored digit-major so that ONE exclusive scan over [256][tiles] gives every
// (digit, tile) its output base; (2) a stable scatter.  A tile is 2048 pairs; warp w of its CTA owns the 256 consecutive
// pairs [256 w, 256 w + 256) and walks them in 8 rounds of 32, so "earlier in the input" is (warp, round, lane) order:
// the rank of a pair is base[digit][tile] + pairs with that digit in lower warps + in this warp's earlier rounds + in
// lower lanes of this round (__match_any_sync).
constexpr int kSortTile = 2048, kSortWarps = 8;
__global__ void __launch_bounds__(256) radix_hist_kernel(const uint64_t* __restrict__ keys, uint32_t n, int shift,
                                                          uint32_t* __restrict__ hist, uint32_t n_tiles) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t base = blockIdx.x * kSortTile;
#pragma unroll
    for (int r = 0; r < kSortTile / 256; ++r) {
        const uint32_t i = base + r * 256 + threadIdx.x;
        if (i < n) atomicAdd(&h[(uint32_t)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * n_tiles + blockIdx.x] = h[threadIdx.x];
}
__global__ void __launch_bounds__(256) radix_scatter_kernel(const uint64_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                                                             uint64_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, uint32_t n,
                                                             int shift, const uint32_t* __restrict__ offsets, uint32_t n_tiles) {
    __shared__ uint32_t wc[kSortWarps][256];  // per-warp digit counts, then each warp's running base
    const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (int k = threadIdx.x; k < kSortWarps * 256; k += 256) (&wc[0][0])[k] = 0;
    __syncthreads();
    const uint32_t warp_base = blockIdx.x * kSortTile + warp * 256;
    uint64_t key[8];
    uint32_t val[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const uint32_t i = warp_base + r * 32 + lane;
        key[r] = i < n ? keys_in[i] : ~0ull;
        val[r] = i < n ? vals_in[i] : 0u;
        if (i < n) atomicAdd(&wc[warp][(uint32_t)(key[r] >> shift) & 255u], 1u);
    }
    __syncthreads();
    {   // thread d: exclusive sum over the warps for digit d, on top of the tile's global base
        const uint32_t d = threadIdx.x;
        uint32_t run = offsets[(size_t)d * n_tiles + blockIdx.x];
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) {
            const uint32_t c = wc[w][d];
            wc[w][d] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const uint32_t i = warp_base + r * 32 + lane;
        const bool valid = i < n;
        const uint32_t d = valid ? (uint32_t)(key[r] >> shift) & 255u : 256u + lane;  // invalid lanes match nobody
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        if (valid) {
            const uint32_t pos = wc[warp][d] + (uint32_t)__popc(peers & ((1u << lane) - 1u));
            keys_out[pos] = key[r];
            vals_out[pos] = val[r];
        }
        __syncwarp();
        if (valid && (int)lane == __ffs(peers) - 1) wc[warp][d] += (uint32_t)__popc(peers);
        __syncwarp();
    }
}
// Sorts (keys, vals) by the low `bits` bits; the result lands in (keys_b, vals_b) when the number of passes is odd, else
// in (keys_a, vals_a): the return value says which (0 = a, 1 = b).  d_hist: 256 * tiles words, d_scratch: scan_scratch_words(256 * tiles).
int radix_sort_pairs(uint64_t* keys_a, uint32_t* vals_a, uint64_t* keys_b, uint32_t* vals_b, uint32_t n, int bits, uint32_t* d_hist,
                     uint32_t* d_scratch, cudaStream_t s) {
    const uint32_t tiles = (n + kSortTile - 1) / kSortTile;
    int where = 0;
    for (int shift = 0; shift < bits; shift += 8) {
        uint64_t* kin = where ? keys_b : keys_a;
        uint64_t* kout = where ? keys_a : keys_b;
        uint32_t* vin = where ? vals_b : vals_a;
        uint32_t* vout = where ? vals_a : vals_b;
        radix_hist_kernel<<<tiles, 256, 0, s>>>(kin, n, shift, d_hist, tiles);
        exclusive_scan_u32(d_hist, d_hist, 256u * tiles, d_scratch, s);
        radix_scatter_kernel<<<tiles, 256, 0, s>>>(kin, vin, kout, vout, n, shift, d_hist, tiles);
        where ^= 1;
    }
    return where;
}

template <bool QUANT>
__global__ void __launch_bounds__(256) emit_kernel(uint32_t n_internal, const RadixNode* __restrict__ nodes,
                                                    const uint32_t* __restrict__ keep, const uint32_t* __restrict__ new_index,
                                                    const BoxF* __restrict__ leaf_box, const BoxF* __restrict__ node_box, EmitParams P,
                                                    void* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_internal || keep[i] == 0u) return;
    const RadixNode r = nodes[i];
    const BoxF b0 = r.left < 0 ? leaf_box[~r.left] : node_box[r.left];
    const BoxF b1 = r.right < 0 ? leaf_box[~r.right] : node_box[r.right];
    const int32_t r0 = child_ref(r.left, nodes, new_index, P.max_leaf), r1 = child_ref(r.right, nodes, new_index, P.max_leaf);
    if (QUANT) emit32(b0, b1, r0, r1, P, static_cast<Node32*>(out) + new_index[i]);
    else emit64(b0, b1, r0, r1, P, static_cast<Node64*>(out) + new_index[i]);
}

// Depth of the emitted tree (kept ancestors of a primitive) and the number of leaf references.
__global__ void __launch_bounds__(256) depth_kernel(uint32_t n, const RadixNode* __restrict__ nodes, const uint32_t* __restrict__ keep,
                                                     const int32_t* __restrict__ parent_of_node, const int32_t* __restrict__ parent_of_leaf,
                                                     uint32_t* __restrict__ out2) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    uint32_t depth = 0;
    int32_t node = parent_of_leaf[p];
    bool leaf_head = true;  // p opens a leaf iff it is the first position of the topmost collapsed subtree above it
    while (node >= 0) {
        if (keep[node]) depth += 1;
        else if (nodes[node].first != p) leaf_head = false;
        node = parent_of_node[node];
    }
    atomicMax(out2, depth);
    if (leaf_head) atomicAdd(out2 + 1, 1u);
}

}  // namespace

namespace {

struct Lap {
    bool on = std::getenv("RRT_BUILD_TIMING") != nullptr;
    std::chrono::steady_clock::time_point last = std::chrono::steady_clock::now();
    void operator()(const char* what) {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "RRT_BUILD_TIMING   lbvh: %-18s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - last).count());
        last = now;
    }
};

// Every scratch array of a build over n primitives in ONE allocation (15 cudaMalloc + 15 cudaFree cost 30-80 ms).
struct ArenaLayout {
    size_t o_boxes, o_leaf_box, o_node_box, o_keys, o_keys_sorted, o_vals, o_order, o_visits, o_keep, o_new, o_out2, o_nodes,
        o_pnode, o_pleaf, o_tmp, hist_words, total = 0;
    explicit ArenaLayout(uint32_t n) {
        const uint32_t ni = n - 1;
        const uint32_t sort_tiles = (n + kSortTile - 1) / kSortTile;
        hist_words = 256 * (size_t)sort_tiles;
        const size_t scratch_words = std::max(scan_scratch_words(hist_words), scan_scratch_words(ni));
        o_boxes = reserve((size_t)n * sizeof(BoxF));
        o_leaf_box = reserve((size_t)n * sizeof(BoxF));
        o_node_box = reserve((size_t)ni * sizeof(BoxF));
        o_keys = reserve((size_t)n * sizeof(uint64_t));
        o_keys_sorted = reserve((size_t)n * sizeof(uint64_t));
        o_vals = reserve((size_t)n * sizeof(uint32_t));
        o_order = reserve((size_t)n * sizeof(uint32_t));
        o_visits = reserve((size_t)ni * sizeof(uint32_t));
        o_keep = reserve((size_t)ni * sizeof(uint32_t));
        o_new = reserve((size_t)ni * sizeof(uint32_t));
        o_out2 = reserve(2 * sizeof(uint32_t));
        o_nodes = reserve((size_t)ni * sizeof(RadixNode));
        o_pnode = reserve((size_t)ni * sizeof(int32_t));
        o_pleaf = reserve((size_t)n * sizeof(int32_t));
        o_tmp = reserve((hist_words + scratch_words) * sizeof(uint32_t));
    }
    size_t reserve(size_t bytes) {
        const size_t at = total;
        total += (bytes + 255) & ~(size_t)255;
        return at;
    }
};

// The build from the fp32 boxes already in the arena (layout ArenaLayout(n)) and their centroid frame: keys, sort,
// hierarchy, boxes, collapse, emitted nodes.  out->d_order points into the arena.
int build_in_arena(uint32_t n, char* d_arena, const CentroidFrame& fr, uint32_t max_leaf, double delta, bool quantise,
                   const double grid_lo[3], const float grid_ext[3], LbvhResult* out, std::string* err, Lap& lap) {
    const ArenaLayout L(n);
    EmitParams P;
    P.max_leaf = max_leaf;
    P.quantise = quantise ? 1 : 0;
    P.delta = delta;
    for (int k = 0; k < 3; ++k) {
        P.grid_lo[k] = grid_lo[k];
        P.grid_ext[k] = (double)grid_ext[k];
    }
    BoxF* d_boxes = reinterpret_cast<BoxF*>(d_arena + L.o_boxes);
    BoxF* d_leaf_box = reinterpret_cast<BoxF*>(d_arena + L.o_leaf_box);
    BoxF* d_node_box = reinterpret_cast<BoxF*>(d_arena + L.o_node_box);
    uint64_t* d_keys = reinterpret_cast<uint64_t*>(d_arena + L.o_keys);
    uint64_t* d_keys_sorted = reinterpret_cast<uint64_t*>(d_arena + L.o_keys_sorted);
    uint32_t* d_vals = reinterpret_cast<uint32_t*>(d_arena + L.o_vals);
    uint32_t* d_order = reinterpret_cast<uint32_t*>(d_arena + L.o_order);
    uint32_t* d_visits = reinterpret_cast<uint32_t*>(d_arena + L.o_visits);
    uint32_t* d_keep = reinterpret_cast<uint32_t*>(d_arena + L.o_keep);
    uint32_t* d_new = reinterpret_cast<uint32_t*>(d_arena + L.o_new);
    uint32_t* d_out2 = reinterpret_cast<uint32_t*>(d_arena + L.o_out2);
    RadixNode* d_nodes = reinterpret_cast<RadixNode*>(d_arena + L.o_nodes);
    int32_t* d_pnode = reinterpret_cast<int32_t*>(d_arena + L.o_pnode);
    int32_t* d_pleaf = reinterpret_cast<int32_t*>(d_arena + L.o_pleaf);
    void* d_tmp = d_arena + L.o_tmp;
    void* d_emit = nullptr;
#define LB_TRY(call)                                                            \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) {                                                \
            if (err) *err = std::string(#call) + ": " + cudaGetErrorString(e_); \
            if (d_emit) cudaFree(d_emit);                                       \
            return RRT_ERR_CUDA;                                                \
        }                                                                       \
    } while (0)
    const uint32_t ni = n - 1;
    LB_TRY(cudaMemset(d_visits, 0, (size_t)ni * sizeof(uint32_t)));
    LB_TRY(cudaMemset(d_out2, 0, 2 * sizeof(uint32_t)));

    cudaEvent_t e0, e1;
    LB_TRY(cudaEventCreate(&e0));
    LB_TRY(cudaEventCreate(&e1));
    LB_TRY(cudaEventRecord(e0, 0));
    const unsigned gb = (n + 255) / 256, gi = (ni + 255) / 256;
    keys_kernel<<<gb, 256>>>(n, d_boxes, fr, d_keys, d_vals);
    uint32_t* d_hist = static_cast<uint32_t*>(d_tmp);
    uint32_t* d_scan_scratch = d_hist + L.hist_words;
    // 63-bit Morton keys: eight 8-bit passes (an even number: the sorted pairs end where they started, then swap names)
    if (radix_sort_pairs(d_keys, d_vals, d_keys_sorted, d_order, n, 64, d_hist, d_scan_scratch, 0) == 0) {
        std::swap(d_keys, d_keys_sorted);
        std::swap(d_vals, d_order);
    }
    hierarchy_kernel<<<gi, 256>>>(n, d_keys_sorted, d_nodes, d_pnode, d_pleaf);
    refit_kernel<<<gb, 256>>>(n, d_boxes, d_order, d_nodes, d_pnode, d_pleaf, d_leaf_box, d_node_box, d_visits);
    flag_kernel<<<gi, 256>>>(ni, d_nodes, max_leaf, d_keep);
    exclusive_scan_u32(d_keep, d_new, ni, d_scan_scratch, 0);
    uint32_t last_keep = 0, last_new = 0;
    LB_TRY(cudaMemcpy(&last_keep, d_keep + (ni - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost));
    LB_TRY(cudaMemcpy(&last_new, d_new + (ni - 1), sizeof(uint32_t), cudaMemcpyDeviceToHost));
    const uint32_t n_kept = last_new + last_keep;
    const size_t node_size = quantise ? sizeof(Node32) : sizeof(Node64);
    LB_TRY(cudaMalloc(&d_emit, (size_t)n_kept * node_size));
    if (quantise) emit_kernel<true><<<gi, 256>>>(ni, d_nodes, d_keep, d_new, d_leaf_box, d_node_box, P, d_emit);
    else emit_kernel<false><<<gi, 256>>>(ni, d_nodes, d_keep, d_new, d_leaf_box, d_node_box, P, d_emit);
    depth_kernel<<<gb, 256>>>(n, d_nodes, d_keep, d_pnode, d_pleaf, d_out2);
    LB_TRY(cudaEventRecord(e1, 0));
    LB_TRY(cudaGetLastError());
    LB_TRY(cudaEventSynchronize(e1));
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    lap("kernels");
    uint32_t out2[2] = {0, 0};
    LB_TRY(cudaMemcpy(out2, d_out2, sizeof(out2), cudaMemcpyDeviceToHost));
    // the root's box (for the caller's world bound): node 0 of the radix tree
    BoxF root;
    LB_TRY(cudaMemcpy(&root, d_node_box, sizeof(BoxF), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 3; ++k) {
        out->root_lo[k] = root.lo[k];
        out->root_hi[k] = root.hi[k];
    }
    out->d_order = d_order;
    out->d_nodes = d_emit;
    out->node_bytes = (size_t)n_kept * node_size;
    out->n_nodes = n_kept;
    out->max_depth = out2[0];
    out->n_leaves = out2[1];
    out->device_ms = ms;
    return RRT_OK;
#undef LB_TRY
}

CentroidFrame centroid_frame(const double clo[3], const double chi[3]) {
    CentroidFrame fr;
    for (int k = 0; k < 3; ++k) {
        fr.lo[k] = down_f(clo[k]);
        const double ext = chi[k] - (double)fr.lo[k];
        fr.inv_ext[k] = ext > 0.0 ? (float)(1.0 / ext) : 0.0f;
    }
    return fr;
}

// f64 boxes -> fp32 boxes rounded outward (the host conversion's down_f / up_f), and the bounds of their centroids:
// a min / max, so the same values whatever order the blocks fold in.
struct CentroidBounds {
    double lo[3], hi[3];
};
__global__ void __launch_bounds__(256) boxes_f32_kernel(uint32_t n, const Aabb* __restrict__ boxes, BoxF* __restrict__ out,
                                                         CentroidBounds* __restrict__ cb) {
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        BoxF f;
        for (int k = 0; k < 3; ++k) {
            f.lo[k] = down_f(boxes[i].lo[k]);
            f.hi[k] = up_f(boxes[i].hi[k]);
            const double c = 0.5 * (double)f.lo[k] + 0.5 * (double)f.hi[k];
            lo[k] = fmin(lo[k], c);
            hi[k] = fmax(hi[k], c);
        }
        out[i] = f;
    }
    for (int k = 0; k < 3; ++k) {
        lo[k] = warp_min_f64(lo[k]);
        hi[k] = warp_max_f64(hi[k]);
    }
    if ((threadIdx.x & 31u) == 0)
        for (int k = 0; k < 3; ++k) {
            atomic_min_f64(&cb->lo[k], lo[k]);
            atomic_max_f64(&cb->hi[k], hi[k]);
        }
}

}  // namespace

LbvhArena::~LbvhArena() {
    if (d) cudaFree(d);
}

int build_lbvh_device(int device, AabbSpan boxes, uint32_t max_leaf, double delta, bool quantise,
                      const double grid_lo[3], const float grid_ext[3], LbvhResult* out, std::string* err) {
    const auto t0 = std::chrono::steady_clock::now();
    Lap lap;
    const uint32_t n = (uint32_t)boxes.size();
    if (n < 2 || n <= max_leaf) {
        if (err) *err = "device LBVH needs more primitives than one leaf holds";
        return RRT_ERR_UNSUPPORTED;
    }
    LB_CUDA(cudaSetDevice(device));
    // fp32 boxes rounded outward + the centroid frame
    RawBuf<BoxF> hb(n);
    double clo[3] = {INFINITY, INFINITY, INFINITY}, chi[3] = {-INFINITY, -INFINITY, -INFINITY};
    {
        unsigned nt = std::thread::hardware_concurrency();
        nt = nt == 0 ? 1 : (nt > 32 ? 32 : nt);
        if (n < 65536) nt = 1;
        std::vector<std::array<double, 6>> part(nt, {INFINITY, INFINITY, INFINITY, -INFINITY, -INFINITY, -INFINITY});
        std::vector<std::thread> pool;
        const size_t step = ((size_t)n + nt - 1) / nt;
        auto work = [&](unsigned t) {
            const size_t a = (size_t)t * step, b = std::min<size_t>(n, a + step);
            for (size_t i = a; i < b; ++i)
                for (int k = 0; k < 3; ++k) {
                    hb[i].lo[k] = down_f(boxes[i].lo[k]);
                    hb[i].hi[k] = up_f(boxes[i].hi[k]);
                    const double c = 0.5 * (double)hb[i].lo[k] + 0.5 * (double)hb[i].hi[k];
                    part[t][k] = std::fmin(part[t][k], c);
                    part[t][3 + k] = std::fmax(part[t][3 + k], c);
                }
        };
        for (unsigned t = 1; t < nt; ++t) pool.emplace_back(work, t);
        work(0);
        for (auto& th : pool) th.join();
        for (unsigned t = 0; t < nt; ++t)
            for (int k = 0; k < 3; ++k) {
                clo[k] = std::fmin(clo[k], part[t][k]);
                chi[k] = std::fmax(chi[k], part[t][3 + k]);
            }
    }
    lap("fp32 boxes (host)");
    const CentroidFrame fr = centroid_frame(clo, chi);
    const ArenaLayout L(n);
    char* d_arena = nullptr;
    LB_CUDA(cudaMalloc(&d_arena, L.total));
    lap("cudaMalloc (arena)");
    int rc = RRT_OK;
    cudaError_t e = cudaMemcpy(d_arena + L.o_boxes, hb.get(), (size_t)n * sizeof(BoxF), cudaMemcpyHostToDevice);
    lap("boxes H2D");
    if (e != cudaSuccess) {
        if (err) *err = std::string("cudaMemcpy (boxes): ") + cudaGetErrorString(e);
        rc = RRT_ERR_CUDA;
    }
    if (rc == RRT_OK) rc = build_in_arena(n, d_arena, fr, max_leaf, delta, quantise, grid_lo, grid_ext, out, err, lap);
    if (rc == RRT_OK) {
        out->order.resize(n);
        e = cudaMemcpy(out->order.data(), out->d_order, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost);
        out->d_order = nullptr;
        if (e != cudaSuccess) {
            if (err) *err = std::string("cudaMemcpy (order): ") + cudaGetErrorString(e);
            cudaFree(out->d_nodes);
            out->d_nodes = nullptr;
            rc = RRT_ERR_CUDA;
        }
        lap("order D2H");
    }
    cudaFree(d_arena);
    lap("cudaFree (arena)");
    out->total_usec = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return rc;
}

int build_lbvh_device_boxes(int device, const Aabb* d_boxes, uint32_t n, uint32_t max_leaf, double delta, bool quantise,
                            const double grid_lo[3], const float grid_ext[3], LbvhArena* arena, LbvhResult* out,
                            std::string* err) {
    const auto t0 = std::chrono::steady_clock::now();
    Lap lap;
    if (n < 2 || n <= max_leaf) {
        if (err) *err = "device LBVH needs more primitives than one leaf holds";
        return RRT_ERR_UNSUPPORTED;
    }
    LB_CUDA(cudaSetDevice(device));
    const ArenaLayout L(n);
    // the arena also holds the centroid bounds, after the build's arrays
    const size_t need = L.total + sizeof(CentroidBounds);
    if (arena->bytes < need) {
        if (arena->d) cudaFree(arena->d);
        arena->d = nullptr;
        arena->bytes = 0;
        LB_CUDA(cudaMalloc(&arena->d, need));
        arena->bytes = need;
    }
    char* d_arena = static_cast<char*>(arena->d);
    CentroidBounds* d_cb = reinterpret_cast<CentroidBounds*>(d_arena + L.total);
    const CentroidBounds init = {{INFINITY, INFINITY, INFINITY}, {-INFINITY, -INFINITY, -INFINITY}};
    LB_CUDA(cudaMemcpy(d_cb, &init, sizeof(init), cudaMemcpyHostToDevice));
    boxes_f32_kernel<<<std::min<uint32_t>((n + 255) / 256, 1024u), 256>>>(n, d_boxes, reinterpret_cast<BoxF*>(d_arena + L.o_boxes), d_cb);
    LB_CUDA(cudaGetLastError());
    CentroidBounds cb;
    LB_CUDA(cudaMemcpy(&cb, d_cb, sizeof(cb), cudaMemcpyDeviceToHost));
    lap("fp32 boxes (device)");
    const int rc = build_in_arena(n, d_arena, centroid_frame(cb.lo, cb.hi), max_leaf, delta, quantise, grid_lo, grid_ext, out, err, lap);
    out->total_usec = (uint64_t)std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count();
    return rc;
}

// Host run of the same per-element code, for the CPU tests (a checker, not a product path): returns the emitted
// Node64 array, the primitive order and (max depth, leaves).
int lbvh_host_probe(const std::vector<Aabb>& boxes, uint32_t max_leaf, double delta, bool quantise, const double grid_lo[3],
                    const float grid_ext[3], std::vector<uint8_t>* nodes_out, std::vector<uint32_t>* order_out, uint32_t* depth_out,
                    uint32_t* leaves_out) {
    const uint32_t n = (uint32_t)boxes.size();
    if (n < 2 || n <= max_leaf) return RRT_ERR_UNSUPPORTED;
    RawBuf<BoxF> hb(n);
    double clo[3] = {INFINITY, INFINITY, INFINITY}, chi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (uint32_t i = 0; i < n; ++i)
        for (int k = 0; k < 3; ++k) {
            hb[i].lo[k] = down_f(boxes[i].lo[k]);
            hb[i].hi[k] = up_f(boxes[i].hi[k]);
            const double c = 0.5 * (double)hb[i].lo[k] + 0.5 * (double)hb[i].hi[k];
            clo[k] = std::fmin(clo[k], c);
            chi[k] = std::fmax(chi[k], c);
        }
    float flo[3], finv[3];
    for (int k = 0; k < 3; ++k) {
        flo[k] = down_f(clo[k]);
        const double ext = chi[k] - (double)flo[k];
        finv[k] = ext > 0.0 ? (float)(1.0 / ext) : 0.0f;
    }
    std::vector<std::pair<uint64_t, uint32_t>> kv(n);
    for (uint32_t i = 0; i < n; ++i) kv[i] = {morton63(hb[i], flo, finv), i};
    std::stable_sort(kv.begin(), kv.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
    std::vector<uint64_t> keys(n);
    std::vector<uint32_t>& order = *order_out;
    order.resize(n);
    for (uint32_t i = 0; i < n; ++i) {
        keys[i] = kv[i].first;
        order[i] = kv[i].second;
    }
    const uint32_t ni = n - 1;
    std::vector<RadixNode> nodes(ni);
    std::vector<int32_t> pnode(ni, -1), pleaf(n, -1);
    for (uint32_t i = 0; i < ni; ++i) {
        const RadixNode r = radix_node(keys.data(), n, i);
        nodes[i] = r;
        if (r.left < 0) pleaf[~r.left] = (int32_t)i; else pnode[r.left] = (int32_t)i;
        if (r.right < 0) pleaf[~r.right] = (int32_t)i; else pnode[r.right] = (int32_t)i;
    }
    std::vector<BoxF> leaf_box(n), node_box(ni);
    std::vector<uint32_t> visits(ni, 0);
    for (uint32_t p = 0; p < n; ++p) leaf_box[p] = hb[order[p]];
    for (uint32_t p = 0; p < n; ++p) {
        int32_t node = pleaf[p];
        while (node >= 0) {
            if (visits[node]++ == 0) break;
            const RadixNode& r = nodes[node];
            node_box[node] = box_union(r.left < 0 ? leaf_box[~r.left] : node_box[r.left], r.right < 0 ? leaf_box[~r.right] : node_box[r.right]);
            node = pnode[node];
        }
    }
    std::vector<uint32_t> keep(ni), new_index(ni);
    uint32_t n_kept = 0;
    for (uint32_t i = 0; i < ni; ++i) {
        keep[i] = nodes[i].last - nodes[i].first + 1u > max_leaf ? 1u : 0u;
        new_index[i] = n_kept;
        n_kept += keep[i];
    }
    EmitParams P;
    P.max_leaf = max_leaf;
    P.quantise = quantise ? 1 : 0;
    P.delta = delta;
    for (int k = 0; k < 3; ++k) {
        P.grid_lo[k] = grid_lo[k];
        P.grid_ext[k] = (double)grid_ext[k];
    }
    const size_t node_size = quantise ? sizeof(Node32) : sizeof(Node64);
    nodes_out->assign((size_t)n_kept * node_size, 0);
    for (uint32_t i = 0; i < ni; ++i) {
        if (!keep[i]) continue;
        const RadixNode& r = nodes[i];
        const BoxF b0 = r.left < 0 ? leaf_box[~r.left] : node_box[r.left], b1 = r.right < 0 ? leaf_box[~r.right] : node_box[r.right];
        const int32_t r0 = child_ref(r.left, nodes.data(), new_index.data(), max_leaf), r1 = child_ref(r.right, nodes.data(), new_index.data(), max_leaf);
        if (quantise) emit32(b0, b1, r0, r1, P, reinterpret_cast<Node32*>(nodes_out->data()) + new_index[i]);
        else emit64(b0, b1, r0, r1, P, reinterpret_cast<Node64*>(nodes_out->data()) + new_index[i]);
    }
    uint32_t depth = 0, leaves = 0;
    for (uint32_t p = 0; p < n; ++p) {
        uint32_t d = 0;
        bool head = true;
        for (int32_t node = pleaf[p]; node >= 0; node = pnode[node]) {
            if (keep[node]) d += 1;
            else if (nodes[node].first != p) head = false;
        }
        depth = std::max(depth, d);
        leaves += head ? 1 : 0;
    }
    *depth_out = depth;
    *leaves_out = leaves;
    return RRT_OK;
}

}  // namespace rrt
