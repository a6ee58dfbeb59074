// sah_build.cuh — device-side, top-down binned-SAH BVH construction: the trees of the host builder
// (flatten.cpp, BvhBuilder::build_range) built on the GPU, for scenes whose primitive count makes the host
// build the bottleneck. Same contract as lbvh_build / ploc_build (lbvh.cuh), except that leaves hold up to
// BvhPolicy::max_leaf records, so the builder also reorders the world's records into leaf order.
//
// Level-synchronous (Wald, "On fast construction of SAH-based bounding volume hierarchies", RT 2007; Garanzha
// et al., "Simpler and faster HLBVH with work queues", HPG 2011). A segment is a contiguous run [begin, + count)
// of the item array, the primitives of one node-to-be. Per level, over the segments of that level:
//   bin     one pass over the items: per segment, 3 axes x nb bins of (count, box, centroid bounds), privatised in
//           shared memory per CTA and merged with global atomics. Floats are min/max-ed as order-preserving ints,
//           so the result does not depend on the order of the atomics.
//   decide  one warp per segment: prefix / suffix scans over the bins of each axis, the host's rule for the plane
//           (half-area x count on both sides, first minimum in axis-then-plane order) and for leaves.
//   emit    a scan over the segments hands out the node indices of the level's inner segments (no atomicAdd:
//           two builds of a scene are byte-identical, the root is node_base and the top of the tree is
//           contiguous); each segment writes its box and its node index or leaf code into its parent's slot and
//           makes its two child segments.
//   split   flag each item (goes left), one exclusive scan over all items, scatter: a stable partition inside
//           every segment. Items of leaves stay where they are.
// The host reads the number of child segments once per level. After the last level the item array is the leaf
// order; the world's records are gathered into it.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include <algorithm>

#include <cub/device/device_scan.cuh>

#include "device_types.h"
#include "flatten.hpp"

namespace rtx {

// One item of the work array: its fp32 box (rounded outward) and what it is.
struct alignas(16) SahItem {
    float lo[3], hi[3];
    int32_t item;  // index into the world's items / records
    int32_t seg;   // segment of the current level, -1: in a finished leaf
};
static_assert(sizeof(SahItem) == 32, "SahItem must be 32 bytes");

// A bin: count, box, centroid bounds. The six bounds each are order-preserving ints of floats (sah_key).
constexpr int kSahBinInts = 13;
struct SahSeg {
    int32_t begin, count;
    int32_t parent, side;  // the slot this segment fills: child `side` of node `parent` (-1: the root)
    int32_t bin_off;       // first bin of this segment (3 axes x sah_nb(count) bins)
    float clo[3], chi[3];  // centroid bounds (bounds the items' centroids; exact for every plane split)
};
struct SahDecision {
    int32_t axis;   // split axis, -1: median split of the index range
    int32_t split;  // last bin of the left side
    int32_t lc;     // items that go left
    int32_t inner;  // 0: the segment is a leaf
    float box[6];   // the segment's box (lo.xyz, hi.xyz)
    float cb[2][6]; // centroid bounds of the two children (lo.xyz, hi.xyz)
};

__device__ __forceinline__ int32_t sah_key(float f) {
    const int32_t i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float sah_unkey(int32_t k) { return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff); }
__host__ __device__ __forceinline__ int sah_nb(int n) { return n <= 1 ? 1 : (n < kBvhBins ? n : kBvhBins); }
__device__ __forceinline__ float sah_scale(int nb, float lo, float hi) { return hi > lo ? (float)nb / (hi - lo) : 0.f; }
// The bin of a centroid coordinate: the same expression in the bin pass and in the split pass.
__device__ __forceinline__ int sah_bin(float c, float lo, float scale, int nb) {
    return min(nb - 1, max(0, (int)(__fsub_rn(c, lo) * scale)));
}
__device__ __forceinline__ float sah_centroid(const SahItem& it, int a) { return 0.5f * (it.lo[a] + it.hi[a]); }

__global__ void sah_init_kernel(int n, const float* __restrict__ boxes, SahItem* __restrict__ items, SahSeg* __restrict__ root,
                                int32_t* __restrict__ cbk) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    int32_t kmin[3] = {0x7f800000, 0x7f800000, 0x7f800000}, kmax[3] = {(int32_t)0x807fffff, (int32_t)0x807fffff, (int32_t)0x807fffff};
    if (i < n) {
        SahItem it;
        for (int a = 0; a < 3; ++a) { it.lo[a] = boxes[6 * (size_t)i + a]; it.hi[a] = boxes[6 * (size_t)i + 3 + a]; }
        it.item = i;
        it.seg = 0;
        items[i] = it;
        for (int a = 0; a < 3; ++a) kmin[a] = kmax[a] = sah_key(sah_centroid(it, a));
    }
    for (int a = 0; a < 3; ++a) {  // the root's centroid bounds, as keys (finished by sah_root_kernel)
        const int32_t lo = __reduce_min_sync(0xffffffffu, kmin[a]), hi = __reduce_max_sync(0xffffffffu, kmax[a]);
        if ((threadIdx.x & 31) == 0) { atomicMin(&cbk[a], lo); atomicMax(&cbk[3 + a], hi); }
    }
}

__global__ void sah_root_kernel(int n, const int32_t* __restrict__ cbk, SahSeg* __restrict__ seg) {
    SahSeg s;
    s.begin = 0; s.count = n; s.parent = -1; s.side = 0; s.bin_off = 0;
    for (int a = 0; a < 3; ++a) { s.clo[a] = sah_unkey(cbk[a]); s.chi[a] = sah_unkey(cbk[3 + a]); }
    seg[0] = s;
}

__global__ void sah_bins_reset_kernel(int n_ints, int32_t* __restrict__ bins) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_ints) return;
    const int f = i % kSahBinInts;
    bins[i] = f == 0 ? 0 : (f < 4 || (f >= 7 && f < 10) ? 0x7f800000 /* key(+inf) */ : (int32_t)0x807fffff /* key(-inf) */);
}

constexpr int kSahBinBlock = 256;
constexpr int kSahBinPerThread = 8;
constexpr int kSahWindow = 4 * 3 * kBvhBins;  // bins privatised per CTA: four whole segments

__device__ __forceinline__ void sah_bin_add(int32_t* b, bool shared, const SahItem& it, const float c[3]) {
    int32_t k[12];
    for (int a = 0; a < 3; ++a) {
        k[a] = sah_key(it.lo[a]); k[3 + a] = sah_key(it.hi[a]);
        k[6 + a] = sah_key(c[a]); k[9 + a] = k[6 + a];
    }
    if (shared) {
        atomicAdd_block(&b[0], 1);
        for (int j = 0; j < 3; ++j) { atomicMin_block(&b[1 + j], k[j]); atomicMax_block(&b[4 + j], k[3 + j]); }
        for (int j = 0; j < 3; ++j) { atomicMin_block(&b[7 + j], k[6 + j]); atomicMax_block(&b[10 + j], k[9 + j]); }
    } else {
        atomicAdd(&b[0], 1);
        for (int j = 0; j < 3; ++j) { atomicMin(&b[1 + j], k[j]); atomicMax(&b[4 + j], k[3 + j]); }
        for (int j = 0; j < 3; ++j) { atomicMin(&b[7 + j], k[6 + j]); atomicMax(&b[10 + j], k[9 + j]); }
    }
}

// Each CTA bins a chunk of items. Segments are numbered in item order, so the bins a chunk touches are
// contiguous: the first kSahWindow of them (from the chunk's first active segment) are accumulated in shared
// memory, the rest (small segments, where contention is low) go straight to global memory.
__global__ void __launch_bounds__(kSahBinBlock) sah_bin_kernel(int n, const SahItem* __restrict__ items, const SahSeg* __restrict__ segs,
                                                               int32_t* __restrict__ bins) {
    __shared__ int32_t s_bins[kSahWindow * kSahBinInts];
    __shared__ int32_t s_first;
    const int chunk = blockIdx.x * kSahBinBlock * kSahBinPerThread;
    if (threadIdx.x == 0) s_first = INT32_MAX;
    __syncthreads();
    for (int k = 0; k < kSahBinPerThread; ++k) {
        const int i = chunk + k * kSahBinBlock + threadIdx.x;
        if (i < n && items[i].seg >= 0) atomicMin_block(&s_first, segs[items[i].seg].bin_off);
    }
    __syncthreads();
    const int32_t w0 = s_first;
    if (w0 == INT32_MAX) return;  // nothing active in this chunk
    for (int k = threadIdx.x; k < kSahWindow * kSahBinInts; k += kSahBinBlock) {
        const int f = k % kSahBinInts;
        s_bins[k] = f == 0 ? 0 : (f < 4 || (f >= 7 && f < 10) ? 0x7f800000 : (int32_t)0x807fffff);
    }
    __syncthreads();
    for (int k = 0; k < kSahBinPerThread; ++k) {
        const int i = chunk + k * kSahBinBlock + threadIdx.x;
        if (i >= n) break;
        const SahItem it = items[i];
        if (it.seg < 0) continue;
        const SahSeg s = segs[it.seg];
        const int nb = sah_nb(s.count);
        float c[3];
        for (int a = 0; a < 3; ++a) c[a] = sah_centroid(it, a);
        for (int a = 0; a < 3; ++a) {
            const int b = s.bin_off + a * nb + sah_bin(c[a], s.clo[a], sah_scale(nb, s.clo[a], s.chi[a]), nb);
            const bool sh = b - w0 < kSahWindow;
            sah_bin_add(sh ? s_bins + (b - w0) * kSahBinInts : bins + (size_t)b * kSahBinInts, sh, it, c);
        }
    }
    __syncthreads();
    for (int k = threadIdx.x; k < kSahWindow; k += kSahBinBlock) {
        const int32_t* sb = s_bins + k * kSahBinInts;
        if (sb[0] == 0) continue;
        int32_t* gb = bins + (size_t)(w0 + k) * kSahBinInts;
        atomicAdd(&gb[0], sb[0]);
        for (int j = 0; j < 3; ++j) { atomicMin(&gb[1 + j], sb[1 + j]); atomicMax(&gb[4 + j], sb[4 + j]); }
        for (int j = 0; j < 3; ++j) { atomicMin(&gb[7 + j], sb[7 + j]); atomicMax(&gb[10 + j], sb[10 + j]); }
    }
}

// Inclusive scan of a bin (count + 12 bound keys) over lanes 0 .. 15, towards higher lanes (up) or lower (down).
template <bool kUp>
__device__ __forceinline__ void sah_bin_scan(int32_t v[kSahBinInts], int lane, int nb) {
    for (int d = 1; d < kBvhBins; d *= 2) {
        int32_t o[kSahBinInts];
        for (int j = 0; j < kSahBinInts; ++j) o[j] = kUp ? __shfl_up_sync(0xffffffffu, v[j], d) : __shfl_down_sync(0xffffffffu, v[j], d);
        const bool take = kUp ? lane >= d : lane + d < nb;
        if (take) {
            v[0] += o[0];
            for (int j = 0; j < 3; ++j) {
                v[1 + j] = min(v[1 + j], o[1 + j]); v[4 + j] = max(v[4 + j], o[4 + j]);
                v[7 + j] = min(v[7 + j], o[7 + j]); v[10 + j] = max(v[10 + j], o[10 + j]);
            }
        }
    }
}
__device__ __forceinline__ double sah_half_area(const int32_t v[kSahBinInts]) {
    const double dx = (double)sah_unkey(v[4]) - sah_unkey(v[1]), dy = (double)sah_unkey(v[5]) - sah_unkey(v[2]),
                 dz = (double)sah_unkey(v[6]) - sah_unkey(v[3]);
    if (!(dx >= 0) || !(dy >= 0) || !(dz >= 0)) return 0.0;
    return dx * dy + dy * dz + dz * dx;
}

// One warp per segment: BvhBuilder::build_range's choice of plane and its leaf rule, on the segment's bins.
__global__ void sah_decide_kernel(int n_segs, const SahSeg* __restrict__ segs, const int32_t* __restrict__ bins, int max_leaf, double c_trav,
                                  double c_prim, SahDecision* __restrict__ dec, uint32_t* __restrict__ inner_flag) {
    const int w = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= n_segs) return;  // (whole warps leave together)
    const SahSeg s = segs[w];
    const int n = s.count, nb = sah_nb(n);
    double best_cost = INFINITY;
    int best_axis = -1, best_split = -1, best_lc = 0;
    int32_t box[kSahBinInts];  // the segment's box: all bins of axis 0
    float cb[2][6];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        int32_t v[kSahBinInts];
        for (int j = 0; j < kSahBinInts; ++j) v[j] = lane < nb ? bins[(size_t)(s.bin_off + a * nb + lane) * kSahBinInts + j] : (j == 0 ? 0 : (j < 4 || (j >= 7 && j < 10) ? 0x7f800000 : (int32_t)0x807fffff));
        int32_t l[kSahBinInts], r[kSahBinInts];
        for (int j = 0; j < kSahBinInts; ++j) { l[j] = v[j]; r[j] = v[j]; }
        sah_bin_scan<true>(l, lane, nb);
        sah_bin_scan<false>(r, lane, nb);
        if (a == 0)
            for (int j = 0; j < kSahBinInts; ++j) box[j] = __shfl_sync(0xffffffffu, l[j], nb - 1);
        if (!(s.chi[a] > s.clo[a])) continue;  // all centroids share this coordinate: no plane
        int32_t rn[kSahBinInts];  // the right side of the plane after bin `lane`
        for (int j = 0; j < kSahBinInts; ++j) rn[j] = __shfl_down_sync(0xffffffffu, r[j], 1);
        double cost = INFINITY;
        if (lane < nb - 1 && l[0] > 0 && rn[0] > 0) cost = sah_half_area(l) * l[0] + sah_half_area(rn) * rn[0];
        double bc = cost;
        int bl = lane;
        for (int d = 16; d >= 1; d /= 2) {  // first minimum: smallest cost, then smallest plane
            const double oc = __shfl_xor_sync(0xffffffffu, bc, d);
            const int ol = __shfl_xor_sync(0xffffffffu, bl, d);
            if (oc < bc || (oc == bc && ol < bl)) { bc = oc; bl = ol; }
        }
        if (bc < best_cost) {
            best_cost = bc;
            best_axis = a;
            best_split = bl;
            best_lc = __shfl_sync(0xffffffffu, l[0], bl);
            for (int j = 0; j < 3; ++j) {
                cb[0][j] = sah_unkey(__shfl_sync(0xffffffffu, l[7 + j], bl));
                cb[0][3 + j] = sah_unkey(__shfl_sync(0xffffffffu, l[10 + j], bl));
                cb[1][j] = sah_unkey(__shfl_sync(0xffffffffu, rn[7 + j], bl));
                cb[1][3 + j] = sah_unkey(__shfl_sync(0xffffffffu, rn[10 + j], bl));
            }
        }
    }
    if (lane != 0) return;
    const double area = sah_half_area(box);
    bool leaf;
    if (n <= 1) leaf = true;
    else if (best_axis < 0) leaf = n <= max_leaf;  // all centroids coincide
    else if (n <= max_leaf) leaf = n * c_prim <= c_trav + (area > 0 ? best_cost / area : 0.0) * c_prim;
    else leaf = false;
    SahDecision d;
    for (int j = 0; j < 3; ++j) { d.box[j] = sah_unkey(box[1 + j]); d.box[3 + j] = sah_unkey(box[4 + j]); }
    d.inner = leaf ? 0 : 1;
    d.axis = best_axis;
    d.split = best_split;
    d.lc = best_lc;
    if (best_axis < 0 || best_lc <= 0 || best_lc >= n) {  // degenerate: split the index range; the bounds stay valid
        d.axis = -1;
        d.lc = n / 2;
        for (int k = 0; k < 2; ++k)
            for (int j = 0; j < 3; ++j) { cb[k][j] = s.clo[j]; cb[k][3 + j] = s.chi[j]; }
    }
    for (int k = 0; k < 2; ++k)
        for (int j = 0; j < 6; ++j) d.cb[k][j] = cb[k][j];
    dec[w] = d;
    inner_flag[w] = leaf ? 0u : 1u;
}

__device__ __forceinline__ void sah_set_child(BvhNode& nd, int side, const float b[6], int32_t code) {
    if (side == 0) {
        nd.c0x[0] = b[0]; nd.c0x[1] = b[3]; nd.c0y[0] = b[1]; nd.c0y[1] = b[4]; nd.c0z[0] = b[2]; nd.c0z[1] = b[5];
        nd.child0 = code;
    } else {
        nd.c1x[0] = b[0]; nd.c1x[1] = b[3]; nd.c1y[0] = b[1]; nd.c1y[1] = b[4]; nd.c1z[0] = b[2]; nd.c1z[1] = b[5];
        nd.child1 = code;
    }
}

// Node indices of the level's inner segments from the scan; children of inner segment j are segments 2j, 2j + 1
// of the next level (so the next level is numbered in item order too).
__global__ void sah_emit_kernel(int n_segs, const SahSeg* __restrict__ segs, const SahDecision* __restrict__ dec,
                                const uint32_t* __restrict__ inner_flag, const uint32_t* __restrict__ inner_idx, int32_t first_node,
                                int32_t first_record, BvhNode* __restrict__ nodes, SahSeg* __restrict__ next, uint32_t* __restrict__ next_bins,
                                uint32_t* __restrict__ n_inner) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_segs) return;
    const SahSeg s = segs[i];
    const SahDecision& d = dec[i];
    const uint32_t j = inner_idx[i];
    if (i == n_segs - 1) *n_inner = j + inner_flag[i];
    const int32_t code = d.inner ? first_node + (int32_t)j : ~(((first_record + s.begin) << 4) | s.count);
    if (s.parent >= 0) {
        sah_set_child(nodes[s.parent], s.side, d.box, code);
    } else if (!d.inner) {  // the whole world is one leaf: a root with one child, the other empty
        const float empty[6] = {FLT_MAX, FLT_MAX, FLT_MAX, -FLT_MAX, -FLT_MAX, -FLT_MAX};
        sah_set_child(nodes[first_node], 0, d.box, code);
        sah_set_child(nodes[first_node], 1, empty, kEmptyChild);
    }
    if (!d.inner) return;
    for (int k = 0; k < 2; ++k) {
        SahSeg c;
        c.begin = s.begin + (k == 0 ? 0 : d.lc);
        c.count = k == 0 ? d.lc : s.count - d.lc;
        c.parent = first_node + (int32_t)j;
        c.side = k;
        c.bin_off = 0;  // set after the scan of next_bins
        for (int a = 0; a < 3; ++a) { c.clo[a] = d.cb[k][a]; c.chi[a] = d.cb[k][3 + a]; }
        next[2 * j + k] = c;
        next_bins[2 * j + k] = 3u * (uint32_t)sah_nb(c.count);
    }
}

__global__ void sah_bin_off_kernel(int n_next, const uint32_t* __restrict__ off, SahSeg* __restrict__ next) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_next) next[i].bin_off = (int32_t)off[i];
}

__device__ __forceinline__ bool sah_goes_left(const SahItem& it, int pos, const SahSeg& s, const SahDecision& d) {
    if (d.axis < 0) return pos - s.begin < d.lc;
    const int nb = sah_nb(s.count), a = d.axis;
    return sah_bin(sah_centroid(it, a), s.clo[a], sah_scale(nb, s.clo[a], s.chi[a]), nb) <= d.split;
}

__global__ void sah_flag_kernel(int n, const SahItem* __restrict__ items, const SahSeg* __restrict__ segs, const SahDecision* __restrict__ dec,
                                uint32_t* __restrict__ flag) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const SahItem it = items[i];
    flag[i] = it.seg >= 0 && dec[it.seg].inner && sah_goes_left(it, i, segs[it.seg], dec[it.seg]) ? 1u : 0u;
}

// Stable partition of every inner segment: left items keep their order at [begin, + lc), right ones behind them.
__global__ void sah_scatter_kernel(int n, const SahItem* __restrict__ items, const SahSeg* __restrict__ segs, const SahDecision* __restrict__ dec,
                                   const uint32_t* __restrict__ inner_idx, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos,
                                   SahItem* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    SahItem it = items[i];
    if (it.seg < 0 || !dec[it.seg].inner) {
        it.seg = -1;
        out[i] = it;
        return;
    }
    const SahSeg s = segs[it.seg];
    const int lc = dec[it.seg].lc;
    const int left_before = (int)(pos[i] - pos[s.begin]);  // left items of this segment before position i
    const bool left = flag[i] != 0u;
    const int to = left ? s.begin + left_before : s.begin + lc + (i - s.begin - left_before);
    it.seg = 2 * (int32_t)inner_idx[it.seg] + (left ? 0 : 1);
    out[to] = it;
}

__global__ void sah_gather_kernel(int n, const SahItem* __restrict__ items, const Record* __restrict__ src, Record* __restrict__ dst) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = src[items[i].item];
}

struct SahBuildStats {
    int nodes = 0;                      // nodes written, root at node_base
    int depth = 0;                      // inner nodes on the longest root-to-leaf path (> max_depth: the build stopped there)
    int levels = 0;                     // level-synchronous passes
    unsigned long long launches = 0;    // kernels launched (cub's scans count as two each)
};

// Builds a binned-SAH BVH over n >= 2 boxes (d_boxes: 6 n floats, lo.xyz hi.xyz, rounded outward) into d_nodes
// (node indices node_base ..), and reorders the n world records at d_records into its leaf order. Leaf codes reference
// records first_record + position. Stops once the tree is deeper than max_depth (then stats->depth > max_depth and the
// tree is unusable). Nothing else in the arena refers to a world record by its position: the face records of
// REC_BOX items are pushed before the world's records and the media records after them (flatten.cpp, build_world).
inline cudaError_t sah_build(cudaStream_t stream, int n, const float* d_boxes, int32_t first_record, Record* d_records, int32_t node_base,
                             BvhNode* d_nodes, const BvhPolicy& pol, int max_depth, SahBuildStats* stats) {
    const size_t un = (size_t)n;
    SahBuildStats st;
    cudaError_t e = cudaSuccess;
    uint8_t* block = nullptr;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    // active segments hold >= 2 items, except children of one item: at most n per level; bins: 3 sah_nb(count) <= 3 count
    const size_t o_items = take(un * sizeof(SahItem)), o_items2 = take(un * sizeof(SahItem)), o_seg = take(un * sizeof(SahSeg)),
                 o_seg2 = take(un * sizeof(SahSeg)), o_dec = take(un * sizeof(SahDecision)), o_iflag = take(un * 4), o_iidx = take(un * 4),
                 o_nbins = take((2 * un + 1) * 4), o_boff = take((2 * un + 1) * 4), o_flag = take(un * 4), o_pos = take(un * 4),
                 o_bins = take(3 * un * kSahBinInts * 4), o_scalars = take(64);
    size_t scan_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const uint32_t*)nullptr, (uint32_t*)nullptr, 2 * n + 1, stream);
    const size_t o_cub = take(scan_bytes);
    if ((e = cudaMalloc(&block, off)) != cudaSuccess) return e;
    SahItem* items[2] = {(SahItem*)(block + o_items), (SahItem*)(block + o_items2)};
    SahSeg* segs[2] = {(SahSeg*)(block + o_seg), (SahSeg*)(block + o_seg2)};
    SahDecision* dec = (SahDecision*)(block + o_dec);
    uint32_t *iflag = (uint32_t*)(block + o_iflag), *iidx = (uint32_t*)(block + o_iidx), *nbins = (uint32_t*)(block + o_nbins),
             *boff = (uint32_t*)(block + o_boff), *flag = (uint32_t*)(block + o_flag), *pos = (uint32_t*)(block + o_pos);
    int32_t* bins = (int32_t*)(block + o_bins);
    int32_t* cbk = (int32_t*)(block + o_scalars);          // [6] root centroid bounds as keys
    uint32_t* n_inner = (uint32_t*)(block + o_scalars + 32);
    void* cub_temp = block + o_cub;
    const int tb = 256;
    const int gn = (n + tb - 1) / tb;
    {
        const int32_t init[6] = {0x7f800000, 0x7f800000, 0x7f800000, (int32_t)0x807fffff, (int32_t)0x807fffff, (int32_t)0x807fffff};
        e = cudaMemcpyAsync(cbk, init, sizeof(init), cudaMemcpyHostToDevice, stream);
    }
    if (e == cudaSuccess) {
        sah_init_kernel<<<gn, tb, 0, stream>>>(n, d_boxes, items[0], segs[0], cbk);
        sah_root_kernel<<<1, 1, 0, stream>>>(n, cbk, segs[0]);
        st.launches += 2;
        e = cudaGetLastError();
    }
    int n_segs = 1, cur = 0;
    uint32_t n_bins = 3u * (uint32_t)sah_nb(n);
    int32_t first_node = node_base;
    while (e == cudaSuccess && n_segs > 0) {
        const int n_ints = (int)n_bins * kSahBinInts;
        sah_bins_reset_kernel<<<(n_ints + tb - 1) / tb, tb, 0, stream>>>(n_ints, bins);
        sah_bin_kernel<<<(n + kSahBinBlock * kSahBinPerThread - 1) / (kSahBinBlock * kSahBinPerThread), kSahBinBlock, 0, stream>>>(n, items[cur], segs[cur],
                                                                                                                                   bins);
        sah_decide_kernel<<<(n_segs * 32 + tb - 1) / tb, tb, 0, stream>>>(n_segs, segs[cur], bins, pol.max_leaf, pol.cost_traverse, pol.cost_prim,
                                                                           dec, iflag);
        size_t cb = scan_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(cub_temp, cb, iflag, iidx, n_segs, stream)) != cudaSuccess) break;
        if ((e = cudaMemsetAsync(nbins, 0, (2 * (size_t)n_segs + 1) * 4, stream)) != cudaSuccess) break;
        const int gs = (n_segs + tb - 1) / tb;
        sah_emit_kernel<<<gs, tb, 0, stream>>>(n_segs, segs[cur], dec, iflag, iidx, first_node, first_record, d_nodes - node_base, segs[cur ^ 1], nbins,
                                               n_inner);
        cb = scan_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(cub_temp, cb, nbins, boff, 2 * n_segs + 1, stream)) != cudaSuccess) break;
        const int n_next_max = std::min(2 * n_segs, n);  // (an inner segment holds >= 2 items: at most n children)
        sah_bin_off_kernel<<<(n_next_max + tb - 1) / tb, tb, 0, stream>>>(n_next_max, boff, segs[cur ^ 1]);
        sah_flag_kernel<<<gn, tb, 0, stream>>>(n, items[cur], segs[cur], dec, flag);
        cb = scan_bytes;
        if ((e = cub::DeviceScan::ExclusiveSum(cub_temp, cb, flag, pos, n, stream)) != cudaSuccess) break;
        sah_scatter_kernel<<<gn, tb, 0, stream>>>(n, items[cur], segs[cur], dec, iidx, flag, pos, items[cur ^ 1]);
        st.launches += 13;
        if ((e = cudaGetLastError()) != cudaSuccess) break;
        uint32_t inner = 0;
        e = cudaMemcpyAsync(&inner, n_inner, sizeof(inner), cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(&n_bins, boff + 2 * n_segs, sizeof(n_bins), cudaMemcpyDeviceToHost, stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) break;
        ++st.levels;
        if (inner > 0) st.depth = st.levels;
        st.nodes += (int)inner;
        first_node += (int32_t)inner;
        n_segs = 2 * (int)inner;
        cur ^= 1;
        if (st.depth > max_depth) break;
    }
    if (st.nodes == 0) { st.nodes = 1; st.depth = 1; }  // the whole world is one leaf under a root of its own
    if (e == cudaSuccess && st.depth <= max_depth) {
        // records into leaf order, through a copy of the world's range (pos[] is free again: take the bins' space)
        Record* scratch = (Record*)bins;
        static_assert(sizeof(Record) <= 3 * kSahBinInts * 4, "the bins' space holds a record per item");
        e = cudaMemcpyAsync(scratch, d_records, un * sizeof(Record), cudaMemcpyDeviceToDevice, stream);
        if (e == cudaSuccess) {
            sah_gather_kernel<<<gn, tb, 0, stream>>>(n, items[cur], scratch, d_records);
            st.launches += 1;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    }
    cudaFree(block);
    if (stats) *stats = st;
    return e;
}

}  // namespace rtx
