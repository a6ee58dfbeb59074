// adaptive.cuh — adaptive sampling (rtx_render_adaptive): the kernels that decide, after each round, which 8x4 tiles
// keep sampling.
//
// Every pixel of a tile ends with the samples [spp_begin, spp_begin + n) of the uniform render, n shared by the tile.
// A second accumulator `aux` receives the samples with an odd global index only, so with even spp_begin and even n it
// holds n / 2 of them. The pixel error compares the two halves' means in the form Cycles uses, with the sqrt gamma of
// main.rs:217-225 in the denominator:
//     e_p = (|I_r - A_r| + |I_g - A_g| + |I_b - A_b|) / (1e-4 + sqrt(I_r + I_g + I_b)),  I = accum.rgb / accum.w,
//                                                                                          A = aux.rgb / aux.w
// A tile's error is the largest e_p over its pixels inside the frame. A tile stops for good after a round in which its
// error fell below the threshold, or when n reaches max_spp.
//
// The list of tiles that keep sampling holds dispenser order indices (tile_of_order) in ascending order: it is the same
// for the same errors, and consecutive entries stay in the dispenser's 32 x 128-pixel blocks.
#pragma once
#include <cub/device/device_scan.cuh>

#include "kernels.cuh"

namespace rtx {

constexpr int kAdaptiveBlock = 128;  // 4 tiles per CTA in the error kernel

// One warp per tile (row-major tile index, row 0 = top tiles), one lane per pixel. A pixel outside the frame, or one
// without samples in either buffer, contributes 0. Computed in f64: the two means are close, and their difference
// is what is measured.
__global__ void adaptive_error_kernel(const float4* __restrict__ accum, const float4* __restrict__ aux, int width, int height,
                                      int tiles_x, int n_tiles, float* __restrict__ tile_error) {
    const int tile = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (tile >= n_tiles) return;  // (whole warps)
    const int ty = tile / tiles_x, tx = tile - ty * tiles_x;
    const int px = tx * kTileW + (lane & (kTileW - 1));
    const int row = ty * kTileH + lane / kTileW;
    float e = 0.f;
    if (px < width && row < height) {
        const float4 s = accum[(size_t)row * width + px], h = aux[(size_t)row * width + px];
        if (s.w > 0.f && h.w > 0.f) {
            const double ir = (double)s.x / s.w, ig = (double)s.y / s.w, ib = (double)s.z / s.w;
            const double ar = (double)h.x / h.w, ag = (double)h.y / h.w, ab = (double)h.z / h.w;
            e = (float)((fabs(ir - ar) + fabs(ig - ag) + fabs(ib - ab)) / (1e-4 + sqrt(ir + ig + ib)));
        }
    }
    for (int off = 16; off > 0; off >>= 1) e = fmaxf(e, __shfl_xor_sync(0xffffffffu, e, off));
    if (lane == 0) tile_error[tile] = e;
}

// flag[k] for dispenser order index k: 1 while tile_of_order(k) keeps sampling. tile_error == nullptr starts the frame
// (every tile samples); otherwise a tile stops when its error is below the threshold (a NaN error does not stop it).
__global__ void adaptive_flag_kernel(const float* __restrict__ tile_error, double threshold, int tiles_x, int tiles_y,
                                     float inv_per_block_row, uint32_t* __restrict__ flag) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= tiles_x * tiles_y) return;
    if (!tile_error) { flag[k] = 1u; return; }
    if (!flag[k]) return;
    int tx, ty;
    tile_of_order((unsigned int)k, tiles_x, tiles_y, inv_per_block_row, tx, ty);
    if ((double)tile_error[ty * tiles_x + tx] < threshold) flag[k] = 0u;
}

// What the host reads back after each decision.
struct AdaptiveRound {
    unsigned long long tiles;   // entries of the list
    unsigned long long pixels;  // pixels of those tiles inside the frame
};

// list[pos[k]] = k for every flagged k (pos = exclusive scan of flag), plus the list's length and pixel count.
__global__ void adaptive_scatter_kernel(const uint32_t* __restrict__ flag, const uint32_t* __restrict__ pos, int width, int height,
                                        int tiles_x, int tiles_y, float inv_per_block_row, uint32_t* __restrict__ list,
                                        AdaptiveRound* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = tiles_x * tiles_y;
    if (k >= n) return;
    if (k == n - 1) out->tiles = (unsigned long long)(pos[k] + flag[k]);
    if (!flag[k]) return;
    list[pos[k]] = (uint32_t)k;
    int tx, ty;
    tile_of_order((unsigned int)k, tiles_x, tiles_y, inv_per_block_row, tx, ty);
    const int w = min(kTileW, width - tx * kTileW), h = min(kTileH, height - ty * kTileH);
    atomicAdd(&out->pixels, (unsigned long long)(w * h));
}

// max_depth == 0: color() is black (main.rs:27-29), only the sample counts of the listed tiles move.
__global__ void adaptive_black_kernel(const uint32_t* __restrict__ list, int n_list, int width, int height, int tiles_x, int tiles_y,
                                      float inv_per_block_row, int spp_begin, int spp_count, float4* __restrict__ accum,
                                      float4* __restrict__ aux) {
    const int j = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (j >= n_list) return;
    int tx, ty;
    tile_of_order(list[j], tiles_x, tiles_y, inv_per_block_row, tx, ty);
    const int px = tx * kTileW + (lane & (kTileW - 1));
    const int row = ty * kTileH + lane / kTileW;
    if (px >= width || row >= height) return;
    // odd global indices in [spp_begin, spp_begin + spp_count)
    const int odd = (spp_begin + spp_count) / 2 - spp_begin / 2;
    accum[(size_t)row * width + px].w += (float)spp_count;
    aux[(size_t)row * width + px].w += (float)odd;
}

}  // namespace rtx
