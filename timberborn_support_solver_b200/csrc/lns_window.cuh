// Bitboard helpers of the window decompositions on grids larger than 32x32: the 1x1 search (lns.cu) and the placement
// search (lns_placements.cu).  Grids are bit-packed rows of wpr = ceil(w / 32) words, bit x of word x / 32 = column x.
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

namespace tss {
namespace lns {

// dst = (src | its 4-neighbours) & C: one ceiling-masked dilation step (validate(), platform_layout.rs:127-141).
// (static: every translation unit that launches it owns a copy)
static __global__ void dilate_global_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst, const uint32_t* __restrict__ C, int nw, int wpr) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nw) return;
    int col = i % wpr;
    uint32_t x = src[i], l = x << 1, r = x >> 1;
    if (col > 0) l |= src[i - 1] >> 31;
    if (col + 1 < wpr) r |= src[i + 1] << 31;
    uint32_t up = i >= wpr ? src[i - wpr] : 0u, down = i + wpr < nw ? src[i + wpr] : 0u;
    dst[i] = (x | l | r | up | down) & C[i];
}

// 32 bits of row gy of a bit-packed grid starting at column gx0 (may be negative / beyond the grid: zeros)
__device__ __forceinline__ uint32_t fetch32(const uint32_t* __restrict__ X, int gy, int gx0, int h, int wpr) {
    if (gy < 0 || gy >= h) return 0u;
    int wq = gx0 >> 5, sh = gx0 & 31;  // arithmetic shift: floor division also for negative gx0
    uint32_t lo = (wq >= 0 && wq < wpr) ? X[gy * wpr + wq] : 0u;
    uint32_t hi = (wq + 1 >= 0 && wq + 1 < wpr) ? X[gy * wpr + wq + 1] : 0u;
    return __funnelshift_r(lo, hi, sh);
}

}  // namespace lns
}  // namespace tss
