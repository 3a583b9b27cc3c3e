// The row-per-lane board of the warp-per-chain SLS kernels (sls.cu: one chain per warp, sls_h16.cu: one chain per
// half-warp): lane r owns grid row r of the ceiling C, the supports S and the five cover-count planes c0..c4
// (sls_spec.hpp), and scores a candidate with shuffles of the rows of its reach window.
#pragma once
#include "sls_spec.hpp"

namespace tss {
namespace sls {

constexpr unsigned FULL = 0xffffffffu;

struct Lane {
    uint32_t C, S, c0, c1, c2, c3, c4, U, O;
};

__device__ __forceinline__ void derive(Lane& L) {
    uint32_t hi = L.c1 | L.c2 | L.c3 | L.c4;
    L.U = L.C & ~(L.c0 | hi);
    L.O = L.c0 & ~hi & L.C;  // (in WINDOW mode tiles covered by frozen supports are not a loss)
}

// Reach windows are 7 rows x 7 columns; window row dy is grid row y-3+dy, window column 0 is grid column
// ax = max(x-3, 0) (anchoring at 0 near the left edge keeps every extraction a single right shift).
__device__ __forceinline__ int anchor(int x) { return max(x - 3, 0); }

// Row `row` of the reach mask of site (x, y) in grid coordinates.
__device__ __forceinline__ uint32_t row_mask(uint2 win, int x, int y, int row) {
    int dy = row - y + 3;
    int d = min(max(dy, 0), 6);
    uint32_t m = d < 4 ? (win.x >> (7 * d)) : (win.y >> (7 * (d - 4)));
    m = dy == d ? (m & 0x7fu) : 0u;
    return m << anchor(x);
}

__device__ __forceinline__ void planes_add(Lane& L, uint32_t m) {
    uint32_t t;
    t = L.c0 & m; L.c0 ^= m; m = t;
    t = L.c1 & m; L.c1 ^= m; m = t;
    t = L.c2 & m; L.c2 ^= m; m = t;
    t = L.c3 & m; L.c3 ^= m; m = t;
    L.c4 ^= m;
}
__device__ __forceinline__ void planes_sub(Lane& L, uint32_t m) {
    uint32_t t;
    t = ~L.c0 & m; L.c0 ^= m; m = t;
    t = ~L.c1 & m; L.c1 ^= m; m = t;
    t = ~L.c2 & m; L.c2 ^= m; m = t;
    t = ~L.c3 & m; L.c3 ^= m; m = t;
    L.c4 ^= m;
}

// popcount(B & R(site at (x, y))) where B is a row-distributed bitboard (lane r of each group of WIDTH lanes holds row r)
// and `win` the site's reach window.  Every lane scores its own site; all 32 lanes must call.  The shuffles take the source
// row modulo WIDTH: rows outside the grid, or wrapped around it, meet zero window bits (with WIDTH = 16 the grid has at
// most 16 rows).
template <int WIDTH = 32>
__device__ __forceinline__ int score(uint32_t B, int x, int y, uint2 win) {
    const int ax = anchor(x);
    uint32_t lo = 0, hi = 0;
#pragma unroll
    for (int j = 6; j >= 4; j--) {
        uint32_t row = __shfl_sync(FULL, B, y - 3 + j, WIDTH);
        hi = hi * 128u + ((row >> ax) & 0x7fu);
    }
#pragma unroll
    for (int j = 3; j >= 0; j--) {
        uint32_t row = __shfl_sync(FULL, B, y - 3 + j, WIDTH);
        lo = lo * 128u + ((row >> ax) & 0x7fu);
    }
    return __popc(lo & win.x) + __popc(hi & win.y);
}

}  // namespace sls
}  // namespace tss
