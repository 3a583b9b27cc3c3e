// The fractional packing lower bound of lp.cu on grids larger than 32x32 (up to 256x256), solved by a first-order method
// instead of the dense simplex: C4 (256x256, p = 0.7) has 45 903 ceiling tiles and as many 1x1 placements, a tableau of
// 2 * 10^9 cells.  The certificate is lp.cu's and needs no optimality: any y >= 0 is rounded to integer weights and every
// in-bounds placement's load is recomputed exactly, so the bound is valid whatever the iteration did.
//
// The LP  max 1'y  s.t.  R y <= c,  y >= 0  is the zero-sum game  min over tile distributions y of max over placements p of
// (R y)_p / c_p  (value 1 / LP optimum).  Both players run optimistic multiplicative weights:
//     g = (R y)_p / c_p,   z_pi += 2 g - g_prev,   pi ∝ exp( eta z_pi)
//     h = R' (pi / c),     z_y  += 2 h - h_prev,   y  ∝ exp(-eta z_y)
// Every iterate y, and every AVG_EVERY iterations the average of the iterates so far, gives the bound sum(y) / max_p g_p; the best
// one is kept.  The step that works scales with the size of the problem (eta ≈ 0.3 / game value on 32x32 and on 256x256 alike),
// so eta = ETA0 / (smallest max_p g_p seen so far): the loads normalised by the current maximum.
//
// Reach sets: one (kw + 6) x (kh + 6) bit window per placement (key, anchor), window row r = grid row ay - 3 + r, bit c = grid
// column ax - 3 + c; at most 12 rows of 16 bits, stored row-major by (key, row) over the anchor grid so that neighbouring
// threads (neighbouring anchors) read neighbouring words.  Both products are GATHERS over these windows (a tile tests its bit
// in the window of every placement whose window contains it): no atomics, every sum in a fixed order, so two calls give the
// same weights bit for bit.
//
// Kernels: lpb_reach_kernel (windows and the constraint flags), lpb_dead_kernel (the tiles fixed at 0 under a placement that costs
// nothing), lpb_iterate_kernel (persistent, cooperative: one grid barrier after the placement phase, one after the tile phase, one
// after each evaluation of the averaged iterate), lpb_weights_kernel + lpb_certify_kernel (integer certificate over every
// in-bounds placement).
#include <cooperative_groups.h>

#include <algorithm>
#include <cfloat>
#include <cmath>

#include "engine.hpp"
#include "lns_window.cuh"

namespace cg = cooperative_groups;

namespace tss {
namespace lpb {

constexpr int MAX_KEYS = 16;
constexpr int MAX_KEY_DIM = 6;                     // window rows kh + 6 <= 12, columns kw + 6 <= 12 (16-bit rows)
constexpr int WROWS = MAX_KEY_DIM + 6;
constexpr int HALO = kTerrainSupportDistance - 1;  // three dilations around the footprint
constexpr int THREADS = 256;
constexpr float ETA0 = 0.3f;                       // step relative to the game value (see above)
constexpr float EXP_CAP = 60.0f;                   // exponent clamp: the shifts lag one iteration behind (see lpb_iterate_kernel)
constexpr int AVG_EVERY = 50;                      // iterations between two evaluations of the averaged iterate

struct Keys {
    int n;
    int w[MAX_KEYS], h[MAX_KEYS];
    int cost[MAX_KEYS];
    float inv_cost[MAX_KEYS];   // 0 for a key that costs nothing (its placements are no constraints)
};

// Scalars carried from one iteration (and one launch) to the next; read at the start of a launch, written at its end.
struct State {
    double inv_sy;     // 1 / sum of the current y
    float shift_pi;    // largest eta z_pi of the previous placement phase
    float shift_y;     // largest -eta z_y of the previous tile phase
    float maxg_best;   // smallest max_p g_p seen (FLT_MAX before the first iteration)
    float best;        // best bound sum(y) / max g so far (floating point)
    int iterations;
    int pad;
};

struct Part { double sum, sum2; float max_a, max_b; };

// reach windows of every placement; cons[p] = 1 if p is a constraint of the iteration (its reach holds ceiling, it costs
// something); n_cons counts them.  Tiles in the reach of a placement that costs nothing can carry no weight: dead[t] = 1.
__global__ void __launch_bounds__(THREADS) lpb_reach_kernel(const uint32_t* __restrict__ C, int W, int H, int wpr, Keys keys, uint16_t* __restrict__ reach,
                                                            uint8_t* __restrict__ cons, int* __restrict__ n_cons) {
    const int WH = W * H;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= keys.n * WH) return;
    const int k = p / WH, a = p - k * WH, ay = a / W, ax = a - ay * W, kw = keys.w[k], kh = keys.h[k];
    const int rows = kh + 2 * HALO;
    const uint32_t wmask = (1u << (kw + 2 * HALO)) - 1u;
    uint32_t Cw[WROWS], X[WROWS];
    const bool in_bounds = ax + kw <= W && ay + kh <= H;
#pragma unroll
    for (int r = 0; r < WROWS; r++) {
        Cw[r] = (in_bounds && r < rows) ? lns::fetch32(C, ay - HALO + r, ax - HALO, H, wpr) & wmask : 0u;
        X[r] = (r >= HALO && r < HALO + kh) ? Cw[r] & (((1u << kw) - 1u) << HALO) : 0u;
    }
#pragma unroll
    for (int d = 0; d < HALO; d++) {
        uint32_t Y[WROWS];
#pragma unroll
        for (int r = 0; r < WROWS; r++) Y[r] = (X[r] | (X[r] << 1) | (X[r] >> 1) | (r > 0 ? X[r - 1] : 0u) | (r + 1 < WROWS ? X[r + 1] : 0u)) & Cw[r];
#pragma unroll
        for (int r = 0; r < WROWS; r++) X[r] = Y[r];
    }
    bool any = false;
#pragma unroll
    for (int r = 0; r < WROWS; r++) {
        reach[((size_t)k * WROWS + r) * WH + a] = (uint16_t)X[r];
        any = any || X[r] != 0u;
    }
    const bool is_con = any && keys.cost[k] > 0;
    cons[p] = is_con ? 1 : 0;
    if (is_con) atomicAdd(n_cons, 1);
}

// Visit every placement p (key k, anchor (ax, ay)) whose reach holds tile (tx, ty): f(k, anchor index).
template <class F>
__device__ __forceinline__ void for_placements_over(const uint16_t* __restrict__ reach, const Keys& keys, int W, int H, int tx, int ty, F f) {
    const int WH = W * H;
    for (int k = 0; k < keys.n; k++) {
        const int kw = keys.w[k], kh = keys.h[k];
        for (int r = 0; r < kh + 2 * HALO; r++) {
            const int ay = ty + HALO - r;
            if (ay < 0 || ay > H - kh) continue;
            const uint16_t* row = reach + ((size_t)k * WROWS + r) * WH + (size_t)ay * W;
            for (int c = 0; c < kw + 2 * HALO; c++) {
                const int ax = tx + HALO - c;
                if (ax < 0 || ax > W - kw) continue;
                if ((row[ax] >> c) & 1u) f(k, ay * W + ax);
            }
        }
    }
}

// dead[t] = 1 for the tiles in the reach of a placement that costs nothing (fixed at y = 0), live[t] otherwise for ceiling
__global__ void __launch_bounds__(THREADS) lpb_dead_kernel(const uint32_t* __restrict__ C, int W, int H, int wpr, const uint16_t* __restrict__ reach, Keys keys,
                                                           uint8_t* __restrict__ live) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= W * H) return;
    const int ty = t / W, tx = t - ty * W;
    bool ceiling = (C[(size_t)ty * wpr + (tx >> 5)] >> (tx & 31)) & 1u, dead = false;
    if (ceiling)
        for_placements_over(reach, keys, W, H, tx, ty, [&](int k, int) { dead = dead || keys.cost[k] == 0; });
    live[t] = ceiling && !dead ? 1 : 0;
}

__device__ __forceinline__ Part part_merge(Part a, Part b) { return Part{a.sum + b.sum, a.sum2 + b.sum2, fmaxf(a.max_a, b.max_a), fmaxf(a.max_b, b.max_b)}; }

// block-wide reduction in a fixed order; the result is valid in every thread
__device__ __forceinline__ Part block_reduce(Part v, Part* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
        v = part_merge(v, Part{__shfl_xor_sync(0xffffffffu, v.sum, o), __shfl_xor_sync(0xffffffffu, v.sum2, o), __shfl_xor_sync(0xffffffffu, v.max_a, o),
                               __shfl_xor_sync(0xffffffffu, v.max_b, o)});
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    Part r = red[0];
    for (int i = 1; i < THREADS / 32; i++) r = part_merge(r, red[i]);
    return r;
}

// the G block partials of a phase, folded identically by every block
__device__ __forceinline__ Part grid_fold(const Part* __restrict__ parts, int G, Part* red) {
    Part v{0.0, 0.0, -FLT_MAX, -FLT_MAX};
    for (int i = threadIdx.x; i < G; i += blockDim.x)
        v = part_merge(v, Part{__ldcg(&parts[i].sum), __ldcg(&parts[i].sum2), __ldcg(&parts[i].max_a), __ldcg(&parts[i].max_b)});
    return block_reduce(v, red);
}

// sum of v over the reach of placement (k, anchor a), in the window's bit order
template <class T, class A>
__device__ __forceinline__ A window_sum(const uint16_t* __restrict__ reach, const T* __restrict__ v, int W, int WH, int kh, int k, int a, A acc) {
    const int ay = a / W, ax = a - ay * W;
    for (int r = 0; r < kh + 2 * HALO; r++) {
        const T* row = v + (ptrdiff_t)(ay - HALO + r) * W + (ax - HALO);
        for (uint32_t bits = reach[((size_t)k * WROWS + r) * WH + a]; bits; bits &= bits - 1u) acc += (A)row[__ffs(bits) - 1];
    }
    return acc;
}

// Iterations [state.iterations, it1) of the optimistic multiplicative weights, resumable: everything an iteration needs is in
// global memory.
//   placement phase: g = load / (c sum y); z_pi, g_prev; q = pi / c unnormalised (exp(eta z_pi - shift_pi)); partials: sum of the
//                    pi weights, max eta z_pi, max g
//   tile phase:      if the placement phase found a better bound, ybest = y scaled to LP feasibility (max load / c = 1);
//                    h = cov / sum pi; z_y, h_prev; y = exp(-eta z_y - shift_y); yavg += y / sum y; partials: sum y, max -eta z_y,
//                    sum yavg
//   every AVG_EVERY iterations, a third phase: the bound of the averaged iterate, which converges where the last iterate still
//                    oscillates (32x32 .. 48x48 terrains in a CPU model: 99.3-99.5 % of the LP after 2 000 iterations against 87-97 %)
// The shifts are the maxima of the previous phase of the same kind (one grid barrier per phase instead of two); the exponents are
// clamped at EXP_CAP so that a lagging shift cannot overflow.  The certificate does not depend on any of it.
__global__ void __launch_bounds__(THREADS, 4) lpb_iterate_kernel(const uint16_t* __restrict__ reach, const uint8_t* __restrict__ cons, const uint8_t* __restrict__ live,
                                                              int W, int H, Keys keys, int it1, float* __restrict__ z_pi, float* __restrict__ g_prev,
                                                              float* __restrict__ q, float* __restrict__ z_y, float* __restrict__ h_prev, float* __restrict__ y,
                                                              float* __restrict__ yavg, float* __restrict__ ybest, Part* __restrict__ parts /* [3][G] */,
                                                              State* __restrict__ state) {
    cg::grid_group grid = cg::this_grid();
    __shared__ Part red[THREADS / 32];
    const int G = (int)gridDim.x, WH = W * H, n_place = keys.n * WH;
    const int stride = G * THREADS, gtid = blockIdx.x * THREADS + threadIdx.x;
    State s = *state;
    for (int it = s.iterations; it < it1; it++) {
        const float eta = s.maxg_best < FLT_MAX ? ETA0 / s.maxg_best : 0.0f;
        const float inv_sy = (float)s.inv_sy;
        Part v{0.0, 0.0, -FLT_MAX, 0.0f};
        for (int p = gtid; p < n_place; p += stride) {
            if (!cons[p]) continue;
            const int k = p / WH, a = p - k * WH;
            const float g = window_sum(reach, y, W, WH, keys.h[k], k, a, 0.0f) * inv_sy * keys.inv_cost[k];
            const float z = z_pi[p] + 2.0f * g - g_prev[p];
            z_pi[p] = z;
            g_prev[p] = g;
            const float e = __expf(fminf(eta * z - s.shift_pi, EXP_CAP));
            q[p] = e * keys.inv_cost[k];
            v.sum += (double)e;
            v.max_a = fmaxf(v.max_a, eta * z);
            v.max_b = fmaxf(v.max_b, g);
        }
        v = block_reduce(v, red);
        if (threadIdx.x == 0) parts[blockIdx.x] = v;
        grid.sync();
        const Part P = grid_fold(parts, G, red);
        const float maxg = P.max_b;
        const bool improved = maxg > 0.0f && 1.0f / maxg > s.best;
        const float to_feasible = maxg > 0.0f ? inv_sy / maxg : 0.0f;   // y / (sum y * max g): max load / c = 1
        if (improved) s.best = 1.0f / maxg;
        if (maxg > 0.0f) s.maxg_best = fminf(s.maxg_best, maxg);
        s.shift_pi = P.max_a;
        const float eta2 = s.maxg_best < FLT_MAX ? ETA0 / s.maxg_best : 0.0f;
        const float inv_spi = P.sum > 0.0 ? (float)(1.0 / P.sum) : 0.0f;
        Part u{0.0, 0.0, -FLT_MAX, 0.0f};
        for (int t = gtid; t < WH; t += stride) {
            if (improved) ybest[t] = y[t] * to_feasible;
            if (!live[t]) continue;
            const int ty = t / W, tx = t - ty * W;
            float cov = 0.0f;
            for_placements_over(reach, keys, W, H, tx, ty, [&](int k, int a) { cov += q[(size_t)k * WH + a]; });
            const float h = cov * inv_spi;
            const float z = z_y[t] + 2.0f * h - h_prev[t];
            z_y[t] = z;
            h_prev[t] = h;
            const float ya = yavg[t] + y[t] * inv_sy;
            yavg[t] = ya;
            const float yt = __expf(fminf(-eta2 * z - s.shift_y, EXP_CAP));
            y[t] = yt;
            u.sum += (double)yt;
            u.sum2 += (double)ya;
            u.max_a = fmaxf(u.max_a, -eta2 * z);
        }
        u = block_reduce(u, red);
        if (threadIdx.x == 0) parts[G + blockIdx.x] = u;
        grid.sync();
        const Part Q = grid_fold(parts + G, G, red);
        s.inv_sy = Q.sum > 0.0 ? 1.0 / Q.sum : 0.0;
        s.shift_y = Q.max_a;
        s.iterations = it + 1;
        const float avg_sum = (float)Q.sum2;
        if ((it + 1) % AVG_EVERY == 0) {
            Part w{0.0, 0.0, -FLT_MAX, 0.0f};
            for (int p = gtid; p < n_place; p += stride) {
                if (!cons[p]) continue;
                const int k = p / WH;
                w.max_b = fmaxf(w.max_b, window_sum(reach, yavg, W, WH, keys.h[k], k, p - k * WH, 0.0f) * keys.inv_cost[k]);
            }
            w = block_reduce(w, red);
            if (threadIdx.x == 0) parts[2 * G + blockIdx.x] = w;
            grid.sync();
            const float maxl = grid_fold(parts + 2 * G, G, red).max_b;
            if (maxl > 0.0f && avg_sum / maxl > s.best) {   // (ybest is next read after the kernel; yavg next written after a barrier)
                s.best = avg_sum / maxl;
                const float to_feasible_avg = 1.0f / maxl;
                for (int t = gtid; t < WH; t += stride) ybest[t] = yavg[t] * to_feasible_avg;
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *state = s;
}

// the start: y = 1 on every live tile, everything else 0
__global__ void lpb_init_kernel(const uint8_t* __restrict__ live, int WH, float* __restrict__ y, float* __restrict__ yavg, float* __restrict__ ybest,
                                float* __restrict__ z_y, float* __restrict__ h_prev) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= WH) return;
    y[t] = live[t] ? 1.0f : 0.0f;
    yavg[t] = ybest[t] = z_y[t] = h_prev[t] = 0.0f;
}

// integer weights k_t = floor(ybest_t * scale) (lp.cu's rule), their sum into out[0]
__global__ void lpb_weights_kernel(const float* __restrict__ ybest, int WH, double scale, int* __restrict__ weights, unsigned long long* __restrict__ out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    long long k = 0;
    if (t < WH) {
        const double v = (double)ybest[t];
        k = v > 0.0 ? (long long)floor(v * scale) : 0ll;
        k = k > (1ll << 30) ? (1ll << 30) : k;
        weights[t] = (int)k;
    }
    for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xffffffffu, k, o);
    if ((threadIdx.x & 31) == 0 && k) atomicAdd(&out[0], (unsigned long long)k);
}

// lp_certify_kernel's certificate over EVERY in-bounds placement, in 64-bit integers: out[1] = max load, out[2] = min over
// placements with load > 0 of ceil(total * cost / load)
__global__ void __launch_bounds__(THREADS) lpb_certify_kernel(const uint16_t* __restrict__ reach, int W, int H, Keys keys, const int* __restrict__ weights,
                                                              unsigned long long* __restrict__ out) {
    const int WH = W * H;
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= keys.n * WH) return;
    const int k = p / WH, a = p - k * WH, ay = a / W, ax = a - ay * W;
    if (ax + keys.w[k] > W || ay + keys.h[k] > H) return;
    long long load = 0;
    for (int r = 0; r < keys.h[k] + 2 * HALO; r++) {
        const int* wrow = weights + (ptrdiff_t)(ay - HALO + r) * W + (ax - HALO);
        for (uint32_t bits = reach[((size_t)k * WROWS + r) * WH + a]; bits; bits &= bits - 1u) load += wrow[__ffs(bits) - 1];
    }
    if (load > 0) {
        const unsigned long long num = __ldcg(&out[0]) * (unsigned long long)keys.cost[k];
        atomicMax(&out[1], (unsigned long long)load);
        atomicMin(&out[2], (num + (unsigned long long)load - 1ull) / (unsigned long long)load);
    }
}

}  // namespace lpb

// Grids larger than 32x32 (up to 256x256): rows_host bit-packed (wpr = ceil(W / 32) words per row); key_dims at most 16 keys, each at
// most 6x6; key_costs 0..4096.  max_iters <= 0: the default.  target > 0: stop once the certified bound reaches it, checked every
// CHECK iterations.  out_weights[W * H] (host); totals / info as in lp_run: info = (iterations, 0, constraints).
int lp_big_run(tss_engine* e, const uint32_t* rows_host, int W, int H, const std::vector<int2>& key_dims, const std::vector<int>& key_costs, int max_iters,
               long long target, int* out_weights, unsigned long long* totals, int* info) {
    constexpr int DEFAULT_ITERS = 3000, CHECK = 250;
    if (W > 256 || H > 256) return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound_lp: grids larger than 256x256 are not supported (got %dx%d)", W, H);
    if ((int)key_dims.size() > lpb::MAX_KEYS) return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound_lp: more than %d dims keys on a grid larger than 32x32", lpb::MAX_KEYS);
    lpb::Keys keys{};
    keys.n = (int)key_dims.size();
    int max_cost = 1;
    for (int i = 0; i < keys.n; i++) {
        const int2 d = key_dims[(size_t)i];
        if (d.x > lpb::MAX_KEY_DIM || d.y > lpb::MAX_KEY_DIM)
            return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound_lp: platforms larger than %dx%d are not supported on grids larger than 32x32 (got %dx%d)",
                           lpb::MAX_KEY_DIM, lpb::MAX_KEY_DIM, d.x, d.y);
        keys.w[i] = d.x; keys.h[i] = d.y; keys.cost[i] = key_costs[(size_t)i];
        keys.inv_cost[i] = key_costs[(size_t)i] > 0 ? 1.0f / (float)key_costs[(size_t)i] : 0.0f;
        max_cost = std::max(max_cost, key_costs[(size_t)i]);
    }
    double scale = (double)(1 << 20);             // lp.cu's rule: y_t <= the largest cost, keep floor(y * scale) below 2^30
    while (scale * (double)max_cost > (double)(1 << 30)) scale *= 0.5;
    const int WH = W * H, wpr = (W + 31) / 32, n_place = keys.n * WH;
    totals[0] = totals[1] = totals[2] = 0;
    info[0] = info[1] = info[2] = 0;
    // scratch slot 6: reach windows u16 [keys][12][WH] | C rows [H * wpr] | cons u8 [n_place] | live u8 [WH]
    // slot 5: z_pi, g_prev, q [n_place] floats | z_y, h_prev, y, yavg, ybest [WH] floats | weights int [WH]
    // slot 4: partials [3][G] | state | n_cons | totals u64 [3]      (C4 with the 13 keys of the default set: 21 MB + 11 MB + 1 MB)
    const size_t reach_bytes = sizeof(uint16_t) * (size_t)keys.n * lpb::WROWS * WH;
    const size_t c_off = (reach_bytes + 15) & ~(size_t)15, cons_off = c_off + sizeof(uint32_t) * (size_t)H * wpr, live_off = cons_off + (size_t)n_place;
    unsigned char* s6 = (unsigned char*)e->dev(6, live_off + (size_t)WH);
    if (!s6) return TSS_E_CUDA;
    uint16_t* reach = (uint16_t*)s6;
    uint32_t* C = (uint32_t*)(s6 + c_off);
    uint8_t *cons = s6 + cons_off, *live = s6 + live_off;
    float* f = (float*)e->dev(5, sizeof(float) * (3 * (size_t)n_place + 5 * (size_t)WH) + sizeof(int) * (size_t)WH);
    if (!f) return TSS_E_CUDA;
    float *z_pi = f, *g_prev = z_pi + n_place, *q = g_prev + n_place, *z_y = q + n_place, *h_prev = z_y + WH, *y = h_prev + WH, *yavg = y + WH, *ybest = yavg + WH;
    int* weights = (int*)(ybest + WH);

    int per_sm = 0;
    TSS_CUDA(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, lpb::lpb_iterate_kernel, lpb::THREADS, 0));
    int coop = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, e->device);
    if (!coop || per_sm < 1) return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound_lp: grids larger than 32x32 need a device with cooperative launch");
    const int G = e->prop.multiProcessorCount * std::min(per_sm, 4);
    unsigned char* s4 = (unsigned char*)e->dev(4, sizeof(lpb::Part) * 3 * (size_t)G + sizeof(lpb::State) + 16 + sizeof(unsigned long long) * 3);
    if (!s4) return TSS_E_CUDA;
    lpb::Part* parts = (lpb::Part*)s4;
    lpb::State* state = (lpb::State*)(parts + 3 * (size_t)G);
    int* n_cons = (int*)(state + 1);
    unsigned long long* totals_dev = (unsigned long long*)(((uintptr_t)(n_cons + 1) + 7) & ~(uintptr_t)7);

    TSS_CUDA(e, cudaMemcpyAsync(C, rows_host, sizeof(uint32_t) * (size_t)H * wpr, cudaMemcpyHostToDevice, e->stream));
    const lpb::State s0{0.0, 0.0f, 0.0f, FLT_MAX, 0.0f, 0, 0};
    TSS_CUDA(e, cudaMemcpyAsync(state, &s0, sizeof s0, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaMemsetAsync(n_cons, 0, sizeof(int), e->stream));
    TSS_CUDA(e, cudaMemsetAsync(f, 0, sizeof(float) * 3 * (size_t)n_place, e->stream));
    TSS_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    lpb::lpb_reach_kernel<<<(n_place + lpb::THREADS - 1) / lpb::THREADS, lpb::THREADS, 0, e->stream>>>(C, W, H, wpr, keys, reach, cons, n_cons);
    lpb::lpb_dead_kernel<<<(WH + lpb::THREADS - 1) / lpb::THREADS, lpb::THREADS, 0, e->stream>>>(C, W, H, wpr, reach, keys, live);
    lpb::lpb_init_kernel<<<(WH + lpb::THREADS - 1) / lpb::THREADS, lpb::THREADS, 0, e->stream>>>(live, WH, y, yavg, ybest, z_y, h_prev);
    TSS_CHECK_LAUNCH(e);
    // inv_sy of the start (y = 1 on every live tile) comes from the first tile phase's fold otherwise: set it from the live count
    std::vector<uint8_t> live_host((size_t)WH);
    TSS_CUDA(e, cudaMemcpyAsync(live_host.data(), live, (size_t)WH, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(&info[2], n_cons, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    long long n_live = 0;
    for (uint8_t v : live_host) n_live += v;
    lpb::State s1 = s0;
    s1.inv_sy = n_live > 0 ? 1.0 / (double)n_live : 0.0;
    TSS_CUDA(e, cudaMemcpyAsync(state, &s1, sizeof s1, cudaMemcpyHostToDevice, e->stream));
    int launches = 5;

    const int cap = max_iters > 0 ? max_iters : DEFAULT_ITERS;
    int done = 0;
    unsigned long long t[3] = {0, 0, 0};
    while (true) {
        const int next = target > 0 ? std::min(cap, done + CHECK) : cap;
        if (next > done && n_live > 0 && info[2] > 0) {
            int it1 = next;
            void* args[] = {&reach, &cons, &live, &W, &H, &keys, &it1, &z_pi, &g_prev, &q, &z_y, &h_prev, &y, &yavg, &ybest, &parts, &state};
            TSS_CUDA(e, cudaLaunchCooperativeKernel((const void*)lpb::lpb_iterate_kernel, dim3(G), dim3(lpb::THREADS), args, 0, e->stream));
            launches++;
        }
        done = next;
        const unsigned long long init[3] = {0ull, 0ull, ~0ull};
        TSS_CUDA(e, cudaMemcpyAsync(totals_dev, init, sizeof init, cudaMemcpyHostToDevice, e->stream));
        lpb::lpb_weights_kernel<<<(WH + lpb::THREADS - 1) / lpb::THREADS, lpb::THREADS, 0, e->stream>>>(ybest, WH, scale, weights, totals_dev);
        lpb::lpb_certify_kernel<<<(n_place + lpb::THREADS - 1) / lpb::THREADS, lpb::THREADS, 0, e->stream>>>(reach, W, H, keys, weights, totals_dev);
        TSS_CHECK_LAUNCH(e);
        launches += 2;
        TSS_CUDA(e, cudaMemcpyAsync(t, totals_dev, sizeof t, cudaMemcpyDeviceToHost, e->stream));
        TSS_CUDA(e, cudaStreamSynchronize(e->stream));
        const bool reached = target > 0 && t[1] > 0 && t[2] != ~0ull && (long long)t[2] >= target;
        if (done >= cap || reached || n_live == 0 || info[2] == 0) break;
    }
    TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(out_weights, weights, sizeof(int) * (size_t)WH, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    float ms = 0;
    if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) != cudaSuccess) cudaGetLastError();
    e->stats.device_ms = ms;
    e->stats.kernel_launches += launches;
    totals[0] = t[0]; totals[1] = t[1]; totals[2] = t[2];
    info[0] = (n_live > 0 && info[2] > 0) ? done : 0;
    info[1] = 0;
    return TSS_OK;
}

}  // namespace tss
