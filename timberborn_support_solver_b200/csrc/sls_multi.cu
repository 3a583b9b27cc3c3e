// Kernel (b), multi-platform variant: stochastic local search over PLACEMENTS (anchor, dims key) for platform sets
// beyond {1x1} (the reference REPL solves with PLATFORMS_DEFAULT: 1x1, 1x2..1x6 + rotations, 3x3, 5x5 —
// src/platform.rs:23-32, crates/repl/src/main.rs:254).  The objective is the one the REPL tightens: the number of
// platforms (anchors), src/encoder/platform_layout.rs:58-60 / crates/repl/src/main.rs:346.
//
// Feasibility is exactly validate()'s (platform_layout.rs:85-149) and the encoder's overlap / out-of-bounds clauses
// (src/encoder.rs:546-609): footprints lie inside the grid and are pairwise disjoint; a tile is supported iff it is
// within three ceiling-masked 4-neighbour steps of a ceiling tile under some footprint.
//
// One chain per warp, lane r = grid row r (grids up to 32x32).  Registers: ceiling C, occupied tiles Occ, cover counts
// as five bit-planes (a tile is covered by at most 25 pairwise-disjoint platforms), uncovered U, covered-once O.
// Scoring is lane-parallel and exact: lane i takes ONE candidate placement, fetches the (h+6) x (w+6) window of C
// around it with warp shuffles, dilates the footprint three times inside that window in registers (geodesic paths of
// length <= 3 from the footprint never leave it) and counts popcount(U & reach) resp. popcount(O & reach).
// A step: drop / swap as in sls_spec.hpp; addition candidates are 2 x 32 random in-bounds placements whose footprint
// comes within 3 tiles of a random uncovered tile and does not overlap the current platforms.  The first pass draws the
// dims key uniformly, the second one from the keys sorted by area (largest first) with a squared uniform draw, i.e.
// biased towards large platforms: with the count objective a well placed large platform replaces several small ones, and
// uniform draws find e.g. the four 5x5 platforms of test/ex2.toml only with thousands of chains.
//
// Objective: every dims key has an integer cost; the search minimises the total cost of the layout.  With all costs 1
// this is the REPL's platform count.  With the GUI's weights (crates/gui/src/app.rs:53-62) the cost of a platform is
// what PlatformLayout::total_weight charges for it — the sum of the weights of every def contained in its def
// (platform_layout.rs:174-183) — and the bound is the GUI's `weight_limit = weight - 1` (app.rs:235-245).  The step rule
// generalises "k == L-1 -> swap" to "no candidate is affordable (W + min cost >= L) -> remove first", candidates must be
// affordable (W + cost < L) and are ranked by gain per cost.
#include "engine.hpp"
#include "sls_multi.hpp"
#include "sls_spec.hpp"

namespace tss {
namespace slsm {

constexpr unsigned FULL = 0xffffffffu;
constexpr int WARPS = 4;
constexpr int WIN = 12;  // window rows / columns: footprint (<= 6) + 3 on each side

struct Lane {
    uint32_t C, Occ, c0, c1, c2, c3, c4, U, O;
    uint32_t N;   // WINDOW: the tiles this window still has to cover (ceiling not covered by the frozen platforms)
};
template <bool WINDOW>
__device__ __forceinline__ void derive(Lane& L) {
    uint32_t hi = L.c1 | L.c2 | L.c3 | L.c4;
    L.U = (WINDOW ? L.N : L.C) & ~(L.c0 | hi);
    L.O = WINDOW ? (L.N & L.c0 & ~hi) : (L.c0 & ~hi);
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

__device__ __forceinline__ uint32_t span(int x, int w) { return (w >= 32 ? 0xffffffffu : ((1u << w) - 1u)) << x; }

// Row-distributed footprint and reach of ONE placement (all lanes cooperate; lane r = grid row r).
__device__ __forceinline__ void placement_rows(uint32_t C, int lane, int x, int y, int w, int h, uint32_t& foot, uint32_t& reach) {
    foot = (lane >= y && lane < y + h) ? span(x, w) : 0u;
    uint32_t X = foot & C;
#pragma unroll
    for (int round = 0; round < kTerrainSupportDistance - 1; round++) {
        uint32_t up = __shfl_up_sync(FULL, X, 1), down = __shfl_down_sync(FULL, X, 1);
        if (lane == 0) up = 0;
        if (lane == 31) down = 0;
        X = (X | (X << 1) | (X >> 1) | up | down) & C;
    }
    reach = X;
}

// popcount(B & reach(placement)) for this lane's own candidate; all 32 lanes must call.
// Also returns (through `overlap`) whether the footprint intersects the occupancy board.
__device__ __forceinline__ int score_placement(uint32_t C, uint32_t B, uint32_t Occ, int x, int y, int w, int h, bool& overlap) {
    const int ax = max(x - 3, 0);           // window column 0
    const uint32_t fmask = span(x - ax, w); // footprint columns inside the window
    uint32_t Cw[WIN], X[WIN];
    uint32_t occ_hit = 0;
#pragma unroll
    for (int j = 0; j < WIN; j++) {
        const int gy = y - 3 + j;
        const bool in = gy >= 0 && gy < 32 && j < h + 6;
        uint32_t crow = __shfl_sync(FULL, C, gy);
        uint32_t orow = __shfl_sync(FULL, Occ, gy);
        Cw[j] = in ? ((crow >> ax) & 0xfffu) : 0u;
        const bool frow = j >= 3 && j < 3 + h;
        X[j] = frow ? (Cw[j] & fmask) : 0u;
        occ_hit |= (frow && in) ? ((orow >> ax) & fmask) : 0u;
    }
    overlap = occ_hit != 0;
#pragma unroll
    for (int round = 0; round < kTerrainSupportDistance - 1; round++) {
        uint32_t N[WIN];
#pragma unroll
        for (int j = 0; j < WIN; j++) {
            uint32_t v = X[j] | (X[j] << 1) | (X[j] >> 1);
            if (j > 0) v |= X[j - 1];
            if (j < WIN - 1) v |= X[j + 1];
            N[j] = v & Cw[j];
        }
#pragma unroll
        for (int j = 0; j < WIN; j++) X[j] = N[j];
    }
    int s = 0;
#pragma unroll
    for (int j = 0; j < WIN; j++) {
        uint32_t brow = __shfl_sync(FULL, B, y - 3 + j);
        s += __popc(((brow >> ax) & 0xfffu) & X[j]);
    }
    return s;
}

struct Ctx {
    uint16_t* items;
    const int2* keys;  // effective (w, h) per key
    int lane, W, H;
};

__device__ __forceinline__ void unpack(const Ctx& c, int code, int& x, int& y, int& w, int& h) {
    x = code & 31; y = (code >> 5) & 31;
    int2 d = c.keys[code >> 10];
    w = d.x; h = d.y;
}

template <bool WINDOW>
__device__ __forceinline__ int remove_min_loss(Lane& L, const Ctx& c, int& k, uint32_t hl, int exclude) {
    uint32_t best_key = 0xffffffffu;
    int best_i = 0;
    for (int b = 0, chunk = 0; b < k; b += 32, chunk++) {
        int i = b + c.lane;
        bool valid = i < k;
        int code = valid ? c.items[i] : 0, x, y, w, h;
        unpack(c, code, x, y, w, h);
        bool ov;
        int loss = score_placement(L.C, L.O, 0u, x, y, w, h, ov);
        uint32_t key = (valid && !(code == exclude && k > 1)) ? (((uint32_t)loss << 16) | sls::tie_remove_hl(hl, (uint32_t)chunk)) : 0xffffffffu;
        uint32_t mn = __reduce_min_sync(FULL, key);
        if (mn < best_key) { best_key = mn; best_i = b + __ffs(__ballot_sync(FULL, key == mn)) - 1; }
    }
    int code = c.items[best_i];
    __syncwarp();
    if (c.lane == 0) c.items[best_i] = c.items[k - 1];
    __syncwarp();
    k--;
    int x, y, w, h;
    unpack(c, code, x, y, w, h);
    uint32_t foot, reach;
    placement_rows(L.C, c.lane, x, y, w, h, foot, reach);
    planes_sub(L, reach);
    derive<WINDOW>(L);
    L.Occ &= ~foot;
    return code;
}

using sls::pick_rotated;

// ONESHOT = the first epoch of a one-shot solve in ONE launch (tss_solve_upper_bound, first-model mode, workspace of the same
// platform set cached): terrain rows and bound arrive as kernel parameters, chains start empty in registers (no init
// kernel), and the last CTA to finish — a ticket counter — folds the best objective, fetches the winner's placements,
// re-validates them (footprints in bounds and pairwise disjoint, validate()'s three dilations: kernel (a) in one-warp
// form) and writes everything into mapped host memory.  One launch, one synchronisation.
struct OneShotM {
    uint32_t rows[32];            // terrain rows
    int bound;                    // chains look for an objective below this (card_limit + 1, or NO_BOUND)
    uint32_t* rows_out;           // [32] kept on the device for follow-up epochs
    int* bounds_out;              // [1]
    int2* best_out;               // [1]
    unsigned long long* key;      // running (best << 32 | chain) minimum, ~0 between launches
    unsigned int* ticket;         // CTAs finished, 0 between launches
    uint32_t* result_host;        // mapped host memory: [0] best objective, [1] winner chain, [2] placements n, [3] unsupported tiles,
                                  // [4] overlapping, [5] out of bounds, [6..11] totals (candidates, steps, flips) as three u64,
                                  // from word 16: the n placement codes as u16
};

// WINDOW = the window-decomposed placement search on grids larger than 32x32 (lns_placements.cu, see WindowM): chain c works
// on window c / seeds, `terrain_rows` holds 32 ceiling rows per window and the epoch bound is bounds[window].
// (WINDOW: at most 4 CTAs per SM, i.e. up to 128 registers — the window's need rows and box do not fit the 96 registers the
// compiler settles for otherwise without spilling; a phase on 256x256 launches ~1300 chains, 2-3 CTAs per SM.  LIMITS: the
// same, for the class counters; an epoch launches 16 chains = 4 CTAs per SM.  WINDOW and LIMITS together fit the same 128)
template <bool ONESHOT, bool WINDOW, bool LIMITS>
__global__ void __launch_bounds__(WARPS * 32, (WINDOW || LIMITS) ? 4 : 0) sls_multi_kernel(const uint32_t* __restrict__ terrain_rows, int W, int H,
                                                              const int2* __restrict__ keys_g, const int* __restrict__ costs_g,
                                                              const int* __restrict__ order_g, int n_keys,
                                                              MultiState* __restrict__ states,
                                                              int n_chains, uint32_t chain_offset, uint64_t seed, long long steps,
                                                              const int* __restrict__ bounds, int target, int noise_pct,
                                                              const volatile int* interrupt, unsigned long long* __restrict__ totals,
                                                              const OneShotM os, const WindowM wm, const LimitsM lm) {
    static_assert(!(ONESHOT && WINDOW), "a one-shot solve never runs on windows");
    static_assert(!LIMITS || !ONESHOT, "per-type limits never run in a one-shot launch");
    __shared__ uint16_t items_all[WARPS][MAX_ITEMS];
    __shared__ int2 keys[MAX_KEYS];
    __shared__ int costs[MAX_KEYS];
    __shared__ int order[MAX_KEYS];   // keys by area, largest first
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int chain = blockIdx.x * WARPS + warp;
    // a layout within the target is already known for this terrain (found in an earlier epoch): nothing to do.  Lets a host
    // queue several epochs back to back without a round trip in between (one-shot solves, sls_spec.hpp).
    // (windows: the warps of a CTA may belong to different windows, so this test waits until after the barrier)
    if (!ONESHOT && !WINDOW && target >= 0 && bounds[0] <= target) return;
    if (threadIdx.x < n_keys) { keys[threadIdx.x] = keys_g[threadIdx.x]; costs[threadIdx.x] = costs_g[threadIdx.x]; order[threadIdx.x] = order_g[threadIdx.x]; }
    __syncthreads();
    int cmin = costs[0];
    for (int i = 1; i < n_keys; i++) cmin = min(cmin, costs[i]);
    if (!ONESHOT && chain >= n_chains) return;   // (a one-shot launch has whole CTAs of chains: everyone takes part in the ticket)
    const int win = WINDOW ? chain / wm.seeds : 0;
    if (WINDOW && target >= 0 && bounds[win] <= target) return;
    MultiState& st = states[chain];
    if (!ONESHOT && st.done) return;
    if (ONESHOT && blockIdx.x == 0 && threadIdx.x < 32) {
        os.rows_out[threadIdx.x] = os.rows[threadIdx.x];
        if (threadIdx.x == 0) os.bounds_out[0] = os.bound;
    }

    const int epoch_bound = ONESHOT ? os.bound : bounds[win];
    const uint32_t base = sls::chain_base(seed, chain_offset + (uint32_t)chain);
    const uint32_t nq7 = sls::noise_q7(noise_pct);
    Ctx c{items_all[warp], keys, lane, W, H};
    Lane L;
    L.C = ONESHOT ? os.rows[lane] : terrain_rows[win * 32 + lane];
    L.Occ = WINDOW ? wm.occ[win * 32 + lane] : 0u;
    if (WINDOW) L.N = wm.need[win * 32 + lane];
    const int4 box = WINDOW ? wm.box[win] : make_int4(0, 0, W, H);
    L.c0 = L.c1 = L.c2 = L.c3 = L.c4 = 0;
    int k = ONESHOT ? 0 : st.k, best = ONESHOT ? sls::NO_BOUND : st.best, tabu_add = ONESHOT ? -1 : st.tabu_add, tabu_rem = ONESHOT ? -1 : st.tabu_rem, done = 0;
    uint32_t step = ONESHOT ? 0u : st.step;
    if (ONESHOT && lane == 0) st.best_k = 0;
    unsigned long long scored = 0;
    uint32_t flips = 0;   // platforms added + removed
    for (int i = lane; i < k; i += 32) c.items[i] = st.items[i];
    __syncwarp();
    int Wt = 0;  // total cost of the current layout
    // LIMITS: lane i < n_keys holds key i's class mask and cost, lane j < n_classes holds n_j and limit[j]
    const uint32_t kmask = LIMITS && lane < n_keys ? (uint32_t)lm.mask[lane] : 0u;
    const int kcost = LIMITS && lane < n_keys ? costs[lane] : 0x7fffffff;
    const int climit = LIMITS && lane < lm.n_classes ? lm.limit[(WINDOW ? win * MAX_KEYS : 0) + lane] : 0x7fffffff;
    int ncls = 0;
    for (int i = 0; i < k; i++) {
        int x, y, w, h;
        unpack(c, c.items[i], x, y, w, h);
        uint32_t foot, reach;
        placement_rows(L.C, lane, x, y, w, h, foot, reach);
        planes_add(L, reach);
        L.Occ |= foot;
        Wt += costs[c.items[i] >> 10];
        if (LIMITS) ncls += (__shfl_sync(FULL, kmask, c.items[i] >> 10) >> lane) & 1u;
    }
    derive<WINDOW>(L);
    uint32_t full = 0;   // LIMITS: classes at their limit
    int cfree = cmin;    // LIMITS: smallest cost of a key in no full class (1x1 is in none: always defined)
    auto count_flip = [&](int code, int sign) {
        if (!LIMITS) return;
        ncls += sign * (int)((__shfl_sync(FULL, kmask, code >> 10) >> lane) & 1u);
        full = __ballot_sync(FULL, ncls >= climit);
        cfree = (int)__reduce_min_sync(FULL, (kmask & full) ? 0x7fffffffu : (uint32_t)kcost);
    };
    if (LIMITS) count_flip(0, 0);

    long long it = 0;
    for (; it < steps; it++, step++) {
        if ((it & 255) == 255 && *interrupt) break;
        const int limit = min(epoch_bound, best);
        const uint32_t hs = sls::step_hash(base, step);
        const uint32_t hl = sls::lane_hash(hs, (uint32_t)lane);
        if (Wt >= limit) {  // too expensive for an improvement: drop a platform
            if (k == 0) { done = 1; break; }
            scored += (unsigned)k;
            tabu_add = remove_min_loss<WINDOW>(L, c, k, hl, -1);
            Wt -= costs[tabu_add >> 10];
            count_flip(tabu_add, -1);
            flips++;
            continue;
        }
        if (!__any_sync(FULL, L.U != 0)) {  // complete layout with total cost < limit
            best = Wt;
            for (int i = lane; i < k; i += 32) st.best_items[i] = c.items[i];
            if (lane == 0) st.best_k = k;
            if (Wt <= target || k == 0) { done = 1; it++; step++; break; }
            continue;
        }
        if (Wt + (LIMITS ? cfree : cmin) >= limit && k > 0) {  // nothing is affordable: swap = remove + add
            scored += (unsigned)k;
            tabu_add = remove_min_loss<WINDOW>(L, c, k, hl, tabu_rem);
            Wt -= costs[tabu_add >> 10];
            count_flip(tabu_add, -1);
            flips++;
        }
        // a random uncovered tile, then two passes of 32 random placements near it
        const uint32_t rowmask = __ballot_sync(FULL, L.U != 0);
        const int ty = pick_rotated(rowmask, hs & 31u);
        const uint32_t Urow = __shfl_sync(FULL, L.U, ty);
        const int tx = pick_rotated(Urow, (hs >> 5) & 31u);
        const bool noise = ((hs >> 10) & 127u) < nq7;
        uint32_t best_key = 0;
        int best_code = -1;
#pragma unroll 1
        for (int pass = 0; pass < 2; pass++) {
            const uint32_t r = sls::lane_hash(hl, (uint32_t)(pass + 40));
            const uint32_t u = r & 0xffffu;
            const int key = pass == 0 ? (int)((u * (uint32_t)n_keys) >> 16) : order[(((u * u) >> 16) * (uint32_t)n_keys) >> 16];
            const int2 d = keys[key];
            // footprint intersects the 7x7 box around t: x in [tx-3-(w-1), tx+3], y in [ty-3-(h-1), ty+3]
            const int x = tx - 3 - (d.x - 1) + (int)((((r >> 16) & 0xffu) * (uint32_t)(d.x + 6)) >> 8);
            const int y = ty - 3 - (d.y - 1) + (int)(((r >> 24) * (uint32_t)(d.y + 6)) >> 8);
            const bool inb = WINDOW ? (x >= box.x && y >= box.y && x + d.x <= box.z && y + d.y <= box.w)   // inside the window's box
                                    : (x >= 0 && y >= 0 && x + d.x <= W && y + d.y <= H);   // out-of-bounds placements are never valid
            const int code = inb ? ((key << 10) | (y << 5) | x) : 0;
            bool ov;
            int g = score_placement(L.C, L.U, L.Occ, inb ? x : 0, inb ? y : 0, d.x, d.y, ov);
            const int cost = costs[key];
            const bool blocked = LIMITS && (__shfl_sync(FULL, kmask, key) & full) != 0u;
            const bool ok = inb && !ov && g > 0 && code != tabu_add && Wt + cost < limit && !blocked;
            const uint32_t rank = ((uint32_t)g * 64u) / (uint32_t)cost;  // gain per cost (< 2^14)
            uint32_t kk = ok ? ((noise ? 0x10000u : (rank << 16)) | (r >> 16 ^ (r & 0xffffu))) : 0u;
            kk = ok ? (kk | 1u) : 0u;
            uint32_t mx = __reduce_max_sync(FULL, kk);
            scored += (unsigned)__popc(__ballot_sync(FULL, inb));
            if (mx > best_key) {
                best_key = mx;
                best_code = __shfl_sync(FULL, code, __ffs(__ballot_sync(FULL, kk == mx)) - 1);
            }
        }
        if (best_code < 0) continue;  // nothing feasible this step; try again with other placements
        int x, y, w, h;
        unpack(c, best_code, x, y, w, h);
        uint32_t foot, reach;
        placement_rows(L.C, lane, x, y, w, h, foot, reach);
        planes_add(L, reach);
        derive<WINDOW>(L);
        L.Occ |= foot;
        if (lane == 0) c.items[k] = (uint16_t)best_code;
        __syncwarp();
        k++;
        Wt += costs[best_code >> 10];
        count_flip(best_code, +1);
        tabu_rem = best_code;
        flips++;
    }

    for (int i = lane; i < k; i += 32) st.items[i] = c.items[i];
    if (lane == 0) {
        st.k = k; st.best = best; st.step = step; st.tabu_add = tabu_add; st.tabu_rem = tabu_rem; st.done = done;
        atomicAdd(&totals[0], scored);
        atomicAdd(&totals[1], (unsigned long long)it);
        atomicAdd(&totals[2], (unsigned long long)flips);
        if (ONESHOT && best < sls::NO_BOUND) atomicMin(os.key, ((unsigned long long)(uint32_t)best << 32) | (uint32_t)chain);
    }
    if (ONESHOT) {
        __shared__ bool last;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) last = atomicAdd(os.ticket, 1u) == gridDim.x - 1;
        __syncthreads();
        if (last && warp == 0) {
            __threadfence();
            const unsigned long long key = *(volatile unsigned long long*)os.key;
            const int bobj = key == ~0ull ? sls::NO_BOUND : (int)(key >> 32), bchain = key == ~0ull ? -1 : (int)(key & 0xffffffffu);
            const MultiState* win = bchain >= 0 ? states + bchain : nullptr;
            const int n = win ? __ldcg(&win->best_k) : 0;
            uint16_t* codes_host = reinterpret_cast<uint16_t*>(os.result_host + 16);
            // validate()'s view of the winner (platform_layout.rs:85-149): footprints stamped row by row (lane = row), overlap and
            // bounds flags, then three ceiling-masked dilations from the ceiling under the footprints
            uint32_t occ = 0, overlap = 0, oob = 0;
            for (int i = 0; i < n; i++) {
                const int code = __ldcg(&win->best_items[i]);
                const int2 d = keys[code >> 10];
                const int x = code & 31, y = (code >> 5) & 31;
                if (x + d.x > W || y + d.y > H) oob = 1;
                const uint32_t sp = (lane >= y && lane < y + d.y) ? span(x, d.x) : 0u;
                overlap |= occ & sp;
                occ |= sp;
                if (lane == (i & 31)) codes_host[i] = (uint16_t)code;
            }
            uint32_t X = occ & L.C;
            for (int round = 0; round < 3; round++) {
                uint32_t up = __shfl_up_sync(FULL, X, 1), down = __shfl_down_sync(FULL, X, 1);
                if (lane == 0) up = 0;
                if (lane == 31) down = 0;
                X = (X | (X << 1) | (X >> 1) | up | down) & L.C;
            }
            const int unc = __reduce_add_sync(FULL, __popc(L.C & ~X));
            const bool any_overlap = __any_sync(FULL, overlap != 0);
            if (lane == 0) {
                os.best_out[0] = make_int2(bobj, bchain);
                if (bobj < os.bound) os.bounds_out[0] = bobj;
                const unsigned long long t0 = *(volatile unsigned long long*)&totals[0], t1 = *(volatile unsigned long long*)&totals[1];
                os.result_host[0] = (uint32_t)bobj; os.result_host[1] = (uint32_t)bchain; os.result_host[2] = (uint32_t)n;
                os.result_host[3] = (uint32_t)unc; os.result_host[4] = any_overlap ? 1u : 0u; os.result_host[5] = oob;
                os.result_host[6] = (uint32_t)t0; os.result_host[7] = (uint32_t)(t0 >> 32);
                os.result_host[8] = (uint32_t)t1; os.result_host[9] = (uint32_t)(t1 >> 32);
                const unsigned long long t2 = *(volatile unsigned long long*)&totals[2];
                os.result_host[10] = (uint32_t)t2; os.result_host[11] = (uint32_t)(t2 >> 32);
                *os.key = ~0ull;
                *os.ticket = 0u;
                __threadfence_system();
            }
        }
    }
}

__global__ void multi_init_kernel(MultiState* states, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    states[i].k = 0; states[i].best_k = 0; states[i].best = sls::NO_BOUND; states[i].step = 0; states[i].tabu_add = -1; states[i].tabu_rem = -1; states[i].done = 0;
}

// smallest best over all chains (ties: lowest chain); also folds it into bounds[0]
__global__ void multi_best_kernel(const MultiState* __restrict__ states, int n_chains, int2* __restrict__ out, int* __restrict__ bounds) {
    __shared__ unsigned long long sm[256];
    unsigned long long key = ~0ull;
    for (int c = threadIdx.x; c < n_chains; c += blockDim.x) {
        unsigned long long kk = ((unsigned long long)(uint32_t)states[c].best << 32) | (uint32_t)c;
        key = kk < key ? kk : key;
    }
    sm[threadIdx.x] = key;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
        if (threadIdx.x < o && sm[threadIdx.x + o] < sm[threadIdx.x]) sm[threadIdx.x] = sm[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        int2 r = sm[0] == ~0ull ? make_int2(sls::NO_BOUND, -1) : make_int2((int)(sm[0] >> 32), (int)(sm[0] & 0xffffffffu));
        out[0] = r;
        if (r.x < bounds[0]) bounds[0] = r.x;
    }
}

// One-shot solves: the best chain's placements as codes + count and as the (x, y, w, h) records / offsets the platform
// evaluator (kernel (a)) reads, all on the device so fetching and re-validating the witness stay in the epoch's stream.
__global__ void multi_witness_kernel(const MultiState* __restrict__ states, const int2* __restrict__ best, const int2* __restrict__ keys,
                                     uint16_t* __restrict__ codes, int4* __restrict__ plats, uint32_t* __restrict__ offsets) {
    const int c = best[0].y;
    const int n = c >= 0 ? states[c].best_k : 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int code = states[c].best_items[i];
        const int2 d = keys[code >> 10];
        codes[i] = (uint16_t)code;
        plats[i] = make_int4(code & 31, (code >> 5) & 31, d.x, d.y);
    }
    if (threadIdx.x == 0) { offsets[0] = 0; offsets[1] = (uint32_t)n; }
}

}  // namespace slsm

size_t slsm_state_bytes() { return sizeof(slsm::MultiState); }
int slsm_max_keys() { return slsm::MAX_KEYS; }

int slsm_init(tss_engine* e, void* states, int n) {
    slsm::multi_init_kernel<<<(n + 127) / 128, 128, 0, e->stream>>>((slsm::MultiState*)states, n);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}
// limits_dev: class masks per key [MAX_KEYS] then limits per class [MAX_KEYS] (see slsm::LimitsM); n_classes == 0: no limits
int slsm_run(tss_engine* e, const uint32_t* rows_dev, int W, int H, const int2* keys_dev, const int* costs_dev, const int* order_dev, int n_keys, void* states, int n_chains,
             uint32_t chain_offset, uint64_t seed, long long steps, int* bounds_dev, int target, int noise_pct, unsigned long long* totals_dev,
             int2* best_dev, const int* limits_dev, int n_classes) {
    int blocks = (n_chains + slsm::WARPS - 1) / slsm::WARPS;
    if (n_classes > 0)
        slsm::sls_multi_kernel<false, false, true><<<blocks, slsm::WARPS * 32, 0, e->stream>>>(rows_dev, W, H, keys_dev, costs_dev, order_dev, n_keys, (slsm::MultiState*)states,
                                                                                             n_chains, chain_offset, seed, steps, bounds_dev, target, noise_pct,
                                                                                             e->interrupt_dev, totals_dev, slsm::OneShotM{}, slsm::WindowM{},
                                                                                             slsm::LimitsM{limits_dev, limits_dev + slsm::MAX_KEYS, n_classes});
    else
        slsm::sls_multi_kernel<false, false, false><<<blocks, slsm::WARPS * 32, 0, e->stream>>>(rows_dev, W, H, keys_dev, costs_dev, order_dev, n_keys, (slsm::MultiState*)states,
                                                                                              n_chains, chain_offset, seed, steps, bounds_dev, target, noise_pct,
                                                                                              e->interrupt_dev, totals_dev, slsm::OneShotM{}, slsm::WindowM{}, slsm::LimitsM{});
    TSS_CHECK_LAUNCH(e);
    slsm::multi_best_kernel<<<1, 256, 0, e->stream>>>((const slsm::MultiState*)states, n_chains, best_dev, bounds_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches += 2;
    return TSS_OK;
}
// The fused first epoch of a one-shot solve (see slsm::OneShotM).  n_chains must be a multiple of 4 (whole CTAs);
// result_host_mapped: mapped pinned memory of 16 + 512 words; key_dev holds ~0 and ticket_dev 0 (both re-arm themselves).
int slsm_run_oneshot(tss_engine* e, const uint32_t* rows32_host, int bound, uint32_t* rows_dev, int W, int H, const int2* keys_dev, const int* costs_dev,
                     const int* order_dev, int n_keys, void* states, int n_chains, uint64_t seed, long long steps, int* bounds_dev, int2* best_dev,
                     unsigned long long* key_dev, unsigned int* ticket_dev, int target, int noise_pct, unsigned long long* totals_dev,
                     uint32_t* result_host_mapped) {
    if (n_chains <= 0 || n_chains % slsm::WARPS != 0) return e->fail(TSS_E_INVALID, "one-shot launch needs whole CTAs of chains");
    slsm::OneShotM os;
    for (int r = 0; r < 32; r++) os.rows[r] = rows32_host[r];
    os.bound = bound; os.rows_out = rows_dev; os.bounds_out = bounds_dev; os.best_out = best_dev; os.key = key_dev; os.ticket = ticket_dev;
    os.result_host = result_host_mapped;
    slsm::sls_multi_kernel<true, false, false><<<n_chains / slsm::WARPS, slsm::WARPS * 32, 0, e->stream>>>(nullptr, W, H, keys_dev, costs_dev, order_dev, n_keys,
                                                                                                          (slsm::MultiState*)states, n_chains, 0u, seed, steps, nullptr,
                                                                                                          target, noise_pct, e->interrupt_dev, totals_dev, os,
                                                                                                          slsm::WindowM{}, slsm::LimitsM{});
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}
// One epoch of every window's chains (the window-decomposed placement search, lns_placements.cu); chains are numbered
// window * wm.seeds + j.  No best-reduce here: the caller picks a winner per window.  lm.n_classes > 0: per-window class budgets
// (slsm::LimitsM).
int slsm_run_windows(tss_engine* e, const uint32_t* rows_dev, const slsm::WindowM& wm, const int2* keys_dev, const int* costs_dev, const int* order_dev,
                     int n_keys, slsm::MultiState* states, int n_chains, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev,
                     int target, int noise_pct, unsigned long long* totals_dev, const slsm::LimitsM& lm) {
    const int blocks = (n_chains + slsm::WARPS - 1) / slsm::WARPS;
    if (lm.n_classes > 0)
        slsm::sls_multi_kernel<false, true, true><<<blocks, slsm::WARPS * 32, 0, e->stream>>>(rows_dev, 32, 32, keys_dev, costs_dev, order_dev, n_keys, states, n_chains,
                                                                                            chain_offset, seed, steps, bounds_dev, target, noise_pct, e->interrupt_dev,
                                                                                            totals_dev, slsm::OneShotM{}, wm, lm);
    else
        slsm::sls_multi_kernel<false, true, false><<<blocks, slsm::WARPS * 32, 0, e->stream>>>(rows_dev, 32, 32, keys_dev, costs_dev, order_dev, n_keys, states, n_chains,
                                                                                             chain_offset, seed, steps, bounds_dev, target, noise_pct, e->interrupt_dev,
                                                                                             totals_dev, slsm::OneShotM{}, wm, slsm::LimitsM{});
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}

int slsm_witness(tss_engine* e, const void* states, const int2* best_dev, const int2* keys_dev, uint16_t* codes_dev, int4* plats_dev, uint32_t* offsets_dev) {
    slsm::multi_witness_kernel<<<1, 128, 0, e->stream>>>((const slsm::MultiState*)states, best_dev, keys_dev, codes_dev, plats_dev, offsets_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}
int slsm_max_items() { return slsm::MAX_ITEMS; }
// best items of one chain -> host codes (key << 10 | y << 5 | x)
int slsm_read_best(tss_engine* e, const void* states, int chain, std::vector<uint16_t>& codes) {
    const slsm::MultiState* st = (const slsm::MultiState*)states + chain;
    int count = 0;
    TSS_CUDA(e, cudaMemcpy(&count, &st->best_k, sizeof(int), cudaMemcpyDeviceToHost));
    if (count < 0 || count > slsm::MAX_ITEMS) return e->fail(TSS_E_CUDA, "corrupt chain state (best_k = %d)", count);
    codes.resize((size_t)count);
    if (count > 0) TSS_CUDA(e, cudaMemcpy(codes.data(), st->best_items, sizeof(uint16_t) * (size_t)count, cudaMemcpyDeviceToHost));
    return TSS_OK;
}

// every chain's state -> host arrays (parity tests replay the search on the CPU model); any pointer may be null
int slsm_read_states(tss_engine* e, const void* states, int n_chains, uint16_t* items, int32_t* k, uint16_t* best_items, int32_t* best_k,
                     int32_t* best, uint32_t* step) {
    std::vector<slsm::MultiState> st((size_t)n_chains);
    TSS_CUDA(e, cudaMemcpy(st.data(), states, sizeof(slsm::MultiState) * st.size(), cudaMemcpyDeviceToHost));
    for (size_t c = 0; c < st.size(); c++) {
        const int kc = st[c].k, bk = st[c].best_k;
        if (kc < 0 || kc > slsm::MAX_ITEMS || bk < 0 || bk > slsm::MAX_ITEMS) return e->fail(TSS_E_CUDA, "corrupt chain state (k = %d, best_k = %d)", kc, bk);
        if (items) for (int i = 0; i < slsm::MAX_ITEMS; i++) items[c * slsm::MAX_ITEMS + i] = i < kc ? st[c].items[i] : 0;
        if (best_items) for (int i = 0; i < slsm::MAX_ITEMS; i++) best_items[c * slsm::MAX_ITEMS + i] = i < bk ? st[c].best_items[i] : 0;
        if (k) k[c] = kc;
        if (best_k) best_k[c] = bk;
        if (best) best[c] = st[c].best;
        if (step) step[c] = st[c].step;
    }
    return TSS_OK;
}

}  // namespace tss
