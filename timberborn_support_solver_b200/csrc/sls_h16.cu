// Kernel (b), half-warp variant for grids of at most 16 rows (rect 16x16, test/ex1-3): TWO chains per warp.
//
// ncu on the one-chain-per-warp kernel (profiles/r1_sls_kernel.md) shows the ALU pipe as the limiter and most of a
// step's ~340 warp instructions are per-chain "uniform" control work (hashes, picks, ballots, key building) that all
// 32 lanes repeat.  With <= 16 grid rows only 16 lanes hold data, so each half-warp runs its own chain here: the same
// instruction stream now advances two layouts.  The step rule, RNG and tie-breaks are EXACTLY those of sls_spec.hpp /
// sls.cu (the parity tests replay both kernels against the same CPU model); only the lane mapping differs:
//   lane = 16*half + row; removal candidates are scored 16 per pass, the 25 diamond cells in two passes of 16;
//   the step is fully predicated (drop / record / swap flags per half) so both halves stay convergent for the shuffles.
#include "engine.hpp"
#include "sls_spec.hpp"
#include "sls_warp.cuh"

namespace tss {
namespace sls16 {

using namespace tss::sls;

constexpr int WARPS = 4;          // 8 chains per CTA
constexpr int MAX_SITES16 = 512;  // tiles of a 32x16 grid

__device__ __forceinline__ uint32_t half_min(uint32_t v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(FULL, v, o, 16));
    return v;
}
__device__ __forceinline__ uint32_t half_max(uint32_t v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(FULL, v, o, 16));
    return v;
}

// ONESHOT = the whole first epoch of a one-shot solve in ONE launch (tss_solve_upper_bound, latency mode): the terrain
// rows arrive as kernel parameters (no upload), every CTA derives the reach table in its own shared memory (CTA 0 also
// stores it for follow-up epochs), chains start empty in registers (no init kernel), and the last CTA to finish — a
// ticket counter, no cooperative launch — folds the best count, fetches the winner's layout, re-validates it
// (kernel (a) in one-warp form) and writes the results straight into mapped host memory.  The host enqueues one kernel
// and synchronises once; the instances are small, so launch and round-trip overhead is what there is to save.
struct OneShot {
    uint32_t rows[32];            // terrain rows (row r, bit x = ceiling at (x, r))
    int bound;                    // chains look for fewer than this many supports (card_limit + 1, or NO_BOUND)
    uint32_t* rows_out;           // [32]   kept on the device for follow-up epochs
    uint2* tabs_out;              // [1024]
    int* bounds_out;              // [1]
    int2* best_out;               // [1]
    unsigned long long* key;      // running (best << 32 | chain) minimum, ~0 between launches
    unsigned int* ticket;         // CTAs finished, 0 between launches
    uint32_t* result_host;        // mapped host memory: [0..31] rows of the best layout, [32] unsupported tiles, [33] supports,
                                  // [34] best count, [35] winner chain, [36..41] totals (candidates, steps, flips) as three u64
};

template <bool ONESHOT>
__global__ void __launch_bounds__(WARPS * 32, 8) sls_h16_kernel(const uint32_t* __restrict__ terrain_rows, const uint2* __restrict__ rtabs,
                                                            ChainState* __restrict__ states, int n_chains, int chains_per_terrain,
                                                            uint32_t chain_offset, uint64_t seed, long long steps,
                                                            const int* __restrict__ bounds, int target, int noise_pct,
                                                            const volatile int* interrupt, unsigned long long* __restrict__ totals,
                                                            const OneShot os) {
    __shared__ uint2 tab[1024];
    __shared__ uint16_t sites_all[WARPS * 2][MAX_SITES16];
    __shared__ uint16_t stamps_all[WARPS * 2][MAX_SITES16];   // flip step of every site (site ids < 512 for <= 16 rows)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, half = lane >> 4, row = lane & 15;
    const int chain = (blockIdx.x * WARPS + warp) * 2 + half;
    const int terrain = chains_per_terrain > 0 ? (blockIdx.x * WARPS * 2) / chains_per_terrain : 0;
    // a layout within the target is already known for this terrain (found in an earlier epoch): nothing to do.  Lets a host
    // queue several epochs back to back without a round trip in between (one-shot solves, sls_spec.hpp).
    __shared__ uint32_t crows[32];
    if (ONESHOT) {
        if (threadIdx.x < 32) {
            crows[threadIdx.x] = os.rows[threadIdx.x];
            if (blockIdx.x == 0) os.rows_out[threadIdx.x] = os.rows[threadIdx.x];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) {
            const uint2 win = i < 512 ? reach_window(crows, i) : make_uint2(0u, 0u);   // (at most 16 rows: sites 512.. have no ceiling)
            tab[i] = win;
            if (blockIdx.x == 0) os.tabs_out[i] = win;
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) os.bounds_out[0] = os.bound;
    } else {
        if (target >= 0 && bounds[chains_per_terrain > 0 ? terrain : 0] <= target) return;
        for (int i = threadIdx.x; i < 1024; i += blockDim.x) tab[i] = rtabs[(size_t)terrain * 1024 + i];
    }
    __syncthreads();
    const bool exists = chain < n_chains;
    ChainState& st = states[exists ? chain : 0];
    if (!ONESHOT && !__any_sync(FULL, exists && !st.done)) return;   // (a one-shot launch has every warp take part in the final ticket)

    const int epoch_bound = ONESHOT ? os.bound : bounds[chains_per_terrain > 0 ? terrain : 0];
    const uint32_t base = chain_base(seed, chain_offset + (uint32_t)chain);
    const uint32_t nq7 = noise_q7(noise_pct);
    const unsigned hshift = half * 16;
    uint16_t* sites = sites_all[warp * 2 + half];
    Lane L;
    L.C = ONESHOT ? crows[row] : terrain_rows[(size_t)terrain * 32 + row];
    L.S = (exists && !ONESHOT) ? st.S[row] : 0u;
    uint32_t bestS = (exists && !ONESHOT) ? st.bestS[row] : 0u;
    int k = (exists && !ONESHOT) ? st.k : 0, best = exists ? (ONESHOT ? NO_BOUND : st.best) : 0;
    const int tenure = tenure_of(chain_offset + (uint32_t)chain);
    uint16_t* stamps = stamps_all[warp * 2 + half];
    int done = exists ? (ONESHOT ? 0 : st.done) : 1;
    const int done_at_start = done;
    uint32_t step = (exists && !ONESHOT) ? st.step : 0u;
    unsigned long long scored = 0;
    long long my_steps = 0;
    uint32_t flips = 0;   // supports added + removed

    {   // site list (row-major) and cover planes from S, per half
        for (int i = row; i < MAX_SITES16; i += 16) stamps[i] = stamp_reset(step);
        int c = __popc(L.S), off = c;
        for (int o = 1; o < 16; o <<= 1) { int t = __shfl_up_sync(FULL, off, o, 16); if (row >= o) off += t; }
        off -= c;
        for (uint32_t bits = L.S; bits; bits &= bits - 1) sites[off++] = (uint16_t)(row * 32 + __ffs(bits) - 1);
        __syncwarp();
        L.c0 = L.c1 = L.c2 = L.c3 = L.c4 = 0;
        const int kmax = max(k, __shfl_xor_sync(FULL, k, 16));
        for (int i = 0; i < kmax; i++) {
            int v = i < k ? sites[i] : 0;
            planes_add(L, i < k ? row_mask(tab[v], v & 31, v >> 5, row) : 0u);
        }
        derive(L);
    }

    // the 25 diamond cells in two passes of 16 lanes: cell = 16*pass + row
    int dx0, dy0, dx1, dy1;
    diamond_cell(row, dx0, dy0);
    diamond_cell(min(16 + row, 24), dx1, dy1);
    const bool cell1 = 16 + row < 25;

    for (long long it = 0; it < steps; it++) {
        if ((it & 1023) == 1023 && *interrupt) break;
        if (!__any_sync(FULL, !done)) break;
        const bool active = !done;
        const int limit = min(epoch_bound, best);
        const uint32_t hs = step_hash(base, step);
        const int ten = effective_tenure(tenure, k);  // fixed for the whole step
        bool inc = active;  // this chain consumes a step
        // ---- classify the step (uniform per half)
        const bool drop = active && k >= limit;
        if (drop && k == 0) { done = 1; inc = false; }
        const uint32_t ub = (__ballot_sync(FULL, L.U != 0) >> hshift) & 0xffffu;
        const bool complete = active && !drop && ub == 0;
        if (complete) {
            best = k;
            bestS = L.S;
            if (k <= target || k == 0) done = 1;
        }
        const bool swap_rem = active && !drop && !complete && k == limit - 1 && k > 0;
        const bool do_remove = (drop && k > 0) || swap_rem;
        const bool do_add = active && !drop && !complete;
        // ---- removal: min-loss support, random ties (supports younger than the tenure only as a last resort, except when dropping)
        if (__any_sync(FULL, do_remove)) {
            const int kk = do_remove ? k : 0, kmax = max(kk, __shfl_xor_sync(FULL, kk, 16));
            uint32_t best_key = 0xffffffffu;
            int best_i = 0;
            for (int b = 0; b < kmax; b += 16) {
                const int i = b + row;
                const bool valid = i < kk;
                const int v = valid ? sites[i] : 0;
                const int loss = score<16>(L.O, v & 31, v >> 5, tab[v]);
                const uint32_t tie = tie_remove(hs, (uint32_t)i);
                const uint32_t young = (!drop && is_tabu(step, stamps[v], ten)) ? TABU_BIT : 0u;
                const uint32_t key = valid ? (young | ((uint32_t)loss << 16) | tie) : 0xffffffffu;
                const uint32_t mn = half_min(key);
                const uint32_t eq = (__ballot_sync(FULL, key == mn) >> hshift) & 0xffffu;
                if (mn < best_key) { best_key = mn; best_i = b + __ffs(eq) - 1; }
            }
            const int u = do_remove ? sites[best_i] : 0;
            __syncwarp();
            if (do_remove && row == 0) { sites[best_i] = sites[k - 1]; stamps[u] = (uint16_t)step; }
            __syncwarp();
            planes_sub(L, do_remove ? row_mask(tab[u], u & 31, u >> 5, row) : 0u);
            derive(L);
            if (do_remove) {
                if (row == (u >> 5)) L.S &= ~(1u << (u & 31));
                scored += (unsigned)k;
                k--;
                flips++;
            }
        }
        // ---- addition at a random uncovered tile
        if (__any_sync(FULL, do_add)) {
            const uint32_t rowmask = (__ballot_sync(FULL, L.U != 0) >> hshift) & 0xffffu;
            const bool adding = do_add && rowmask != 0;   // (rowmask is never empty for an adding chain)
            const int y = adding ? pick_rotated(rowmask, hs & 31u) : 0;
            const uint32_t Urow = __shfl_sync(FULL, L.U, y, 16);
            const int x = adding ? pick_rotated(Urow, (hs >> 5) & 31u) : 0;
            const uint2 wt = tab[y * 32 + x];
            const int xoff = min(x, 3);
            // pass 0: cells 0..15, pass 1: cells 16..24
            const int col0 = dx0 + xoff, col1 = dx1 + xoff;
            const int r0 = dy0 + 3, r1 = dy1 + 3;
            const bool v0 = adding && col0 >= 0 && ((((r0 >= 4) ? wt.y : wt.x) >> (7 * (r0 & 3) + col0)) & 1u);
            const bool v1 = adding && cell1 && col1 >= 0 && ((((r1 >= 4) ? wt.y : wt.x) >> (7 * (r1 & 3) + col1)) & 1u);
            const int cv0 = v0 ? (y + dy0) * 32 + x + dx0 : 0, cv1 = v1 ? (y + dy1) * 32 + x + dx1 : 0;
            const uint32_t vb0 = (__ballot_sync(FULL, v0) >> hshift) & 0xffffu, vb1 = (__ballot_sync(FULL, v1) >> hshift) & 0xffffu;
            const int nc = __popc(vb0) + __popc(vb1);
            const bool noise = ((hs >> 10) & 127u) < nq7;
            const uint32_t t0 = tie_add(hs, (uint32_t)row), t1 = tie_add(hs, (uint32_t)(16 + row));
            uint32_t key0, key1;
            if (__any_sync(FULL, adding && !noise)) {
                const int g0 = score<16>(L.U, cv0 & 31, cv0 >> 5, tab[cv0]);
                const int g1 = score<16>(L.U, cv1 & 31, cv1 >> 5, tab[cv1]);
                const uint32_t f0 = is_tabu(step, stamps[cv0], ten) ? 0u : TABU_BIT, f1 = is_tabu(step, stamps[cv1], ten) ? 0u : TABU_BIT;
                key0 = noise ? (0x10000u | t0) : (f0 | ((uint32_t)(g0 + 1) << 16) | t0);
                key1 = noise ? (0x10000u | t1) : (f1 | ((uint32_t)(g1 + 1) << 16) | t1);
            } else {
                key0 = 0x10000u | t0;
                key1 = 0x10000u | t1;
            }
            key0 = v0 ? key0 : 0u;
            key1 = v1 ? key1 : 0u;
            const uint32_t mx = half_max(max(key0, key1));
            // lowest diamond cell among the maxima (cells 0..15 before 16..24)
            const uint32_t e0 = (__ballot_sync(FULL, key0 == mx) >> hshift) & 0xffffu, e1 = (__ballot_sync(FULL, key1 == mx) >> hshift) & 0xffffu;
            const int src = (e0 ? __ffs(e0) : __ffs(e1)) - 1;
            const int pick0 = __shfl_sync(FULL, cv0, src, 16), pick1 = __shfl_sync(FULL, cv1, src, 16);
            const int v = e0 ? pick0 : pick1;
            planes_add(L, adding ? row_mask(tab[v], v & 31, v >> 5, row) : 0u);
            derive(L);
            if (adding) {
                if (row == (v >> 5)) L.S |= 1u << (v & 31);
                if (row == 0) { sites[k] = (uint16_t)v; stamps[v] = (uint16_t)step; }
                if (!noise) scored += (unsigned)nc;
                k++;
                flips++;
            }
            __syncwarp();
        }
        if (inc) { step++; my_steps++; }
    }

    if (exists && !done_at_start) {
        st.S[row] = L.S;
        st.bestS[row] = bestS;
        if (ONESHOT) { st.S[16 + row] = 0u; st.bestS[16 + row] = 0u; }   // (a fresh record: no init kernel ran)
        if (row == 0) {
            st.k = k; st.best = best; st.step = step; st.done = done;
            unsigned long long tot = ONESHOT ? scored : ((unsigned long long)st.scored_hi << 32 | st.scored_lo) + scored;
            st.scored_lo = (uint32_t)tot; st.scored_hi = (uint32_t)(tot >> 32);
            st.steps_done = (ONESHOT ? 0u : st.steps_done) + (uint32_t)my_steps;
            atomicAdd(&totals[0], scored);
            atomicAdd(&totals[1], (unsigned long long)my_steps);
            atomicAdd(&totals[2], (unsigned long long)flips);
            if (ONESHOT && best < NO_BOUND) atomicMin(os.key, ((unsigned long long)(uint32_t)best << 32) | (uint32_t)chain);
        }
    }
    if (ONESHOT) {
        // the last CTA to arrive publishes the result: every CTA's writes above are fenced before its ticket
        __shared__ bool last;
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) last = atomicAdd(os.ticket, 1u) == gridDim.x - 1;
        __syncthreads();
        if (last && warp == 0) {
            __threadfence();
            const unsigned long long key = *(volatile unsigned long long*)os.key;
            const int bcount = key == ~0ull ? NO_BOUND : (int)(key >> 32), bchain = key == ~0ull ? -1 : (int)(key & 0xffffffffu);
            // the winner's layout (written by another CTA: read around L1) and validate()'s three ceiling-masked dilations on it
            const uint32_t S = bchain >= 0 ? __ldcg(&states[bchain].bestS[lane]) : 0u, C = crows[lane];
            uint32_t X = S & C;
            for (int round = 0; round < 3; round++) {
                uint32_t up = __shfl_up_sync(FULL, X, 1), down = __shfl_down_sync(FULL, X, 1);
                if (lane == 0) up = 0;
                if (lane == 31) down = 0;
                X = (X | (X << 1) | (X >> 1) | up | down) & C;
            }
            const int unc = __reduce_add_sync(FULL, __popc(C & ~X)), cnt = __reduce_add_sync(FULL, __popc(S));
            os.result_host[lane] = S;
            if (lane == 0) {
                os.best_out[0] = make_int2(bcount, bchain);
                if (bcount < os.bound) os.bounds_out[0] = bcount;
                const unsigned long long t0 = *(volatile unsigned long long*)&totals[0], t1 = *(volatile unsigned long long*)&totals[1];
                const unsigned long long t2 = *(volatile unsigned long long*)&totals[2];
                os.result_host[40] = (uint32_t)t2; os.result_host[41] = (uint32_t)(t2 >> 32);
                os.result_host[32] = (uint32_t)unc; os.result_host[33] = (uint32_t)cnt;
                os.result_host[34] = (uint32_t)bcount; os.result_host[35] = (uint32_t)bchain;
                os.result_host[36] = (uint32_t)t0; os.result_host[37] = (uint32_t)(t0 >> 32);
                os.result_host[38] = (uint32_t)t1; os.result_host[39] = (uint32_t)(t1 >> 32);
                *os.key = ~0ull;       // re-armed for the next launch
                *os.ticket = 0u;
                __threadfence_system();
            }
        }
    }
}

}  // namespace sls16

int sls_run_h16(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, int n_chains,
                int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
                int noise_pct, unsigned long long* totals_dev) {
    const int per_cta = sls16::WARPS * 2;
    int blocks = (n_chains + per_cta - 1) / per_cta;
    sls16::sls_h16_kernel<false><<<blocks, sls16::WARPS * 32, 0, e->stream>>>(rows_dev, tabs_dev, states, n_chains, chains_per_terrain, chain_offset, seed,
                                                                            steps, bounds_dev, target, noise_pct, e->interrupt_dev, totals_dev,
                                                                            sls16::OneShot{});
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}

// The fused first epoch of a one-shot solve (see sls16::OneShot).  n_chains must be a multiple of 8 (whole CTAs);
// result_host is mapped pinned memory of at least 40 words; key_dev must hold ~0 and ticket_dev 0 (both re-arm themselves).
int sls_run_h16_oneshot(tss_engine* e, const uint32_t* rows32_host, int bound, uint32_t* rows_dev, uint2* tabs_dev, sls::ChainState* states,
                        int n_chains, uint64_t seed, long long steps, int* bounds_dev, int2* best_dev, unsigned long long* key_dev,
                        unsigned int* ticket_dev, int target, int noise_pct, unsigned long long* totals_dev, uint32_t* result_host_mapped) {
    if (n_chains <= 0 || n_chains % (sls16::WARPS * 2) != 0) return e->fail(TSS_E_INVALID, "one-shot launch needs whole CTAs of chains");
    sls16::OneShot os;
    for (int r = 0; r < 32; r++) os.rows[r] = rows32_host[r];
    os.bound = bound; os.rows_out = rows_dev; os.tabs_out = tabs_dev; os.bounds_out = bounds_dev; os.best_out = best_dev;
    os.key = key_dev; os.ticket = ticket_dev; os.result_host = result_host_mapped;
    sls16::sls_h16_kernel<true><<<n_chains / (sls16::WARPS * 2), sls16::WARPS * 32, 0, e->stream>>>(nullptr, nullptr, states, n_chains, 0, 0u, seed, steps, nullptr,
                                                                                                target, noise_pct, e->interrupt_dev, totals_dev, os);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}

}  // namespace tss
