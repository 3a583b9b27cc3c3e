// Kernel (b): batched stochastic local search over support sites (see sls_spec.hpp for the algorithm).
// One layout per warp, lane r = grid row r, cover counts as five bit-planes in registers, reach windows of all
// sites in an 8 KB shared-memory table per CTA, counter-based RNG.  No HBM traffic inside the step loop: the chain
// state (288 B) is read at the start of an epoch and written back at its end.
//
// Candidate scoring is lane-parallel: lane i scores ONE candidate layout (the current layout with site v_i added or
// u_i removed) exactly, as popcount(U & R(v_i)) resp. popcount(O & R(u_i)): seven indexed warp shuffles fetch the
// window rows, each is shifted/masked to its 7 window bits and packed (Horner, on the FMA pipe) into the same 28+21
// bit layout as the reach table, so two AND + POPC finish the score.  A swap step scores k removals and up to 25
// additions.  The ALU pipe is the limiter (ncu: profiles/), so the step is written to minimise ALU instructions:
// two hashes per step, no divisions, no selects on the shift direction.
#include "engine.hpp"
#include "sls_spec.hpp"
#include "sls_warp.cuh"

namespace tss {
namespace sls {

constexpr int WARPS = 4;  // chains per CTA

// Reach windows: one thread per tile, three masked dilations inside the tile's own 7x7 window (geodesic paths of
// length <= 3 never leave it).  rows: [n_terrains][32] ; out: [n_terrains][1024].
__global__ void build_reach_kernel(const uint32_t* __restrict__ rows, int n_terrains, uint2* __restrict__ out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n_terrains * 1024) return;
    out[i] = reach_window(rows + (size_t)(i >> 10) * 32, (int)(i & 1023));
}

struct WarpCtx {
    const uint2* tab;
    uint16_t* sites;
    uint16_t* stamps;  // step of the last flip of every site (16 bit)
    int lane, tenure;
};

// Removes the support with the smallest loss (random ties); supports added fewer than `tenure` steps ago are only
// chosen when every support is that young (use_tabu = false when dropping).  Returns the removed site.  Scores k
// candidate layouts.
__device__ __forceinline__ int remove_min_loss(Lane& L, const WarpCtx& w, int& k, uint32_t hs, uint32_t step, int ten, bool use_tabu) {
    uint32_t best_key = 0xffffffffu;
    int best_i = 0;
    for (int b = 0; b < k; b += 32) {
        int i = b + w.lane;
        bool valid = i < k;
        int v = valid ? w.sites[i] : 0;
        uint2 win = w.tab[v];
        int loss = score(L.O, v & 31, v >> 5, win);
        const uint32_t young = (use_tabu && is_tabu(step, w.stamps[v], ten)) ? TABU_BIT : 0u;
        uint32_t key = valid ? (young | ((uint32_t)loss << 16) | tie_remove(hs, (uint32_t)i)) : 0xffffffffu;
        uint32_t mn = __reduce_min_sync(FULL, key);
        if (mn < best_key) {
            best_key = mn;
            best_i = b + __ffs(__ballot_sync(FULL, key == mn)) - 1;
        }
    }
    int u = w.sites[best_i];
    __syncwarp();
    if (w.lane == 0) { w.sites[best_i] = w.sites[k - 1]; w.stamps[u] = (uint16_t)step; }
    __syncwarp();
    k--;
    planes_sub(L, row_mask(w.tab[u], u & 31, u >> 5, w.lane));
    derive(L);
    if (w.lane == (u >> 5)) L.S &= ~(1u << (u & 31));
    return u;
}

// WINDOW mode (large-neighbourhood search on grids larger than 32x32, lns.cu): the chain works on a 32x32 window of a
// bigger grid.  `terrain_rows` is the true ceiling of the window (reach tables are built from it), `need_rows` the
// tiles of the window NOT already covered by frozen supports outside the window's movable core, and only sites with
// core_lo <= x, y < core_hi may receive supports (their reach never leaves the window).
template <bool WINDOW>
__global__ void __launch_bounds__(WARPS * 32, 8) sls_kernel(const uint32_t* __restrict__ terrain_rows, const uint2* __restrict__ rtabs,
                                                        const uint32_t* __restrict__ need_rows, int core_lo, int core_hi,
                                                        ChainState* __restrict__ states, int n_chains, int chains_per_terrain,
                                                        uint32_t chain_offset, uint64_t seed, long long steps,
                                                        const int* __restrict__ bounds, int target, int noise_pct,
                                                        const volatile int* interrupt,
                                                        unsigned long long* __restrict__ totals) {
    __shared__ uint2 tab[1024];
    __shared__ uint16_t sites_all[WARPS][MAX_SITES];
    __shared__ uint16_t stamps_all[WARPS][1024];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int chain = blockIdx.x * WARPS + warp;
    const int terrain = chains_per_terrain > 0 ? (blockIdx.x * WARPS) / chains_per_terrain : 0;
    // a layout within the target is already known for this terrain (found in an earlier epoch): nothing to do.  Lets a host
    // queue several epochs back to back without a round trip in between (one-shot solves, sls_spec.hpp).
    if (target >= 0 && bounds[chains_per_terrain > 0 ? terrain : 0] <= target) return;
    for (int i = threadIdx.x; i < 1024; i += blockDim.x) tab[i] = rtabs[(size_t)terrain * 1024 + i];
    __syncthreads();
    if (chain >= n_chains) return;
    ChainState& st = states[chain];
    if (st.done) return;

    // bound of this epoch: smallest complete count known for this terrain when the epoch started (group = terrain)
    const int epoch_bound = bounds[chains_per_terrain > 0 ? terrain : 0];
    const uint32_t base = chain_base(seed, chain_offset + (uint32_t)chain);
    const uint32_t nq7 = noise_q7(noise_pct);
    WarpCtx w{tab, sites_all[warp], stamps_all[warp], lane, tenure_of(chain_offset + (uint32_t)chain)};
    Lane L;
    L.C = WINDOW ? need_rows[(size_t)terrain * 32 + lane] : terrain_rows[(size_t)terrain * 32 + lane];  // tiles that need cover
    L.S = st.S[lane];
    uint32_t bestS = st.bestS[lane];
    int k = st.k, best = st.best, done = 0;
    uint32_t step = st.step;
    unsigned long long scored = 0;
    uint32_t flips = 0;   // supports added + removed (the unit of SURVEY.md §8(d): one flip = one candidate layout evaluated incrementally)

    // rebuild the site list (row-major) and the cover-count planes from S; flip stamps start "half a period ago"
    {
        for (int i = lane; i < 1024; i += 32) w.stamps[i] = stamp_reset(step);
        int c = __popc(L.S), off = c;
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(FULL, off, o); if (lane >= o) off += t; }
        off -= c;
        for (uint32_t bits = L.S; bits; bits &= bits - 1) w.sites[off++] = (uint16_t)(lane * 32 + __ffs(bits) - 1);
        __syncwarp();
        L.c0 = L.c1 = L.c2 = L.c3 = L.c4 = 0;
        for (int i = 0; i < k; i++) { int v = w.sites[i]; planes_add(L, row_mask(tab[v], v & 31, v >> 5, lane)); }
        derive(L);
    }

    // diamond of the 25 window positions within Manhattan distance 3 (a superset of every reach set)
    int ldx, ldy;
    {
        int i = lane, r = (i >= 1) + (i >= 4) + (i >= 9) + (i >= 16) + (i >= 21) + (i >= 24);
        int start = r <= 4 ? r * r : (r == 5 ? 21 : 24);
        ldy = r - 3;
        ldx = (i - start) - (3 - abs(ldy));
    }
    const bool diamond = lane < 25, lhi = ldy >= 1;   // window rows 4..6 live in the second table word
    const int lrowsh = 7 * ((ldy + 3) & 3);

    long long it = 0;
    for (; it < steps; it++, step++) {
        if ((it & 1023) == 1023 && *interrupt) break;
        const int limit = min(epoch_bound, best);
        const uint32_t hs = step_hash(base, step);
        const uint32_t tie = tie_add(hs, (uint32_t)lane);
        const int ten = effective_tenure(w.tenure, k);  // fixed for the whole step
        if (k >= limit) {  // 1. too many supports for an improvement: drop one
            if (k == 0) { done = 1; break; }
            scored += (unsigned)k;
            remove_min_loss(L, w, k, hs, step, ten, false);
            flips++;
            continue;
        }
        if (!__any_sync(FULL, L.U != 0)) {  // 2. complete layout with k < limit supports
            best = k;
            bestS = L.S;
            if (k <= target || k == 0) { done = 1; it++; step++; break; }
            continue;
        }
        if (k == limit - 1 && k > 0) {  // 3. at capacity: swap = remove + add
            scored += (unsigned)k;
            remove_min_loss(L, w, k, hs, step, ten, true);
            flips++;
        }
        const uint32_t rowmask = __ballot_sync(FULL, L.U != 0);
        const int y = pick_rotated(rowmask, hs & 31u);
        const uint32_t Urow = __shfl_sync(FULL, L.U, y);
        const int x = pick_rotated(Urow, (hs >> 5) & 31u);
        const uint2 wt = tab[y * 32 + x];
        const int col = ldx + min(x, 3);  // window column of the candidate (window anchored at max(x-3, 0))
        bool valid = diamond && col >= 0 && (((lhi ? wt.y : wt.x) >> (lrowsh + col)) & 1u);
        if (WINDOW) valid = valid && x + ldx >= core_lo && x + ldx < core_hi && y + ldy >= core_lo && y + ldy < core_hi;
        const int cv = valid ? (y + ldy) * 32 + x + ldx : 0;
        const int nc = __popc(__ballot_sync(FULL, valid));
        if (WINDOW && nc == 0) { done = 1; break; }  // cannot happen from a complete start layout; never spin on it
        uint32_t key;
        if (((hs >> 10) & 127u) < nq7) {  // noise: uniformly random site of R(t)
            key = valid ? (0x10000u | tie) : 0u;
        } else {
            int g = score(L.U, cv & 31, cv >> 5, tab[cv]);
            const uint32_t fresh = is_tabu(step, w.stamps[cv], ten) ? 0u : TABU_BIT;  // recently removed sites only as a last resort
            key = valid ? (fresh | ((uint32_t)(g + 1) << 16) | tie) : 0u;
            scored += (unsigned)nc;
        }
        const uint32_t mx = __reduce_max_sync(FULL, key);
        const int v = __shfl_sync(FULL, cv, __ffs(__ballot_sync(FULL, key == mx)) - 1);
        planes_add(L, row_mask(tab[v], v & 31, v >> 5, lane));
        derive(L);
        if (lane == (v >> 5)) L.S |= 1u << (v & 31);
        if (lane == 0) { w.sites[k] = (uint16_t)v; w.stamps[v] = (uint16_t)step; }
        __syncwarp();
        k++;
        flips++;
    }

    st.S[lane] = L.S;
    st.bestS[lane] = bestS;
    if (lane == 0) {
        st.k = k; st.best = best; st.step = step; st.done = done;
        unsigned long long tot = ((unsigned long long)st.scored_hi << 32 | st.scored_lo) + scored;
        st.scored_lo = (uint32_t)tot; st.scored_hi = (uint32_t)(tot >> 32);
        st.steps_done += (uint32_t)it;
        atomicAdd(&totals[0], scored);
        atomicAdd(&totals[1], (unsigned long long)it);
        atomicAdd(&totals[2], (unsigned long long)flips);
    }
}

// Smallest `best` over chains [c0, c0+count) per group (ties: lowest chain).  One CTA per group.
// out[group] = (best count or NO_BOUND, chain index)
__global__ void best_reduce_kernel(const ChainState* __restrict__ states, int chains_per_group, int n_chains, int2* __restrict__ out,
                                   int* __restrict__ bounds) {
    __shared__ unsigned long long sm[256];
    const int c0 = blockIdx.x * chains_per_group, c1 = min(c0 + chains_per_group, n_chains);
    unsigned long long key = ~0ull;
    for (int c = c0 + threadIdx.x; c < c1; c += blockDim.x) {
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
        int2 r = sm[0] == ~0ull ? make_int2(NO_BOUND, -1) : make_int2((int)(sm[0] >> 32), (int)(sm[0] & 0xffffffffu));
        out[blockIdx.x] = r;
        if (r.x < bounds[blockIdx.x]) bounds[blockIdx.x] = r.x;  // next epoch looks for fewer than the best known
    }
}

// Single-group portfolios with many chains (56832 per GPU for the thread-per-chain kernel): the same reduction spread
// over the device, folded with a 64-bit atomicMin on (best << 32 | chain); best_finalize_kernel publishes it and re-arms
// the key.  (One CTA walking 56832 chain states took 125 us per epoch.)
__global__ void best_reduce_wide_kernel(const ChainState* __restrict__ states, int n_chains, unsigned long long* __restrict__ key_out) {
    unsigned long long key = ~0ull;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < n_chains; c += gridDim.x * blockDim.x) {
        unsigned long long kk = ((unsigned long long)(uint32_t)states[c].best << 32) | (uint32_t)c;
        key = kk < key ? kk : key;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long other = __shfl_xor_sync(FULL, key, o);
        key = other < key ? other : key;
    }
    if ((threadIdx.x & 31) == 0 && key != ~0ull) atomicMin(key_out, key);
}
__global__ void best_finalize_kernel(unsigned long long* __restrict__ key, int2* __restrict__ out, int* __restrict__ bounds) {
    const unsigned long long k = *key;
    int2 r = k == ~0ull ? make_int2(NO_BOUND, -1) : make_int2((int)(k >> 32), (int)(k & 0xffffffffu));
    out[0] = r;
    if (r.x < bounds[0]) bounds[0] = r.x;
    *key = ~0ull;
}

__global__ void init_states_kernel(ChainState* states, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ChainState s;
    for (int r = 0; r < 32; r++) { s.S[r] = 0; s.bestS[r] = 0; }
    s.k = 0; s.best = NO_BOUND; s.step = 0; s.done = 0;
    s.scored_lo = s.scored_hi = 0; s.steps_done = 0;
    s.reserved = 0;
    states[i] = s;
}

}  // namespace sls

// ---------------------------------------------------------------------------------------------- launch helpers
int sls_build_reach(tss_engine* e, const uint32_t* rows_dev, int n_terrains, uint2* tabs_dev) {
    long long total = (long long)n_terrains * 1024;
    sls::build_reach_kernel<<<(unsigned)((total + 255) / 256), 256, 0, e->stream>>>(rows_dev, n_terrains, tabs_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}
int sls_init_states(tss_engine* e, sls::ChainState* states, int n) {
    sls::init_states_kernel<<<(n + 127) / 128, 128, 0, e->stream>>>(states, n);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}
int sls_run(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, int n_chains,
            int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
            int noise_pct, unsigned long long* totals_dev) {
    int blocks = (n_chains + sls::WARPS - 1) / sls::WARPS;
    sls::sls_kernel<false><<<blocks, sls::WARPS * 32, 0, e->stream>>>(rows_dev, tabs_dev, nullptr, 0, 32, states, n_chains, chains_per_terrain,
                                                                    chain_offset, seed, steps, bounds_dev, target, noise_pct, e->interrupt_dev,
                                                                    totals_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}
int sls_run_windows(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, const uint32_t* need_dev, int core_lo, int core_hi,
                    sls::ChainState* states, int n_chains, int chains_per_window, uint32_t chain_offset, uint64_t seed, long long steps,
                    const int* bounds_dev, unsigned long long* totals_dev, int noise_pct) {
    int blocks = (n_chains + sls::WARPS - 1) / sls::WARPS;
    sls::sls_kernel<true><<<blocks, sls::WARPS * 32, 0, e->stream>>>(rows_dev, tabs_dev, need_dev, core_lo, core_hi, states, n_chains,
                                                                   chains_per_window, chain_offset, seed, steps, bounds_dev, 0, noise_pct,
                                                                   e->interrupt_dev, totals_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}
int sls_best_reduce(tss_engine* e, const sls::ChainState* states, int chains_per_group, int n_chains, int n_groups, int2* out_dev,
                    int* bounds_dev, unsigned long long* key_dev) {
    if (n_groups == 1 && key_dev && n_chains >= 1024) {  // key_dev holds ~0 between calls
        sls::best_reduce_wide_kernel<<<(n_chains + 255) / 256, 256, 0, e->stream>>>(states, n_chains, key_dev);
        sls::best_finalize_kernel<<<1, 1, 0, e->stream>>>(key_dev, out_dev, bounds_dev);
        TSS_CHECK_LAUNCH(e);
        e->stats.kernel_launches += 2;
        return TSS_OK;
    }
    sls::best_reduce_kernel<<<n_groups, n_groups > 1 ? 32 : 256, 0, e->stream>>>(states, chains_per_group, n_chains, out_dev, bounds_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}

}  // namespace tss
