// Large grids (wider or taller than 32, e.g. SURVEY.md C4: 256x256): large-neighbourhood search by window
// decomposition around the per-warp SLS kernel (sls.cu, WINDOW mode).
//
// The global layout S (bit-packed rows in HBM) is ALWAYS a complete layout (it starts as "a support under every ceiling
// tile").  A phase tiles the grid with 32x32 windows at offset (ox, oy); each window's movable CORE is its inner 26x26
// (a support's reach is <= 3, so core supports only ever cover tiles of their own window and cores of different
// windows never interact); supports in the 6-wide gaps between cores are frozen for the phase.
//   1. F = S & gaps;  covF = three ceiling-masked dilations of F & C        (exact geodesic cover of the frozen supports)
//   2. per window: ceiling rows, need = ceiling & ~covF, core supports -> initial state of `seeds` chains (best = current)
//   3. reach tables, then the SLS kernel: every chain looks for a complete window layout with FEWER core supports
//   4. per window the best chain wins; its core supports are written back into S
// Completeness is invariant: every tile belongs to exactly one window and stays covered by frozen + core supports.
// Phases alternate the offset between 0 and -16 per axis so that every site is movable in some phase.
#include "engine.hpp"
#include "lns_window.cuh"
#include "sls_spec.hpp"

namespace tss {
int sls_build_reach(tss_engine* e, const uint32_t* rows_dev, int n_terrains, uint2* tabs_dev);
int sls_run_windows(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, const uint32_t* need_dev, int core_lo, int core_hi,
                    sls::ChainState* states, int n_chains, int chains_per_window, uint32_t chain_offset, uint64_t seed, long long steps,
                    const int* bounds_dev, unsigned long long* totals_dev, int noise_pct);
int sls_best_reduce(tss_engine* e, const sls::ChainState* states, int chains_per_group, int n_chains, int n_groups, int2* out_dev,
                    int* bounds_dev, unsigned long long* key_dev);

namespace lns {

constexpr int CORE_LO = 3, CORE_HI = 29;
constexpr uint32_t CORE_COLS = 0x1FFFFFF8u;  // window columns 3..28

__device__ __forceinline__ bool core_row(int y, int oy) { int r = (y - oy) & 31; return r >= CORE_LO && r < CORE_HI; }

// frozen supports of the phase: everything outside the cores.  colmask = core columns of one 32-bit word for this ox.
__global__ void gap_supports_kernel(const uint32_t* __restrict__ S, const uint32_t* __restrict__ C, uint32_t* __restrict__ F, int nw, int wpr,
                                    int oy, uint32_t colmask) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nw) return;
    int y = i / wpr;
    uint32_t core = core_row(y, oy) ? colmask : 0u;
    F[i] = S[i] & ~core & C[i];  // only supports under a ceiling tile support anything (platform_layout.rs:116-119)
}

// one warp per window: window rows, need mask, core supports -> chain states
__global__ void extract_windows_kernel(const uint32_t* __restrict__ C, const uint32_t* __restrict__ S, const uint32_t* __restrict__ covF, int h,
                                       int wpr, int ox, int oy, int nwx, int n_windows, int seeds, uint32_t phase,
                                       uint32_t* __restrict__ rows_win, uint32_t* __restrict__ need_win, sls::ChainState* __restrict__ states,
                                       int* __restrict__ bounds) {
    const int win = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (win >= n_windows) return;
    const int gx0 = ox + 32 * (win % nwx), gy = oy + 32 * (win / nwx) + lane;
    const uint32_t c = fetch32(C, gy, gx0, h, wpr), s = fetch32(S, gy, gx0, h, wpr), f = fetch32(covF, gy, gx0, h, wpr);
    const uint32_t core = (lane >= CORE_LO && lane < CORE_HI) ? CORE_COLS : 0u;
    const uint32_t score = s & core & c;  // core supports under a non-ceiling tile support nothing: they are dropped right here
    rows_win[win * 32 + lane] = c;
    need_win[win * 32 + lane] = c & ~f;
    int k = __popc(score);
    for (int o = 16; o > 0; o >>= 1) k += __shfl_xor_sync(0xffffffffu, k, o);
    if (lane == 0) bounds[win] = sls::NO_BOUND;
    for (int j = 0; j < seeds; j++) {
        sls::ChainState& st = states[win * seeds + j];
        st.S[lane] = score;
        st.bestS[lane] = score;
        if (lane == 0) {
            st.k = k; st.best = k; st.step = phase << 20; st.done = 0;
            st.scored_lo = st.scored_hi = 0; st.steps_done = 0;
        }
    }
}

// one warp per window: the best chain's core supports replace the window's core in the global layout
__global__ void writeback_windows_kernel(uint32_t* __restrict__ S, int h, int wpr, int ox, int oy, int nwx, int n_windows,
                                         const int2* __restrict__ best, const sls::ChainState* __restrict__ states) {
    const int win = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (win >= n_windows) return;
    const int chain = best[win].y;
    if (chain < 0 || lane < CORE_LO || lane >= CORE_HI) return;
    const int gx0 = ox + 32 * (win % nwx), gy = oy + 32 * (win / nwx) + lane;
    if (gy < 0 || gy >= h) return;
    const uint32_t row = states[chain].bestS[lane] & CORE_COLS;
    const int wq = gx0 >> 5, sh = gx0 & 31;
    // window bit b is grid column gx0 + b: low part lands in word wq (shifted left by sh), high part in word wq + 1
    const uint32_t mask_lo = CORE_COLS << sh, val_lo = row << sh;
    const uint32_t mask_hi = sh ? (CORE_COLS >> (32 - sh)) : 0u, val_hi = sh ? (row >> (32 - sh)) : 0u;
    if (wq >= 0 && wq < wpr) { atomicAnd(&S[gy * wpr + wq], ~mask_lo); atomicOr(&S[gy * wpr + wq], val_lo); }
    if (sh && wq + 1 >= 0 && wq + 1 < wpr) { atomicAnd(&S[gy * wpr + wq + 1], ~mask_hi); atomicOr(&S[gy * wpr + wq + 1], val_hi); }
}

__global__ void popcount_kernel(const uint32_t* __restrict__ X, int nw, int* __restrict__ out) {
    int v = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < nw; i += gridDim.x * blockDim.x) v += __popc(X[i]);
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, v);
}

// ---- multi-GPU portfolio: windows are independent sub-problems within a phase (cores never interact), and every rank starts
// the phase from the same layout with the same window grid but its own chain seeds.  So the ranks' results COMBINE: per window
// the rank whose best chain holds the fewest core supports wins (key = count * 64 + rank, one all-reduce-min over the window
// keys), every rank writes the cores of the windows it won into a zeroed bitboard (rank 0 adds the frozen supports, which
// are the same everywhere), and one all-reduce-sum — each bit has exactly one contributor, so the sum is an OR — gives every
// rank the same next layout: per window the best of (ranks x chains) attempts.  All in-stream, no host round trip.
__global__ void window_keys_kernel(const int2* __restrict__ best, int n_windows, int rank, uint32_t* __restrict__ keys) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_windows) keys[i] = best[i].y >= 0 ? (uint32_t)best[i].x * 64u + (uint32_t)rank : 0xffffffffu;
}
// one warp per window: OR the best chain's core supports into `G` if this rank won the window
__global__ void contribute_windows_kernel(uint32_t* __restrict__ G, int h, int wpr, int ox, int oy, int nwx, int n_windows, const int2* __restrict__ best,
                                          const sls::ChainState* __restrict__ states, const uint32_t* __restrict__ gkeys, int rank) {
    const int win = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (win >= n_windows) return;
    const int chain = best[win].y;
    if (chain < 0 || (int)(gkeys[win] & 63u) != rank || lane < CORE_LO || lane >= CORE_HI) return;
    const int gx0 = ox + 32 * (win % nwx), gy = oy + 32 * (win / nwx) + lane;
    if (gy < 0 || gy >= h) return;
    const uint32_t row = states[chain].bestS[lane] & CORE_COLS;
    const int wq = gx0 >> 5, sh = gx0 & 31;
    const uint32_t val_lo = row << sh, val_hi = sh ? (row >> (32 - sh)) : 0u;
    if (wq >= 0 && wq < wpr && val_lo) atomicOr(&G[gy * wpr + wq], val_lo);
    if (sh && wq + 1 >= 0 && wq + 1 < wpr && val_hi) atomicOr(&G[gy * wpr + wq + 1], val_hi);
}

}  // namespace lns

struct LnsSearch {
    int w = 0, h = 0, wpr = 0, nw = 0, seeds = 0, max_windows = 0, phase = 0, noise = sls::DEFAULT_NOISE_PCT;
    uint64_t seed = 0;
    uint32_t chain_offset = 0;
    uint32_t *C = nullptr, *S = nullptr, *F = nullptr, *T = nullptr;  // ceiling, layout, frozen cover ping/pong
    uint32_t *rows_win = nullptr, *need_win = nullptr;
    uint2* tabs = nullptr;
    sls::ChainState* states = nullptr;
    int2* best = nullptr;
    int* bounds = nullptr;
    unsigned long long* totals = nullptr;
    int* count_dev = nullptr;
    uint32_t* key_dev = nullptr;                 // [2 * max_windows]: this rank's per-window (count, rank) keys and their minima over the ranks
    uint32_t* G = nullptr;                       // this rank's contribution to the next layout (multi-GPU portfolio)
    int* count_host = nullptr;                   // pinned
    unsigned long long* totals_host = nullptr;   // pinned [3]
};

void lns_destroy(LnsSearch* s) {
    if (!s) return;
    cudaFree(s->C); cudaFree(s->S); cudaFree(s->F); cudaFree(s->T); cudaFree(s->rows_win); cudaFree(s->need_win); cudaFree(s->tabs);
    cudaFree(s->states); cudaFree(s->best); cudaFree(s->bounds); cudaFree(s->totals); cudaFree(s->count_dev); cudaFree(s->key_dev); cudaFree(s->G);
    if (s->count_host) cudaFreeHost(s->count_host);
    if (s->totals_host) cudaFreeHost(s->totals_host);
    delete s;
}

int lns_create(tss_engine* e, const uint8_t* grid, int w, int h, int seeds, uint64_t seed, uint32_t chain_offset, int noise, LnsSearch** out) {
    LnsSearch* s = new LnsSearch();
    s->w = w; s->h = h; s->wpr = (w + 31) / 32; s->nw = h * s->wpr; s->seeds = seeds; s->seed = seed; s->chain_offset = chain_offset;
    s->noise = noise;
    s->max_windows = ((w + 31) / 32 + 1) * ((h + 31) / 32 + 1);
    const size_t nwb = sizeof(uint32_t) * (size_t)s->nw, nch = (size_t)s->max_windows * seeds;
    BitGrid bg = BitGrid::from_bytes(grid, w, h);
    cudaError_t err = cudaSuccess;
    auto A = [&](void** p, size_t bytes) { if (err == cudaSuccess) err = cudaMalloc(p, bytes); };
    A((void**)&s->C, nwb); A((void**)&s->S, nwb); A((void**)&s->F, nwb); A((void**)&s->T, nwb);
    A((void**)&s->rows_win, sizeof(uint32_t) * 32 * (size_t)s->max_windows); A((void**)&s->need_win, sizeof(uint32_t) * 32 * (size_t)s->max_windows);
    A((void**)&s->tabs, sizeof(uint2) * 1024 * (size_t)s->max_windows); A((void**)&s->states, sizeof(sls::ChainState) * nch);
    A((void**)&s->best, sizeof(int2) * (size_t)s->max_windows); A((void**)&s->bounds, sizeof(int) * (size_t)s->max_windows);
    A((void**)&s->totals, sizeof(unsigned long long) * 3); A((void**)&s->count_dev, sizeof(int)); A((void**)&s->key_dev, sizeof(uint32_t) * 2 * (size_t)s->max_windows); A((void**)&s->G, nwb);
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->count_host, sizeof(int), cudaHostAllocDefault);
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->totals_host, sizeof(unsigned long long) * 3, cudaHostAllocDefault);
    // the start layout: a support under every ceiling tile (trivially complete)
    if (err == cudaSuccess) err = cudaMemcpyAsync(s->C, bg.rows.data(), nwb, cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) err = cudaMemcpyAsync(s->S, bg.rows.data(), nwb, cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(s->totals, 0, sizeof(unsigned long long) * 3, e->stream);
    if (err == cudaSuccess) err = cudaStreamSynchronize(e->stream);
    if (err != cudaSuccess) { lns_destroy(s); return e->fail(TSS_E_CUDA, "lns_create: %s", cudaGetErrorString(err)); }
    s->count_host[0] = bg.count();
    s->totals_host[0] = s->totals_host[1] = s->totals_host[2] = 0;
    *out = s;
    return TSS_OK;
}

// One phase, asynchronous on the engine stream.
int lns_phase(tss_engine* e, LnsSearch* s, long long steps, bool share) {
    static const int OFF[4][2] = {{0, 0}, {-16, -16}, {0, -16}, {-16, 0}};
    const int ox = OFF[s->phase & 3][0], oy = OFF[s->phase & 3][1];
    const uint32_t colmask = ox == 0 ? lns::CORE_COLS : ((lns::CORE_COLS >> 16) | (lns::CORE_COLS << 16));  // rotate by the offset
    const int nwx = (s->w - ox + 31) / 32, nwy = (s->h - oy + 31) / 32, n_windows = nwx * nwy, n_chains = n_windows * s->seeds;
    const int tb = 256, gb = (s->nw + tb - 1) / tb;
    lns::gap_supports_kernel<<<gb, tb, 0, e->stream>>>(s->S, s->C, s->F, s->nw, s->wpr, oy, colmask);
    lns::dilate_global_kernel<<<gb, tb, 0, e->stream>>>(s->F, s->T, s->C, s->nw, s->wpr);
    lns::dilate_global_kernel<<<gb, tb, 0, e->stream>>>(s->T, s->F, s->C, s->nw, s->wpr);
    lns::dilate_global_kernel<<<gb, tb, 0, e->stream>>>(s->F, s->T, s->C, s->nw, s->wpr);  // covF = T
    lns::extract_windows_kernel<<<(n_windows * 32 + 127) / 128, 128, 0, e->stream>>>(s->C, s->S, s->T, s->h, s->wpr, ox, oy, nwx, n_windows, s->seeds,
                                                                                  (uint32_t)s->phase + 1u, s->rows_win, s->need_win, s->states,
                                                                                  s->bounds);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches += 5;
    int rc = sls_build_reach(e, s->rows_win, n_windows, s->tabs);
    if (rc) return rc;
    rc = sls_run_windows(e, s->rows_win, s->tabs, s->need_win, lns::CORE_LO, lns::CORE_HI, s->states, n_chains, s->seeds, s->chain_offset, s->seed,
                         steps, s->bounds, s->totals, s->noise);
    if (rc) return rc;
    rc = sls_best_reduce(e, s->states, s->seeds, n_chains, n_windows, s->best, s->bounds, nullptr);
    if (rc) return rc;
    const bool combine = share && e->comm && comm_world(e->comm) > 1;
    if (!combine) {
        lns::writeback_windows_kernel<<<(n_windows * 32 + 127) / 128, 128, 0, e->stream>>>(s->S, s->h, s->wpr, ox, oy, nwx, n_windows, s->best, s->states);
        e->stats.kernel_launches++;
    } else {  // per window the best of all ranks (see the kernels above)
        const int rank = comm_rank(e->comm);
        uint32_t *keys = s->key_dev, *gkeys = s->key_dev + s->max_windows;
        lns::window_keys_kernel<<<(n_windows + 127) / 128, 128, 0, e->stream>>>(s->best, n_windows, rank, keys);
        rc = comm_allreduce_min_u32(e, e->comm, keys, gkeys, n_windows);
        if (rc) return rc;
        if (rank == 0) lns::gap_supports_kernel<<<gb, tb, 0, e->stream>>>(s->S, s->C, s->G, s->nw, s->wpr, oy, colmask);   // the frozen supports, once
        else TSS_CUDA(e, cudaMemsetAsync(s->G, 0, sizeof(uint32_t) * (size_t)s->nw, e->stream));
        lns::contribute_windows_kernel<<<(n_windows * 32 + 127) / 128, 128, 0, e->stream>>>(s->G, s->h, s->wpr, ox, oy, nwx, n_windows, s->best, s->states, gkeys, rank);
        TSS_CHECK_LAUNCH(e);
        rc = comm_allreduce_sum_u32(e, e->comm, s->G, s->S, s->nw);
        if (rc) return rc;
        e->stats.kernel_launches += 3;
    }
    TSS_CUDA(e, cudaMemsetAsync(s->count_dev, 0, sizeof(int), e->stream));
    lns::popcount_kernel<<<32, 256, 0, e->stream>>>(s->S, s->nw, s->count_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    TSS_CUDA(e, cudaMemcpyAsync(s->count_host, s->count_dev, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(s->totals_host, s->totals, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost, e->stream));
    s->phase++;
    return TSS_OK;
}

// layout rows (host) after synchronising the stream
int lns_layout(tss_engine* e, LnsSearch* s, std::vector<uint32_t>& rows) {
    rows.resize((size_t)s->nw);
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    TSS_CUDA(e, cudaMemcpy(rows.data(), s->S, sizeof(uint32_t) * rows.size(), cudaMemcpyDeviceToHost));
    return TSS_OK;
}

int lns_count(const LnsSearch* s) { return s->count_host[0]; }
unsigned long long lns_total(const LnsSearch* s, int i) { return s->totals_host[i]; }
int lns_chains(const LnsSearch* s) { return s->max_windows * s->seeds; }

}  // namespace tss
