// Large grids (wider or taller than 32) with platform sets beyond {1x1}: large-neighbourhood search over PLACEMENTS by window
// decomposition around the placement search (sls_multi.cu, WINDOW mode) — TSS_KERNEL_WINDOW_PLACEMENTS.
//
// The global layout lives on the device as an anchor grid A u8[w*h]: 0 = no platform anchored at the tile, otherwise key + 1
// (dims keys numbered as the engine numbers them: defs order, unflipped then flipped).  Footprints are always inside the grid
// and pairwise disjoint, and the layout is always complete; it starts as the greedy placement cover (greedy.cu) with redundant
// platforms pruned, built by the engine.  Phase p tiles the grid with 32x32 windows at offset OFF[p & 3] (as lns.cu), numbered
// row-major.  A platform anchored at (X, Y) with effective dims (pw, ph) is MOVABLE iff 3 <= (X - ox) mod 32 and
// (X - ox) mod 32 + pw <= 29, and the same for Y, oy and ph: its reach (footprint + 3) then stays inside its window, so
// windows never interact.  Every other platform is frozen for the phase (with footprints of at most 6x6 every placement is
// movable at some offset).
//   1. Ff = the frozen footprints;  covF = three ceiling-masked dilations of Ff & C        (exact cover of the frozen platforms)
//   2. per window: ceiling rows, need = C & ~covF, occupancy Ff, the box additions must lie in, and the movable platforms in
//      row-major anchor order -> the start state of `seeds` chains (best = their total cost)
//   3. one epoch of the placement search on every window: each chain looks for a complete window layout of lower cost
//   4. per window the chain with the lowest best wins (lowest chain on ties); the window's movable anchors are cleared and
//      the winner's best placements written back
//   5. the objective (platform count, or total weight) of the global layout, reduced on the device into pinned memory
//
// Per-type limits (tss_search_create_with_limits): class j (tss::card_limit_classes) holds at most L_j platforms.  The windows
// pick their winners independently, so each window gets a budget per class: with n_j = the platforms of the global layout in
// class j (kept current on the device), m_{w,j} = the movable platforms of window w in class j, s_j = L_j - n_j >= 0 and N windows,
// window w's chains run with limits b_{w,j} = m_{w,j} + floor(s_j / N) + [((w - p) mod N) < (s_j mod N)] (the remainder rotates
// with the phase p).  Every chain starts from the window's movable platforms, which fit b_{w,j}, and the LIMITS step rule keeps
// every layout of every chain within b_{w,j}; frozen platforms stay.  So after the write-back n_j <= (n_j - sum_w m_{w,j}) +
// sum_w b_{w,j} = L_j whatever each window's winner is.  n_j is recounted after every write-back and copied to pinned memory next
// to the objective, for the host to check.
#include "engine.hpp"
#include "lns_window.cuh"
#include "sls_multi.hpp"
#include "sls_spec.hpp"

namespace tss {
int slsm_run_windows(tss_engine* e, const uint32_t* rows_dev, const slsm::WindowM& wm, const int2* keys_dev, const int* costs_dev, const int* order_dev,
                     int n_keys, slsm::MultiState* states, int n_chains, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev,
                     int target, int noise_pct, unsigned long long* totals_dev, const slsm::LimitsM& lm);

namespace lnsp {

constexpr int CORE_LO = 3, CORE_HI = 29;

// (lx, ly) = the anchor's position in its window: (X - ox) mod 32, (Y - oy) mod 32
__device__ __forceinline__ bool movable_local(int lx, int ly, int2 d) {
    return lx >= CORE_LO && lx + d.x <= CORE_HI && ly >= CORE_LO && ly + d.y <= CORE_HI;
}

// one thread per tile: the footprints of the frozen platforms OR-ed into F (zeroed before)
__global__ void stamp_frozen_kernel(const uint8_t* __restrict__ A, int w, int h, int wpr, const int2* __restrict__ keys, int ox, int oy,
                                    uint32_t* __restrict__ F) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= w * h || !A[t]) return;
    const int X = t % w, Y = t / w;
    const int2 d = keys[A[t] - 1];
    if (movable_local((X - ox) & 31, (Y - oy) & 31, d)) return;
    const int wq = X >> 5, sh = X & 31;
    const uint32_t bits = (1u << d.x) - 1u;
    for (int y = Y; y < Y + d.y; y++) {
        atomicOr(&F[y * wpr + wq], bits << sh);
        if (sh + d.x > 32) atomicOr(&F[y * wpr + wq + 1], bits >> (32 - sh));
    }
}

__global__ void and_kernel(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, uint32_t* __restrict__ out, int nw) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nw) out[i] = a[i] & b[i];
}

// one warp per window, lane = window row: ceiling, need and occupancy rows, the box, and the movable platforms as the start
// state of the window's chains
__global__ void extract_kernel(const uint8_t* __restrict__ A, const uint32_t* __restrict__ C, const uint32_t* __restrict__ covF,
                               const uint32_t* __restrict__ Ff, int w, int h, int wpr, const int2* __restrict__ keys, const int* __restrict__ costs,
                               int ox, int oy, int nwx, int n_windows, int seeds, uint32_t step0, uint32_t* __restrict__ rows_win,
                               uint32_t* __restrict__ need_win, uint32_t* __restrict__ occ_win, int4* __restrict__ box,
                               slsm::MultiState* __restrict__ states, int* __restrict__ bounds) {
    const int win = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (win >= n_windows) return;
    const int gx0 = ox + 32 * (win % nwx), gy0 = oy + 32 * (win / nwx), gy = gy0 + lane;
    const uint32_t c = lns::fetch32(C, gy, gx0, h, wpr);
    rows_win[win * 32 + lane] = c;
    need_win[win * 32 + lane] = c & ~lns::fetch32(covF, gy, gx0, h, wpr);
    occ_win[win * 32 + lane] = lns::fetch32(Ff, gy, gx0, h, wpr);
    if (lane == 0) {
        box[win] = make_int4(max(CORE_LO, -gx0), max(CORE_LO, -gy0), min(CORE_HI, w - gx0), min(CORE_HI, h - gy0));
        bounds[win] = sls::NO_BOUND;
    }
    // movable anchors of this row: count and cost, then their row-major positions
    const bool row_ok = lane >= CORE_LO && lane < CORE_HI && gy >= 0 && gy < h;
    int n = 0, cost = 0;
    for (int lx = CORE_LO; row_ok && lx < CORE_HI; lx++) {
        const int X = gx0 + lx;
        const int a = (X >= 0 && X < w) ? A[gy * w + X] : 0;
        if (a && movable_local(lx, lane, keys[a - 1])) { n++; cost += costs[a - 1]; }
    }
    int off = n;
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, off, o);
        if (lane >= o) off += v;
    }
    const int k = __shfl_sync(0xffffffffu, off, 31);
    off -= n;
    const int total = __reduce_add_sync(0xffffffffu, cost);
    for (int j = 0; j < seeds; j++) {
        slsm::MultiState& st = states[win * seeds + j];
        int i = off;
        for (int lx = CORE_LO; row_ok && lx < CORE_HI; lx++) {
            const int X = gx0 + lx;
            const int a = (X >= 0 && X < w) ? A[gy * w + X] : 0;
            if (a && movable_local(lx, lane, keys[a - 1])) {
                const uint16_t code = (uint16_t)((a - 1) << 10 | lane << 5 | lx);
                st.items[i] = code;
                st.best_items[i] = code;
                i++;
            }
        }
        if (lane == 0) {
            st.k = k; st.best_k = k; st.best = total; st.step = step0;
            st.tabu_add = -1; st.tabu_rem = -1; st.done = 0;
        }
    }
}

// one thread per tile: n_j += 1 for every class j of the platform anchored there (counts zeroed before)
__global__ void count_classes_kernel(const uint8_t* __restrict__ A, int n, const int* __restrict__ mask, int* __restrict__ ncls) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n || !A[t]) return;
    for (uint32_t m = (uint32_t)mask[A[t] - 1]; m; m &= m - 1) atomicAdd(&ncls[__ffs(m) - 1], 1);
}

// one warp per window, lane = window row: m_{w,j} = the movable platforms of the window in class j, then lane j writes the
// window's budget b_{w,j} = m_{w,j} + its share of the slack s_j = L_j - n_j (the remainder rotates with the phase)
__global__ void budget_kernel(const uint8_t* __restrict__ A, int w, int h, const int2* __restrict__ keys, const int* __restrict__ mask,
                              const int* __restrict__ limit, const int* __restrict__ ncls, int n_classes, int ox, int oy, int nwx, int n_windows,
                              int phase, int* __restrict__ budgets) {
    const int win = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (win >= n_windows) return;
    const int gx0 = ox + 32 * (win % nwx), gy0 = oy + 32 * (win / nwx), gy = gy0 + lane;
    const bool row_ok = lane >= CORE_LO && lane < CORE_HI && gy >= 0 && gy < h;
    int mine = 0;
    for (int j = 0; j < n_classes; j++) {
        int n = 0;
        for (int lx = CORE_LO; row_ok && lx < CORE_HI; lx++) {
            const int X = gx0 + lx;
            const int a = (X >= 0 && X < w) ? A[gy * w + X] : 0;
            if (a && ((mask[a - 1] >> j) & 1) && movable_local(lx, lane, keys[a - 1])) n++;
        }
        n = __reduce_add_sync(0xffffffffu, n);
        if (lane == j) mine = n;
    }
    if (lane < n_classes) {
        const int slack = limit[lane] - ncls[lane], pos = ((win - phase) % n_windows + n_windows) % n_windows;
        budgets[win * slsm::MAX_KEYS + lane] = mine + slack / n_windows + (pos < slack % n_windows ? 1 : 0);
    }
}

// one warp per window: the chain with the lowest best (lowest chain on ties) -> best[win] = (best, chain)
__global__ void window_best_kernel(const slsm::MultiState* __restrict__ states, int n_windows, int seeds, int2* __restrict__ best) {
    const int win = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (win >= n_windows) return;
    unsigned long long key = ~0ull;
    for (int j = lane; j < seeds; j += 32) {
        const int chain = win * seeds + j;
        const unsigned long long kk = ((unsigned long long)(uint32_t)states[chain].best << 32) | (uint32_t)chain;
        key = kk < key ? kk : key;
    }
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long v = __shfl_xor_sync(0xffffffffu, key, o);
        key = v < key ? v : key;
    }
    if (lane == 0) best[win] = make_int2((int)(key >> 32), (int)(key & 0xffffffffu));
}

// one warp per window: clear the movable anchors, then write the winner's best placements back.  Windows touch disjoint tiles:
// movable anchors and the winner's anchors lie in the window's [3, 29)^2.
__global__ void writeback_kernel(uint8_t* __restrict__ A, int w, int h, const int2* __restrict__ keys, int ox, int oy, int nwx, int n_windows,
                                 const int2* __restrict__ best, const slsm::MultiState* __restrict__ states) {
    const int win = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (win >= n_windows) return;
    const int gx0 = ox + 32 * (win % nwx), gy0 = oy + 32 * (win / nwx), gy = gy0 + lane;
    if (lane >= CORE_LO && lane < CORE_HI && gy >= 0 && gy < h)
        for (int lx = CORE_LO; lx < CORE_HI; lx++) {
            const int X = gx0 + lx;
            if (X < 0 || X >= w) continue;
            const int a = A[gy * w + X];
            if (a && movable_local(lx, lane, keys[a - 1])) A[gy * w + X] = 0;
        }
    __syncwarp();
    const slsm::MultiState& st = states[best[win].y];
    for (int i = lane; i < st.best_k; i += 32) {
        const int code = st.best_items[i];
        A[(gy0 + ((code >> 5) & 31)) * w + gx0 + (code & 31)] = (uint8_t)((code >> 10) + 1);
    }
}

// *out += total cost of the layout
__global__ void objective_kernel(const uint8_t* __restrict__ A, int n, const int* __restrict__ costs, int* __restrict__ out) {
    int v = 0;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) v += A[i] ? costs[A[i] - 1] : 0;
    v = __reduce_add_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(out, v);
}

}  // namespace lnsp

struct LnspSearch {
    int w = 0, h = 0, wpr = 0, nw = 0, seeds = 0, max_windows = 0, phase = 0, noise = sls::DEFAULT_NOISE_PCT, n_keys = 0;
    uint64_t seed = 0;
    uint32_t chain_offset = 0;
    const int2* keys = nullptr;                  // owned by the caller: effective dims per key, cost per key, keys by area
    const int* costs = nullptr;
    const int* order = nullptr;
    uint8_t* A = nullptr;                        // anchor grid
    uint32_t *C = nullptr, *F = nullptr, *T0 = nullptr, *T1 = nullptr;   // ceiling, frozen footprints, frozen cover ping/pong
    uint32_t *rows_win = nullptr, *need_win = nullptr, *occ_win = nullptr;
    int4* box = nullptr;
    slsm::MultiState* states = nullptr;
    int2* best = nullptr;
    int* bounds = nullptr;
    unsigned long long* totals = nullptr;
    int* obj_dev = nullptr;
    int* obj_host = nullptr;                     // pinned
    unsigned long long* totals_host = nullptr;   // pinned [3]
    // per-type limits (n_classes > 0): class mask per key [MAX_KEYS] then L_j [MAX_KEYS]; budgets [max_windows][MAX_KEYS]; n_j
    int n_classes = 0;
    std::vector<int> limit;                      // L_j (host)
    int* classes = nullptr;
    int* budgets = nullptr;
    int* ncls_dev = nullptr;
    int* ncls_host = nullptr;                    // pinned [MAX_KEYS]: n_j of the current layout
};

void lnsp_destroy(LnspSearch* s) {
    if (!s) return;
    cudaFree(s->A); cudaFree(s->C); cudaFree(s->F); cudaFree(s->T0); cudaFree(s->T1); cudaFree(s->rows_win); cudaFree(s->need_win); cudaFree(s->occ_win);
    cudaFree(s->box); cudaFree(s->states); cudaFree(s->best); cudaFree(s->bounds); cudaFree(s->totals); cudaFree(s->obj_dev);
    cudaFree(s->classes); cudaFree(s->budgets); cudaFree(s->ncls_dev);
    if (s->obj_host) cudaFreeHost(s->obj_host);
    if (s->ncls_host) cudaFreeHost(s->ncls_host);
    if (s->totals_host) cudaFreeHost(s->totals_host);
    delete s;
}

// The objective of the current layout, in-stream into pinned memory (read after a synchronisation).
int lnsp_objective(tss_engine* e, LnspSearch* s) {
    TSS_CUDA(e, cudaMemsetAsync(s->obj_dev, 0, sizeof(int), e->stream));
    lnsp::objective_kernel<<<32, 256, 0, e->stream>>>(s->A, s->w * s->h, s->costs, s->obj_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    TSS_CUDA(e, cudaMemcpyAsync(s->obj_host, s->obj_dev, sizeof(int), cudaMemcpyDeviceToHost, e->stream));
    return TSS_OK;
}

// n_j of the current layout, in-stream into ncls_dev and pinned memory (read after a synchronisation)
static int lnsp_count_classes(tss_engine* e, LnspSearch* s) {
    TSS_CUDA(e, cudaMemsetAsync(s->ncls_dev, 0, sizeof(int) * slsm::MAX_KEYS, e->stream));
    lnsp::count_classes_kernel<<<(s->w * s->h + 255) / 256, 256, 0, e->stream>>>(s->A, s->w * s->h, s->classes, s->ncls_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    TSS_CUDA(e, cudaMemcpyAsync(s->ncls_host, s->ncls_dev, sizeof(int) * slsm::MAX_KEYS, cudaMemcpyDeviceToHost, e->stream));
    return TSS_OK;
}

// anchors: the start layout (u8[w*h], 0 or key + 1), complete, footprints in bounds and disjoint.  keys / costs / order stay
// owned by the caller and must outlive the search.  n_classes > 0: per-type limits, class_mask[n_keys] and class_limit[n_classes]
// (tss::card_limit_classes), which the start layout keeps.  Synchronises the stream.
int lnsp_create(tss_engine* e, const uint8_t* grid, int w, int h, const uint8_t* anchors, const int2* keys_dev, const int* costs_dev, const int* order_dev,
                int n_keys, int seeds, uint64_t seed, uint32_t chain_offset, int noise, const uint32_t* class_mask, const int* class_limit, int n_classes,
                LnspSearch** out) {
    LnspSearch* s = new LnspSearch();
    s->w = w; s->h = h; s->wpr = (w + 31) / 32; s->nw = h * s->wpr; s->seeds = seeds; s->seed = seed; s->chain_offset = chain_offset; s->noise = noise;
    s->keys = keys_dev; s->costs = costs_dev; s->order = order_dev; s->n_keys = n_keys;
    s->max_windows = ((w + 31) / 32 + 1) * ((h + 31) / 32 + 1);
    const size_t nwb = sizeof(uint32_t) * (size_t)s->nw, winb = sizeof(uint32_t) * 32 * (size_t)s->max_windows;
    BitGrid bg = BitGrid::from_bytes(grid, w, h);
    cudaError_t err = cudaSuccess;
    auto A = [&](void** p, size_t bytes) { if (err == cudaSuccess) err = cudaMalloc(p, bytes); };
    A((void**)&s->A, (size_t)w * h); A((void**)&s->C, nwb); A((void**)&s->F, nwb); A((void**)&s->T0, nwb); A((void**)&s->T1, nwb);
    A((void**)&s->rows_win, winb); A((void**)&s->need_win, winb); A((void**)&s->occ_win, winb); A((void**)&s->box, sizeof(int4) * (size_t)s->max_windows);
    A((void**)&s->states, sizeof(slsm::MultiState) * (size_t)s->max_windows * seeds);
    A((void**)&s->best, sizeof(int2) * (size_t)s->max_windows); A((void**)&s->bounds, sizeof(int) * (size_t)s->max_windows);
    A((void**)&s->totals, sizeof(unsigned long long) * 3); A((void**)&s->obj_dev, sizeof(int));
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->obj_host, sizeof(int), cudaHostAllocDefault);
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->totals_host, sizeof(unsigned long long) * 3, cudaHostAllocDefault);
    if (err == cudaSuccess) err = cudaMemcpyAsync(s->C, bg.rows.data(), nwb, cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) err = cudaMemcpyAsync(s->A, anchors, (size_t)w * h, cudaMemcpyHostToDevice, e->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(s->totals, 0, sizeof(unsigned long long) * 3, e->stream);
    std::vector<int> cls(2 * (size_t)slsm::MAX_KEYS, 0);
    if (n_classes > 0) {
        s->n_classes = n_classes;
        s->limit.assign(class_limit, class_limit + n_classes);
        for (int k = 0; k < n_keys; k++) cls[(size_t)k] = (int)class_mask[k];
        for (int j = 0; j < n_classes; j++) cls[(size_t)slsm::MAX_KEYS + j] = class_limit[j];
        A((void**)&s->classes, sizeof(int) * cls.size()); A((void**)&s->ncls_dev, sizeof(int) * slsm::MAX_KEYS);
        A((void**)&s->budgets, sizeof(int) * slsm::MAX_KEYS * (size_t)s->max_windows);
        if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->ncls_host, sizeof(int) * slsm::MAX_KEYS, cudaHostAllocDefault);
        if (err == cudaSuccess) err = cudaMemcpyAsync(s->classes, cls.data(), sizeof(int) * cls.size(), cudaMemcpyHostToDevice, e->stream);
    }
    if (err != cudaSuccess) { lnsp_destroy(s); return e->fail(TSS_E_CUDA, "lnsp_create: %s", cudaGetErrorString(err)); }
    s->totals_host[0] = s->totals_host[1] = s->totals_host[2] = 0;
    int rc = lnsp_objective(e, s);
    if (rc == TSS_OK && s->n_classes > 0) rc = lnsp_count_classes(e, s);
    if (rc == TSS_OK && cudaStreamSynchronize(e->stream) != cudaSuccess) rc = e->fail(TSS_E_CUDA, "lnsp_create: stream sync failed");
    if (rc != TSS_OK) { lnsp_destroy(s); return rc; }
    *out = s;
    return TSS_OK;
}

// One phase, asynchronous on the engine stream.
int lnsp_phase(tss_engine* e, LnspSearch* s, long long steps) {
    static const int OFF[4][2] = {{0, 0}, {-16, -16}, {0, -16}, {-16, 0}};   // as lns.cu
    const int ox = OFF[s->phase & 3][0], oy = OFF[s->phase & 3][1];
    const int nwx = (s->w - ox + 31) / 32, nwy = (s->h - oy + 31) / 32, n_windows = nwx * nwy, n_chains = n_windows * s->seeds;
    const int tb = 256, gb = (s->nw + tb - 1) / tb, gt = (s->w * s->h + tb - 1) / tb, gwin = (n_windows * 32 + 127) / 128;
    TSS_CUDA(e, cudaMemsetAsync(s->F, 0, sizeof(uint32_t) * (size_t)s->nw, e->stream));
    lnsp::stamp_frozen_kernel<<<gt, tb, 0, e->stream>>>(s->A, s->w, s->h, s->wpr, s->keys, ox, oy, s->F);
    lnsp::and_kernel<<<gb, tb, 0, e->stream>>>(s->F, s->C, s->T0, s->nw);
    lns::dilate_global_kernel<<<gb, tb, 0, e->stream>>>(s->T0, s->T1, s->C, s->nw, s->wpr);
    lns::dilate_global_kernel<<<gb, tb, 0, e->stream>>>(s->T1, s->T0, s->C, s->nw, s->wpr);
    lns::dilate_global_kernel<<<gb, tb, 0, e->stream>>>(s->T0, s->T1, s->C, s->nw, s->wpr);   // covF = T1
    lnsp::extract_kernel<<<gwin, 128, 0, e->stream>>>(s->A, s->C, s->T1, s->F, s->w, s->h, s->wpr, s->keys, s->costs, ox, oy, nwx, n_windows, s->seeds,
                                                      ((uint32_t)s->phase + 1u) << 20, s->rows_win, s->need_win, s->occ_win, s->box, s->states, s->bounds);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches += 6;
    if (s->n_classes > 0) {   // (n_j of the current layout is already in ncls_dev: counted at creation and after every write-back)
        lnsp::budget_kernel<<<gwin, 128, 0, e->stream>>>(s->A, s->w, s->h, s->keys, s->classes, s->classes + slsm::MAX_KEYS, s->ncls_dev, s->n_classes, ox, oy,
                                                         nwx, n_windows, s->phase, s->budgets);
        TSS_CHECK_LAUNCH(e);
        e->stats.kernel_launches++;
    }
    const slsm::WindowM wm{s->need_win, s->occ_win, s->box, s->seeds};
    const slsm::LimitsM lm{s->classes, s->budgets, s->n_classes};
    int rc = slsm_run_windows(e, s->rows_win, wm, s->keys, s->costs, s->order, s->n_keys, s->states, n_chains, s->chain_offset, s->seed, steps, s->bounds,
                              -1, s->noise, s->totals, lm);
    if (rc) return rc;
    lnsp::window_best_kernel<<<gwin, 128, 0, e->stream>>>(s->states, n_windows, s->seeds, s->best);
    lnsp::writeback_kernel<<<gwin, 128, 0, e->stream>>>(s->A, s->w, s->h, s->keys, ox, oy, nwx, n_windows, s->best, s->states);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches += 2;
    rc = lnsp_objective(e, s);
    if (rc == TSS_OK && s->n_classes > 0) rc = lnsp_count_classes(e, s);
    if (rc) return rc;
    TSS_CUDA(e, cudaMemcpyAsync(s->totals_host, s->totals, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost, e->stream));
    s->phase++;
    return TSS_OK;
}

// the anchor grid (host) after synchronising the stream
int lnsp_anchors(tss_engine* e, LnspSearch* s, std::vector<uint8_t>& anchors) {
    anchors.resize((size_t)s->w * s->h);
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    TSS_CUDA(e, cudaMemcpy(anchors.data(), s->A, anchors.size(), cudaMemcpyDeviceToHost));
    return TSS_OK;
}

int lnsp_value(const LnspSearch* s) { return s->obj_host[0]; }
unsigned long long lnsp_total(const LnspSearch* s, int i) { return s->totals_host[i]; }
int lnsp_chains(const LnspSearch* s) { return s->max_windows * s->seeds; }
// per-type limits: a class whose count in the current layout exceeds its limit (after a synchronisation), or -1
int lnsp_over_limit(const LnspSearch* s, int* count, int* limit) {
    for (int j = 0; j < s->n_classes; j++)
        if (s->ncls_host[j] > s->limit[(size_t)j]) { *count = s->ncls_host[j]; *limit = s->limit[(size_t)j]; return j; }
    return -1;
}

}  // namespace tss
