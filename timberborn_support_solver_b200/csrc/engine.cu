// Engine, device buffers and the C ABI entry points that touch the GPU (include/tss.h).  Host-only entry points
// (world / encoder / layout decode) live in capi_host.cpp.
#include <algorithm>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "engine.hpp"

#include <chrono>
#include <cstring>
#include <new>

#include "sls_spec.hpp"

namespace tss {
int sls_build_reach(tss_engine* e, const uint32_t* rows_dev, int n_terrains, uint2* tabs_dev);
int sls_init_states(tss_engine* e, sls::ChainState* states, int n);
int sls_run(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, int n_chains,
            int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
            int noise_pct, unsigned long long* totals_dev);
int sls_best_reduce(tss_engine* e, const sls::ChainState* states, int chains_per_group, int n_chains, int n_groups, int2* out_dev,
                    int* bounds_dev, unsigned long long* key_dev);
// sls_h16.cu — two chains per warp for grids of at most 16 rows (chains_per_terrain must be 0 or a multiple of 8)
int sls_thread_cta_chains();   // chains per CTA of both thread-per-chain kernels (sls_thread.cuh)
// sls_t16.cu — one chain per thread for grids of at most 16 rows x 26 columns (chains_per_terrain 0 or a multiple of the CTA size)
bool sls_t16_fits(int w, int h);
int sls_t16_smem_violations();
int sls_t16_checked_build();
size_t sls_t16_list_words(int n_chains);
int sls_run_t16(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, uint32_t* site_lists, int n_chains,
                int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
                int noise_pct, unsigned long long* totals_dev);
// sls_p16.cu — one chain per thread, two grid rows per word, for grids of at most 16x16 (same site lists as sls_t16.cu)
bool sls_p16_fits(int w, int h);
int sls_p16_smem_violations();
int sls_run_p16(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, uint32_t* site_lists, int n_chains,
                int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
                int noise_pct, unsigned long long* totals_dev);
int sls_run_h16_oneshot(tss_engine* e, const uint32_t* rows32_host, int bound, uint32_t* rows_dev, uint2* tabs_dev, sls::ChainState* states,
                        int n_chains, uint64_t seed, long long steps, int* bounds_dev, int2* best_dev, unsigned long long* key_dev,
                        unsigned int* ticket_dev, int target, int noise_pct, unsigned long long* totals_dev, uint32_t* result_host_mapped);
int sls_run_h16(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, int n_chains,
                int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
                int noise_pct, unsigned long long* totals_dev);
int run_peaks(tss_engine* e, double* out, int n_out);
// lp.cu — fractional packing lower bound
int lp_run(tss_engine* e, const uint32_t* rows32_host, int W, int H, const std::vector<int2>& key_dims, const std::vector<int>& key_costs,
           const std::vector<uint32_t>& key_mask, const std::vector<int>& class_limit, int max_pivots, long long target, int* out_weights,
           unsigned long long* totals, int* info);
constexpr int kLpMaxClasses = 16;   // lp.cu: class columns of per-type limits; the weights buffer holds 1024 tile weights, then these
// lp_big.cu — the same bound on grids larger than 32x32 (first-order method, same certificate)
int lp_big_run(tss_engine* e, const uint32_t* rows_host, int W, int H, const std::vector<int2>& key_dims, const std::vector<int>& key_costs, int max_iters,
               long long target, int* out_weights, unsigned long long* totals, int* info);
// lb.cu — packing lower bound
int lb_run(tss_engine* e, const uint32_t* rows32_host, int W, int H, const std::vector<int2>& key_dims, uint64_t seed, int restarts,
           uint32_t* out_rows32, int* out_count);
int lb_run_big(tss_engine* e, const uint32_t* rows_host, int W, int H, uint64_t seed, int restarts, uint32_t* out_rows, int* out_count);
// lns.cu — window decomposition for grids larger than 32x32
struct LnsSearch;
int lns_create(tss_engine* e, const uint8_t* grid, int w, int h, int seeds, uint64_t seed, uint32_t chain_offset, int noise, LnsSearch** out);
void lns_destroy(LnsSearch* s);
int lns_phase(tss_engine* e, LnsSearch* s, long long steps, bool share);
int lns_layout(tss_engine* e, LnsSearch* s, std::vector<uint32_t>& rows);
int lns_count(const LnsSearch* s);
unsigned long long lns_total(const LnsSearch* s, int i);
int lns_chains(const LnsSearch* s);
// lns_placements.cu — window-decomposed placement search for grids larger than 32x32 (TSS_KERNEL_WINDOW_PLACEMENTS)
struct LnspSearch;
int lnsp_create(tss_engine* e, const uint8_t* grid, int w, int h, const uint8_t* anchors, const int2* keys_dev, const int* costs_dev, const int* order_dev,
                int n_keys, int seeds, uint64_t seed, uint32_t chain_offset, int noise, const uint32_t* class_mask, const int* class_limit, int n_classes,
                LnspSearch** out);
void lnsp_destroy(LnspSearch* s);
int lnsp_phase(tss_engine* e, LnspSearch* s, long long steps);
int lnsp_objective(tss_engine* e, LnspSearch* s);
int lnsp_anchors(tss_engine* e, LnspSearch* s, std::vector<uint8_t>& anchors);
int lnsp_value(const LnspSearch* s);
unsigned long long lnsp_total(const LnspSearch* s, int i);
int lnsp_chains(const LnspSearch* s);
int lnsp_over_limit(const LnspSearch* s, int* count, int* limit);
// sls_multi.cu — placements of several platform types
size_t slsm_state_bytes();
int slsm_max_keys();
int slsm_init(tss_engine* e, void* states, int n);
int slsm_run(tss_engine* e, const uint32_t* rows_dev, int W, int H, const int2* keys_dev, const int* costs_dev, const int* order_dev, int n_keys, void* states, int n_chains,
             uint32_t chain_offset, uint64_t seed, long long steps, int* bounds_dev, int target, int noise_pct, unsigned long long* totals_dev,
             int2* best_dev, const int* limits_dev, int n_classes);
int slsm_read_best(tss_engine* e, const void* states, int chain, std::vector<uint16_t>& codes);
int slsm_run_oneshot(tss_engine* e, const uint32_t* rows32_host, int bound, uint32_t* rows_dev, int W, int H, const int2* keys_dev, const int* costs_dev,
                     const int* order_dev, int n_keys, void* states, int n_chains, uint64_t seed, long long steps, int* bounds_dev, int2* best_dev,
                     unsigned long long* key_dev, unsigned int* ticket_dev, int target, int noise_pct, unsigned long long* totals_dev,
                     uint32_t* result_host_mapped);
int slsm_witness(tss_engine* e, const void* states, const int2* best_dev, const int2* keys_dev, uint16_t* codes_dev, int4* plats_dev, uint32_t* offsets_dev);
int slsm_max_items();
// greedy.cu — parallel greedy placement cover for grids larger than 32x32 (platform sets beyond {1x1})
int greedy_cover(tss_engine* e, const uint32_t* C_rows_host, int w, int h, const std::vector<int2>& keys, std::vector<int4>& out);
int slsm_read_states(tss_engine* e, const void* states, int n_chains, uint16_t* items, int32_t* k, uint16_t* best_items, int32_t* best_k,
                     int32_t* best, uint32_t* step);

// u8 grids [n][w*h] -> rows32 [n][32] (one u32 per row, rows >= h are zero); w, h <= 32
__global__ void pack_rows32_kernel(const uint8_t* __restrict__ bytes, int w, int h, long long n, uint32_t* __restrict__ out) {
    long long total = n * 32;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        long long t = i >> 5;
        int y = (int)(i & 31);
        uint32_t v = 0;
        if (y < h) {
            const uint8_t* src = bytes + t * (long long)w * h + (long long)y * w;
            for (int x = 0; x < w; x++) v |= (uint32_t)(src[x] != 0) << x;
        }
        out[i] = v;
    }
}

// bounds[i] = min(bounds[i], value) (value = NO_BOUND with reset: a plain fill) — in-stream, no host round trip
__global__ void bound_min_kernel(int* __restrict__ bounds, int n, int value, bool reset) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) bounds[i] = reset ? value : min(bounds[i], value);
}

// One-shot solves: the best chain's layout fetched AND re-validated on the device in the same stream as the epoch
// (kernel (a) in its one-warp form: lane r = row r, validate()'s three ceiling-masked dilations with shuffles,
// src/encoder/platform_layout.rs:127-141).  out[0..31] = support rows, out[32] = unsupported tiles, out[33] = supports.
__global__ void witness_kernel(const sls::ChainState* __restrict__ states, const int2* __restrict__ best, const uint32_t* __restrict__ terrain_rows,
                               uint32_t* __restrict__ out) {
    const int lane = threadIdx.x, c = best[0].y;
    const uint32_t S = c >= 0 ? states[c].bestS[lane] : 0u, C = terrain_rows[lane];
    uint32_t X = S & C;
    for (int round = 0; round < kTerrainSupportDistance - 1; round++) {
        uint32_t up = __shfl_up_sync(0xffffffffu, X, 1), down = __shfl_down_sync(0xffffffffu, X, 1);
        if (lane == 0) up = 0;
        if (lane == 31) down = 0;
        X = (X | (X << 1) | (X >> 1) | up | down) & C;
    }
    const int unc = __reduce_add_sync(0xffffffffu, __popc(C & ~X)), cnt = __reduce_add_sync(0xffffffffu, __popc(S));
    out[lane] = S;
    if (lane == 0) { out[32] = (uint32_t)unc; out[33] = (uint32_t)cnt; }
}

// best layout rows of every terrain group: out[group][32] = states[best[group].y].bestS (zeros if the group found nothing)
__global__ void gather_best_rows_kernel(const sls::ChainState* __restrict__ states, const int2* __restrict__ best, int n_groups,
                                        uint32_t* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_groups * 32) return;
    int c = best[i >> 5].y;
    out[i] = c >= 0 ? states[c].bestS[i & 31] : 0u;
}
}  // namespace tss

void* tss_engine::dev(int slot, size_t bytes) {
    TssBuffer& b = scratch[slot];
    if (bytes <= b.cap && b.ptr) return b.ptr;
    if (b.ptr) { cudaStreamSynchronize(stream); cudaFree(b.ptr); b.ptr = nullptr; b.cap = 0; }
    size_t want = bytes < 4096 ? 4096 : bytes + bytes / 4;
    cudaError_t err = cudaMalloc(&b.ptr, want);
    if (err != cudaSuccess) { b.ptr = nullptr; fail(TSS_E_CUDA, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(err)); return nullptr; }
    b.cap = want;
    return b.ptr;
}
void* tss_engine::pin(int slot, size_t bytes) {
    TssBuffer& b = staging[slot];
    if (bytes <= b.cap && b.ptr) return b.ptr;
    if (b.ptr) { cudaStreamSynchronize(stream); cudaFreeHost(b.ptr); b.ptr = nullptr; b.cap = 0; }
    size_t want = bytes < 4096 ? 4096 : bytes + bytes / 4;
    cudaError_t err = cudaHostAlloc(&b.ptr, want, cudaHostAllocDefault);
    if (err != cudaSuccess) { b.ptr = nullptr; fail(TSS_E_CUDA, "cudaHostAlloc(%zu) failed: %s", want, cudaGetErrorString(err)); return nullptr; }
    b.cap = want;
    b.pinned = true;
    return b.ptr;
}

struct tss_search {
    tss_engine* e = nullptr;
    int w = 0, h = 0;
    std::vector<uint8_t> grid;
    int n_chains = 0, n_groups = 1, chains_per_terrain = 0;
    uint32_t chain_offset = 0;
    uint64_t seed = 0;
    int noise = tss::sls::DEFAULT_NOISE_PCT;
    uint32_t* rows_dev = nullptr;
    uint2* tabs_dev = nullptr;
    tss::sls::ChainState* states = nullptr;
    uint32_t* site_lists = nullptr;            // [16*26][n_chains rounded to 32] support lists of the thread-per-chain kernel (allocated on first use)
    int kernel = TSS_KERNEL_AUTO;              // tss_search_params.kernel
    unsigned long long* totals_dev = nullptr;  // [3]: candidates scored, steps, flips (supports added + removed)
    unsigned int* ticket_dev = nullptr;        // CTAs finished in a fused one-shot launch (sls_h16.cu OneShot), 0 between launches
    uint32_t* oneshot_host = nullptr;          // mapped pinned [48]: result block of a fused one-shot launch
    uint32_t* oneshot_host_dev = nullptr;      // ... its device-side address
    uint32_t* witness_dev = nullptr;           // [34] rows + check of the best layout (witness_kernel)
    uint32_t* witness_host = nullptr;          // pinned copy
    unsigned long long* reduce_key_dev = nullptr;  // [1] running (best << 32 | chain) minimum of the wide best-reduce, ~0 between epochs
    int2* best_dev = nullptr;                  // [n_groups]
    int* bounds_dev = nullptr;                 // [n_groups]
    int2* best_host = nullptr;                 // pinned [n_groups]
    unsigned long long* totals_host = nullptr; // pinned [3]
    unsigned long long totals_seen[3] = {0, 0, 0};
    bool dirty = false;
    bool timed = false;                        // ev0 / ev1 bracket an epoch of this search
    bool share = false;                        // all-reduce-min the bound over the engine's communicator after every epoch
    int cap_terrains = 0, cap_chains = 0;      // allocated capacity of a batch workspace (tss_solve_batch reuses it)
    tss::LnsSearch* lns = nullptr;             // grids larger than 32x32: window decomposition (lns.cu)
    tss::LnspSearch* lnsp = nullptr;           // ... with TSS_KERNEL_WINDOW_PLACEMENTS: over placements (lns_placements.cu, keys_dev / costs_dev below)
    int external_bound = tss::sls::NO_BOUND;
    // platform sets beyond {1x1} on grids up to 32x32: placement search (sls_multi.cu)
    bool multi = false;
    std::vector<int2> key_dims;                // effective (w, h) per dims key: defs order, unflipped then flipped
    std::vector<tss_platform> key_proto;       // def dims + rotated flag per key
    std::vector<int> key_costs;                // objective cost per key: 1 = platform count; GUI weights via tss_search_set_weights
    int2* keys_dev = nullptr;
    int* costs_dev = nullptr;                  // [4][MAX_KEYS]: costs | keys by area | class mask per key | limit per class
    int n_classes = 0;                         // per-type limits (tss_search_set_card_limits): classes in costs_dev; 0 = none
    bool started = false;                      // tss_search_run was called
    void* mstates = nullptr;
    // in-stream witness of one-shot solves: codes u16[1024], (x, y, w, h) records, misc = offsets[2] + evaluator result[4]
    std::vector<tss_platform> greedy_plats;    // grids > 32x32, platform sets beyond {1x1}: the greedy placement cover (computed once, it only depends on the terrain)
    bool greedy_done = false;
    uint16_t* mw_codes_dev = nullptr;
    int4* mw_plats_dev = nullptr;
    uint32_t* mw_misc_dev = nullptr;
    uint16_t* mw_codes_host = nullptr;         // pinned
    uint32_t* mw_misc_host = nullptr;          // pinned [8]
};

using namespace tss;

static double now_ms() {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

namespace tss {
static std::mutex g_engines_mutex;
static std::vector<const tss_engine*> g_engines;   // live engines
bool engine_alive(const tss_engine* e) {
    std::lock_guard<std::mutex> lock(g_engines_mutex);
    return std::find(g_engines.begin(), g_engines.end(), e) != g_engines.end();
}
}  // namespace tss

extern "C" {

int tss_version(void) { return TSS_VERSION; }

int tss_debug_smem_violations(void) { return sls_t16_checked_build() ? sls_t16_smem_violations() + sls_p16_smem_violations() : -1; }

int tss_engine_create(int device, tss_engine** out) {
    if (!out) return TSS_E_INVALID;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return TSS_E_CUDA;  // no CPU fallback
    if (device < 0) { if (cudaGetDevice(&device) != cudaSuccess) return TSS_E_CUDA; }
    if (device >= count) return TSS_E_INVALID;
    if (cudaSetDevice(device) != cudaSuccess) return TSS_E_CUDA;
    tss_engine* e = new (std::nothrow) tss_engine();
    if (!e) return TSS_E_INVALID;
    e->device = device;
    e->stats.best_count = -1;
    bool ok = cudaGetDeviceProperties(&e->prop, device) == cudaSuccess && cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreate(&e->ev0) == cudaSuccess && cudaEventCreate(&e->ev1) == cudaSuccess &&
              cudaEventCreate(&e->ev2) == cudaSuccess && cudaEventCreate(&e->ev3) == cudaSuccess;
    void* flag = nullptr;
    ok = ok && cudaHostAlloc(&flag, 2 * sizeof(int), cudaHostAllocDefault) == cudaSuccess;
    if (ok) {
        e->interrupt_host = (volatile int*)flag;
        e->interrupt_host[0] = 0;
        e->interrupt_host[1] = 1;
        ok = cudaMalloc((void**)&e->interrupt_dev, sizeof(int)) == cudaSuccess && cudaMemset(e->interrupt_dev, 0, sizeof(int)) == cudaSuccess &&
             cudaStreamCreateWithFlags(&e->irq_stream, cudaStreamNonBlocking) == cudaSuccess;
    }
    if (ok) {   // the engine's own pool for stream-ordered allocations; freed blocks stay cached (release threshold = everything)
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        uint64_t keep = ~0ull;
        if (cudaMemPoolCreate(&e->pool, &props) != cudaSuccess || cudaMemPoolSetAttribute(e->pool, cudaMemPoolAttrReleaseThreshold, &keep) != cudaSuccess) {
            cudaGetLastError();
            if (e->pool) { cudaMemPoolDestroy(e->pool); e->pool = nullptr; }   // (cudaMallocAsync from the device's default pool then)
        }
    }
    if (!ok) { cudaGetLastError(); tss_engine_destroy(e); return TSS_E_CUDA; }
    e->stream = e->own_stream;
    { std::lock_guard<std::mutex> lock(tss::g_engines_mutex); tss::g_engines.push_back(e); }
    *out = e;
    return TSS_OK;
}

static void search_free(tss_search* s);

void tss_engine_destroy(tss_engine* e) {
    if (!e) return;
    { std::lock_guard<std::mutex> lock(tss::g_engines_mutex); tss::g_engines.erase(std::remove(tss::g_engines.begin(), tss::g_engines.end(), e), tss::g_engines.end()); }
    cudaSetDevice(e->device);
    if (e->own_stream) cudaStreamSynchronize(e->own_stream);
    if (e->cached_search) { search_free(e->cached_search); e->cached_search = nullptr; }
    if (e->cached_batch) { search_free(e->cached_batch); e->cached_batch = nullptr; }
    if (e->cached_multi) { search_free(e->cached_multi); e->cached_multi = nullptr; }
    if (e->comm) { comm_destroy(e->comm); e->comm = nullptr; }
    for (auto& b : e->scratch) if (b.ptr) cudaFree(b.ptr);
    for (auto& b : e->staging) if (b.ptr) cudaFreeHost(b.ptr);
    if (e->irq_stream) { cudaStreamSynchronize(e->irq_stream); cudaStreamDestroy(e->irq_stream); }
    if (e->interrupt_dev) cudaFree(e->interrupt_dev);
    if (e->interrupt_host) cudaFreeHost((void*)e->interrupt_host);
    if (e->ev0) cudaEventDestroy(e->ev0);
    if (e->ev2) cudaEventDestroy(e->ev2);
    if (e->ev3) cudaEventDestroy(e->ev3);
    if (e->ev1) cudaEventDestroy(e->ev1);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    if (e->pool) cudaMemPoolDestroy(e->pool);   // (blocks of CNF handles that outlive the engine stay valid until they are freed, CUDA defers the release)
    delete e;
}

int tss_engine_set_stream(tss_engine* e, void* cuda_stream) {
    if (!e) return TSS_E_INVALID;
    cudaStreamSynchronize(e->stream);
    e->stream = cuda_stream ? (cudaStream_t)cuda_stream : e->own_stream;
    return TSS_OK;
}

const char* tss_last_error(const tss_engine* e) { return e ? e->error.c_str() : "null engine"; }

void tss_interrupt(tss_engine* e) {
    if (!e) return;
    e->interrupt_flag.store(1);  // host loops (epochs, propagation rounds) see this at once
    if (e->interrupt_dev && e->irq_stream) {  // running kernels see the device flag at their next poll
        int cur = -1;
        cudaGetDevice(&cur);  // callable from any thread: that thread's current device may be another GPU
        if (cur != e->device) cudaSetDevice(e->device);
        cudaMemcpyAsync(e->interrupt_dev, (const void*)(e->interrupt_host + 1), sizeof(int), cudaMemcpyHostToDevice, e->irq_stream);
        if (cur >= 0 && cur != e->device) cudaSetDevice(cur);
    }
}
void tss_clear_interrupt(tss_engine* e) {
    if (!e) return;
    e->interrupt_flag.store(0);
    if (e->interrupt_dev && e->irq_stream) {
        cudaMemcpyAsync(e->interrupt_dev, (const void*)e->interrupt_host, sizeof(int), cudaMemcpyHostToDevice, e->irq_stream);
        cudaStreamSynchronize(e->irq_stream);
    }
}
int tss_get_stats(const tss_engine* e, tss_stats* out) {
    if (!e || !out) return TSS_E_INVALID;
    *out = e->stats;
    return TSS_OK;
}
int tss_device_info(const tss_engine* e, char* name, int cap, int* sm_count, int* clock_khz) {
    if (!e) return TSS_E_INVALID;
    if (name && cap > 0) { std::strncpy(name, e->prop.name, (size_t)cap - 1); name[cap - 1] = 0; }
    if (sm_count) *sm_count = e->prop.multiProcessorCount;
    if (clock_khz) { int khz = 0; cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, e->device); *clock_khz = khz; }
    return TSS_OK;
}

size_t tss_compact_row_bytes(int32_t w, int32_t h) { return tss_row_bytes(w, h); }
size_t tss_compact_layout_bytes(int32_t w, int32_t h) { return tss_layout_bytes(w, h); }

// ------------------------------------------------------------------------------------------------ kernel (a)
int tss_eval_compact_dev(tss_engine* e, const void* grid_dev, int32_t w, int32_t h, const void* layouts_dev, int64_t n,
                         int32_t per_layout_terrain, int32_t* out_dev) {
    if (!e) return TSS_E_INVALID;
    if (!grid_dev || !layouts_dev || !out_dev || w <= 0 || h <= 0 || n < 0) return e->fail(TSS_E_INVALID, "tss_eval_compact_dev: bad arguments");
    TSS_CUDA(e, cudaSetDevice(e->device));
    return launch_eval_compact(e, grid_dev, w, h, layouts_dev, n, per_layout_terrain != 0, out_dev);
}

// shared tail: evaluate n compact layouts already on the device (scratch slot 1) against one terrain, copy results out
static int eval_compact_and_fetch(tss_engine* e, const uint8_t* grid_compact_host, int w, int h, const void* layouts_dev, int64_t n,
                                  int32_t* out_uncovered, int32_t* out_count) {
    size_t lb = tss_layout_bytes(w, h);
    void* g = e->dev(2, lb);
    int32_t* out = (int32_t*)e->dev(3, sizeof(int32_t) * 2 * (size_t)n);
    int32_t* host = (int32_t*)e->pin(1, sizeof(int32_t) * 2 * (size_t)n);
    if (!g || !out || !host) return TSS_E_CUDA;
    TSS_CUDA(e, cudaMemcpyAsync(g, grid_compact_host, lb, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    int rc = launch_eval_compact(e, g, w, h, layouts_dev, n, false, out);
    if (rc) return rc;
    TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(host, out, sizeof(int32_t) * 2 * (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->stats.device_ms = ms;
    for (int64_t i = 0; i < n; i++) {
        if (out_uncovered) out_uncovered[i] = host[2 * i];
        if (out_count) out_count[i] = host[2 * i + 1];
    }
    return TSS_OK;
}

int tss_eval_sites(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const uint8_t* sites, int64_t n,
                   int32_t* out_uncovered, int32_t* out_count) {
    if (!e) return TSS_E_INVALID;
    if (!grid || (!sites && n > 0) || w <= 0 || h <= 0 || n < 0) return e->fail(TSS_E_INVALID, "tss_eval_sites: bad arguments");
    if (n == 0) return TSS_OK;
    TSS_CUDA(e, cudaSetDevice(e->device));
    size_t lb = tss_layout_bytes(w, h), tiles = (size_t)w * h;
    uint8_t* bytes = (uint8_t*)e->dev(0, tiles * (size_t)n);
    void* compact = e->dev(1, lb * (size_t)n);
    if (!bytes || !compact) return TSS_E_CUDA;
    TSS_CUDA(e, cudaMemcpyAsync(bytes, sites, tiles * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    int rc = launch_pack_bytes(e, bytes, w, h, n, compact);
    if (rc) return rc;
    std::vector<uint8_t> gc(lb);
    pack_compact_host(grid, w, h, gc.data());
    return eval_compact_and_fetch(e, gc.data(), w, h, compact, n, out_uncovered, out_count);
}

int tss_eval_packed(tss_engine* e, const uint32_t* grid_rows, int32_t w, int32_t h, const uint32_t* layouts, int64_t n,
                    int32_t* out_uncovered, int32_t* out_count) {
    if (!e) return TSS_E_INVALID;
    if (!grid_rows || (!layouts && n > 0) || w <= 0 || h <= 0 || n < 0) return e->fail(TSS_E_INVALID, "tss_eval_packed: bad arguments");
    if (n == 0) return TSS_OK;
    TSS_CUDA(e, cudaSetDevice(e->device));
    const size_t lb = tss_layout_bytes(w, h), nw = (size_t)h * ((w + 31) / 32);
    void* compact = e->dev(1, lb * (size_t)n);
    if (!compact) return TSS_E_CUDA;
    std::vector<uint8_t> gc(lb);
    rows_to_compact_host(grid_rows, w, h, gc.data());
    if (lb == nw * 4) {  // rows are already in the compact format (w > 16 or a large grid)
        TSS_CUDA(e, cudaMemcpyAsync(compact, layouts, lb * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    } else {
        uint8_t* stage = (uint8_t*)e->pin(0, lb * (size_t)n);
        if (!stage) return TSS_E_CUDA;
        for (int64_t i = 0; i < n; i++) rows_to_compact_host(layouts + (size_t)i * nw, w, h, stage + (size_t)i * lb);
        TSS_CUDA(e, cudaMemcpyAsync(compact, stage, lb * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    }
    return eval_compact_and_fetch(e, gc.data(), w, h, compact, n, out_uncovered, out_count);
}

// uploads grid rows + platforms and runs the platform evaluator; outputs stay on the device in scratch slots
//   slot 0 grid rows, 1 plats(int4), 2 offsets, 3 out(int4 per layout), 4 unsupported rows, 5 flags, 6 layers
static int eval_platforms_dev(tss_engine* e, const uint8_t* grid, int w, int h, const tss_platform* plats, const uint32_t* offsets,
                              int64_t n, bool want_rows, bool want_flags, bool want_layers) {
    const int wpr = (w + 31) / 32;
    const size_t nw = (size_t)h * wpr, np = offsets[n];
    BitGrid bg = BitGrid::from_bytes(grid, w, h);
    uint32_t* g = (uint32_t*)e->dev(0, nw * 4);
    int4* p = (int4*)e->dev(1, sizeof(int4) * (np ? np : 1));
    uint32_t* off = (uint32_t*)e->dev(2, sizeof(uint32_t) * (size_t)(n + 1));
    int32_t* out = (int32_t*)e->dev(3, sizeof(int32_t) * 4 * (size_t)n);
    uint32_t* rows = want_rows ? (uint32_t*)e->dev(4, nw * 4 * (size_t)n) : nullptr;
    uint8_t* flags = want_flags ? (uint8_t*)e->dev(5, np ? np : 1) : nullptr;
    uint32_t* layers = want_layers ? (uint32_t*)e->dev(6, nw * 16 * (size_t)n) : nullptr;
    if (!g || !p || !off || !out || (want_rows && !rows) || (want_flags && !flags) || (want_layers && !layers)) return TSS_E_CUDA;
    std::vector<int4> eff(np);
    for (size_t i = 0; i < np; i++) {
        Dims d = platform_dims(plats[i]);
        eff[i] = make_int4(plats[i].x, plats[i].y, d.w, d.h);
    }
    TSS_CUDA(e, cudaMemcpyAsync(g, bg.rows.data(), nw * 4, cudaMemcpyHostToDevice, e->stream));
    if (np) TSS_CUDA(e, cudaMemcpyAsync(p, eff.data(), sizeof(int4) * np, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(off, offsets, sizeof(uint32_t) * (size_t)(n + 1), cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    int rc = launch_eval_platforms(e, g, w, h, p, off, n, out, rows, flags, layers);
    if (rc) return rc;
    TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));  // eff / bg are host temporaries
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->stats.device_ms = ms;
    return TSS_OK;
}

// ONE layout, everything a caller wants back, one synchronisation: inputs staged in pinned memory (slot 4), results copied
// asynchronously into pinned memory (slot 5).  The generic path above costs a blocking cudaMemcpy per result array — 45-65 us per
// call for `validate` and the witness's support layers, which the bound-tightening loop pays every iteration (TSS_TRACE).
struct OneLayout { const int32_t* res; const uint32_t* rows; const uint32_t* layers; const uint8_t* flags; };
static int eval_one_layout(tss_engine* e, const uint8_t* grid, int w, int h, const tss_platform* plats, int n_plats, bool want_rows, bool want_flags,
                           bool want_layers, OneLayout& out) {
    const int wpr = (w + 31) / 32;
    const size_t nw = (size_t)h * wpr, np = (size_t)n_plats;
    uint32_t* g = (uint32_t*)e->dev(0, nw * 4);
    int4* p = (int4*)e->dev(1, sizeof(int4) * (np ? np : 1));
    uint32_t* off = (uint32_t*)e->dev(2, sizeof(uint32_t) * 2);
    int32_t* res = (int32_t*)e->dev(3, sizeof(int32_t) * 4);
    uint32_t* rows = want_rows ? (uint32_t*)e->dev(4, nw * 4) : nullptr;
    uint8_t* flags = want_flags ? (uint8_t*)e->dev(5, np ? np : 1) : nullptr;
    uint32_t* layers = want_layers ? (uint32_t*)e->dev(6, nw * 16) : nullptr;
    const size_t in_bytes = sizeof(int4) * np + 4 * nw + 8, out_bytes = 16 + 4 * nw + 16 * nw + np + 16;
    char* in = (char*)e->pin(4, in_bytes);
    char* ho = (char*)e->pin(5, out_bytes);
    if (!g || !p || !off || !res || (want_rows && !rows) || (want_flags && !flags) || (want_layers && !layers) || !in || !ho) return TSS_E_CUDA;
    int4* in_p = (int4*)in;
    uint32_t* in_g = (uint32_t*)(in + sizeof(int4) * np);
    uint32_t* in_off = in_g + nw;
    for (size_t i = 0; i < np; i++) {
        const Dims d = platform_dims(plats[i]);
        in_p[i] = make_int4(plats[i].x, plats[i].y, d.w, d.h);
    }
    std::memset(in_g, 0, 4 * nw);
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            if (grid[(size_t)y * w + x]) in_g[(size_t)y * wpr + (x >> 5)] |= 1u << (x & 31);
    in_off[0] = 0; in_off[1] = (uint32_t)np;
    if (np) TSS_CUDA(e, cudaMemcpyAsync(p, in_p, sizeof(int4) * np, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(g, in_g, 4 * nw, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(off, in_off, 8, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    int rc = launch_eval_platforms(e, g, w, h, p, off, 1, res, rows, flags, layers);
    if (rc) return rc;
    TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    int32_t* ho_res = (int32_t*)ho;
    uint32_t* ho_rows = (uint32_t*)(ho + 16);
    uint32_t* ho_layers = ho_rows + nw;
    uint8_t* ho_flags = (uint8_t*)(ho_layers + 4 * nw);
    TSS_CUDA(e, cudaMemcpyAsync(ho_res, res, 16, cudaMemcpyDeviceToHost, e->stream));
    if (want_rows) TSS_CUDA(e, cudaMemcpyAsync(ho_rows, rows, 4 * nw, cudaMemcpyDeviceToHost, e->stream));
    if (want_layers) TSS_CUDA(e, cudaMemcpyAsync(ho_layers, layers, 16 * nw, cudaMemcpyDeviceToHost, e->stream));
    if (want_flags && np) TSS_CUDA(e, cudaMemcpyAsync(ho_flags, flags, np, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e->ev0, e->ev1);
    e->stats.device_ms = ms;
    out = OneLayout{ho_res, ho_rows, ho_layers, ho_flags};
    return TSS_OK;
}

int tss_eval_platforms(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_platform* plats,
                       const uint32_t* offsets, int64_t n, int32_t* out) {
    if (!e) return TSS_E_INVALID;
    if (!grid || !offsets || !out || w <= 0 || h <= 0 || n < 0 || (!plats && offsets[n] > 0)) return e->fail(TSS_E_INVALID, "tss_eval_platforms: bad arguments");
    if (n == 0) return TSS_OK;
    TSS_CUDA(e, cudaSetDevice(e->device));
    int rc = eval_platforms_dev(e, grid, w, h, plats, offsets, n, false, false, false);
    if (rc) return rc;
    TSS_CUDA(e, cudaMemcpy(out, e->scratch[3].ptr, sizeof(int32_t) * 4 * (size_t)n, cudaMemcpyDeviceToHost));
    return TSS_OK;
}

int tss_validate(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_platform* plats, int32_t n,
                 uint8_t* out_unsupported, uint8_t* out_flags) {
    if (!e) return TSS_E_INVALID;
    if (!grid || w <= 0 || h <= 0 || n < 0 || (!plats && n > 0)) return e->fail(TSS_E_INVALID, "tss_validate: bad arguments");
    TSS_CUDA(e, cudaSetDevice(e->device));
    OneLayout r;
    int rc = eval_one_layout(e, grid, w, h, plats, n, true, true, false, r);
    if (rc) return rc;
    const int wpr = (w + 31) / 32;
    const uint32_t* rows = r.rows;
    const int32_t* res = r.res;
    if (out_flags && n > 0) std::memcpy(out_flags, r.flags, (size_t)n);
    if (out_unsupported)
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) out_unsupported[(size_t)y * w + x] = (rows[(size_t)y * wpr + (x >> 5)] >> (x & 31)) & 1u;
    return res[0];
}

// declared in tss.h next to the encoder; needs the evaluator's support layers
int tss_layout_to_assignment_impl(tss_engine* e, const Encoding& enc, const uint8_t* grid, const tss_platform* plats, int32_t n_plats,
                                  uint8_t* assignment) {
    TSS_CUDA(e, cudaSetDevice(e->device));
    const int w = enc.w, h = enc.h, wpr = (w + 31) / 32, K = enc.K();
    OneLayout r;
    int rc = eval_one_layout(e, grid, w, h, plats, n_plats, false, false, true, r);
    if (rc) return rc;
    const uint32_t* layers = r.layers;
    for (int v = 0; v <= enc.base.n_vars; v++) assignment[v] = v == 0 ? 2 : 0;
    for (int i = 0; i < n_plats; i++) {  // every dims key contained in the platform's effective dims (DAG implications)
        if (plats[i].x < 0 || plats[i].y < 0 || plats[i].x >= w || plats[i].y >= h) continue;
        Dims d = platform_dims(plats[i]);
        int tile = plats[i].y * w + plats[i].x;
        for (int k = 0; k < K; k++)
            if (dims_le(enc.keys[k], d)) assignment[enc.plat_var[(size_t)tile * K + k]] = 1;
    }
    for (int t = 0; t < w * h; t++)
        for (int l = 0; l < 4; l++) {
            int var = enc.terr_var[(size_t)t * 4 + l];
            if (!var) continue;
            int x = t % w, y = t / w;
            const uint32_t* plane = layers + (size_t)(3 - l) * h * wpr;  // T3 = directly supported ... T0 = after 3 rounds
            assignment[var] = (plane[(size_t)y * wpr + (x >> 5)] >> (x & 31)) & 1u;
        }
    return TSS_OK;
}

// ------------------------------------------------------------------------------------------------ kernel (b)
static void search_free(tss_search* s) {
    if (!s) return;
    if (s->lns) lns_destroy(s->lns);
    if (s->lnsp) lnsp_destroy(s->lnsp);
    cudaFree(s->keys_dev);
    cudaFree(s->costs_dev);
    cudaFree(s->mstates);
    cudaFree(s->mw_codes_dev); cudaFree(s->mw_plats_dev); cudaFree(s->mw_misc_dev);
    if (s->mw_codes_host) cudaFreeHost(s->mw_codes_host);
    if (s->mw_misc_host) cudaFreeHost(s->mw_misc_host);
    cudaFree(s->site_lists);
    cudaFree(s->reduce_key_dev);
    cudaFree(s->witness_dev);
    cudaFree(s->ticket_dev);
    if (s->oneshot_host) cudaFreeHost(s->oneshot_host);
    if (s->witness_host) cudaFreeHost(s->witness_host);
    cudaFree(s->rows_dev); cudaFree(s->tabs_dev); cudaFree(s->states); cudaFree(s->totals_dev); cudaFree(s->best_dev); cudaFree(s->bounds_dev);
    if (s->best_host) cudaFreeHost(s->best_host);
    if (s->totals_host) cudaFreeHost(s->totals_host);
    delete s;
}

// rows32_host: [n_terrains][32]
static int search_alloc(tss_engine* e, tss_search* s, const uint32_t* rows32_host, int n_terrains) {
    TSS_CUDA(e, cudaMalloc(&s->rows_dev, sizeof(uint32_t) * 32 * (size_t)n_terrains));
    TSS_CUDA(e, cudaMalloc(&s->tabs_dev, sizeof(uint2) * 1024 * (size_t)n_terrains));
    TSS_CUDA(e, cudaMalloc(&s->states, sizeof(sls::ChainState) * (size_t)s->n_chains));
    TSS_CUDA(e, cudaMalloc(&s->totals_dev, sizeof(unsigned long long) * 3));
    TSS_CUDA(e, cudaMalloc(&s->reduce_key_dev, sizeof(unsigned long long)));
    TSS_CUDA(e, cudaMalloc(&s->witness_dev, sizeof(uint32_t) * 34));
    TSS_CUDA(e, cudaMalloc(&s->ticket_dev, sizeof(unsigned int)));
    TSS_CUDA(e, cudaMemsetAsync(s->ticket_dev, 0, sizeof(unsigned int), e->stream));
    TSS_CUDA(e, cudaHostAlloc((void**)&s->oneshot_host, sizeof(uint32_t) * 48, cudaHostAllocMapped));
    TSS_CUDA(e, cudaHostGetDevicePointer((void**)&s->oneshot_host_dev, s->oneshot_host, 0));
    TSS_CUDA(e, cudaHostAlloc((void**)&s->witness_host, sizeof(uint32_t) * 34, cudaHostAllocDefault));
    TSS_CUDA(e, cudaMalloc(&s->best_dev, sizeof(int2) * (size_t)s->n_groups));
    TSS_CUDA(e, cudaMalloc(&s->bounds_dev, sizeof(int) * (size_t)s->n_groups));
    TSS_CUDA(e, cudaHostAlloc((void**)&s->best_host, sizeof(int2) * (size_t)s->n_groups, cudaHostAllocDefault));
    TSS_CUDA(e, cudaHostAlloc((void**)&s->totals_host, sizeof(unsigned long long) * 3, cudaHostAllocDefault));
    if (rows32_host) TSS_CUDA(e, cudaMemcpyAsync(s->rows_dev, rows32_host, sizeof(uint32_t) * 32 * (size_t)n_terrains, cudaMemcpyHostToDevice, e->stream));
    return TSS_OK;
}

// the placement search's buffers (sls_multi.cu) for one terrain and s->n_chains chains
static cudaError_t multi_alloc(tss_engine* e, tss_search* s) {
    cudaError_t err = cudaMalloc(&s->rows_dev, sizeof(uint32_t) * 32);
    if (err == cudaSuccess) err = cudaMalloc(&s->keys_dev, sizeof(int2) * (size_t)slsm_max_keys());
    if (err == cudaSuccess) err = cudaMalloc(&s->costs_dev, sizeof(int) * 4 * (size_t)slsm_max_keys());   // costs | keys by area | limit classes
    if (err == cudaSuccess) err = cudaMalloc(&s->mstates, slsm_state_bytes() * (size_t)s->n_chains);
    if (err == cudaSuccess) err = cudaMalloc(&s->totals_dev, sizeof(unsigned long long) * 3);
    if (err == cudaSuccess) err = cudaMalloc(&s->best_dev, sizeof(int2));
    if (err == cudaSuccess) err = cudaMalloc(&s->bounds_dev, sizeof(int));
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->best_host, sizeof(int2), cudaHostAllocDefault);
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->totals_host, sizeof(unsigned long long) * 3, cudaHostAllocDefault);
    if (err == cudaSuccess) err = cudaMalloc(&s->mw_codes_dev, sizeof(uint16_t) * (size_t)slsm_max_items());
    if (err == cudaSuccess) err = cudaMalloc(&s->mw_plats_dev, sizeof(int4) * (size_t)slsm_max_items());
    if (err == cudaSuccess) err = cudaMalloc(&s->mw_misc_dev, sizeof(uint32_t) * 8);
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->mw_codes_host, sizeof(uint16_t) * (size_t)slsm_max_items(), cudaHostAllocDefault);
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->mw_misc_host, sizeof(uint32_t) * 8, cudaHostAllocDefault);
    if (err == cudaSuccess) err = cudaMalloc(&s->reduce_key_dev, sizeof(unsigned long long));
    if (err == cudaSuccess) err = cudaMalloc(&s->ticket_dev, sizeof(unsigned int));
    if (err == cudaSuccess) err = cudaMemsetAsync(s->reduce_key_dev, 0xff, sizeof(unsigned long long), e->stream);
    if (err == cudaSuccess) err = cudaMemsetAsync(s->ticket_dev, 0, sizeof(unsigned int), e->stream);
    if (err == cudaSuccess) err = cudaHostAlloc((void**)&s->oneshot_host, sizeof(uint32_t) * (16 + (size_t)slsm_max_items() / 2), cudaHostAllocMapped);
    if (err == cudaSuccess) err = cudaHostGetDevicePointer((void**)&s->oneshot_host_dev, s->oneshot_host, 0);
    return err;
}

// a cached workspace takes the terrain of a new call: its grid and seed, the default chain offset and noise, no outside bound
static void reuse_for_terrain(tss_search* s, const uint8_t* grid, int w, int h, uint64_t seed) {
    s->w = w; s->h = h; s->seed = seed; s->chain_offset = 0; s->noise = sls::DEFAULT_NOISE_PCT;
    s->grid.assign(grid, grid + (size_t)w * h);
    s->external_bound = sls::NO_BOUND;
}

// u8 grid -> one u32 per row (w, h <= 32; rows >= h are zero), the host side of pack_rows32_kernel
static void pack_rows32(const uint8_t* grid, int w, int h, uint32_t rows[32]) {
    for (int y = 0; y < 32; y++) rows[y] = 0;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            if (grid[(size_t)y * w + x]) rows[y] |= 1u << x;
}

// A platform set every entry point takes: no empty def, and 1x1 among the defs (none at all stands for {1x1}).  `fn` names the
// caller in the message.  *only_1x1 (may be null) = every def is 1x1.
static int check_defs(tss_engine* e, const tss_dims* defs, int n_defs, const char* fn, bool* only_1x1) {
    bool has_1x1 = n_defs == 0, only = true;
    for (int i = 0; i < n_defs; i++) {
        if (defs[i].w <= 0 || defs[i].h <= 0) return e->fail(TSS_E_INVALID, "%s: empty platform dimensions", fn);
        has_1x1 = has_1x1 || (defs[i].w == 1 && defs[i].h == 1);
        only = only && defs[i].w == 1 && defs[i].h == 1;
    }
    if (!has_1x1) return e->fail(TSS_E_INVALID, "the platform set must contain 1x1 (src/encoder.rs:564-566)");
    if (only_1x1) *only_1x1 = only;
    return TSS_OK;
}

// what a platform of a key costs under GUI weights: the sum of the weights of every def contained in its def, exactly what
// PlatformLayout::total_weight charges it (platform_layout.rs:174-183); weights = (w, h, weight) records
static long key_cost(const tss_platform& proto, const int32_t* weights, int n_weights) {
    const Dims def{proto.def_w, proto.def_h};
    long cost = 0;
    for (int i = 0; i < n_weights; i++)
        if (dims_le(Dims{weights[3 * i], weights[3 * i + 1]}, def)) cost += weights[3 * i + 2];
    return cost;
}

static int search_init_device(tss_engine* e, tss_search* s, int n_terrains) {
    TSS_CUDA(e, cudaMemsetAsync(s->totals_dev, 0, sizeof(unsigned long long) * 3, e->stream));
    TSS_CUDA(e, cudaMemsetAsync(s->reduce_key_dev, 0xff, sizeof(unsigned long long), e->stream));
    bound_min_kernel<<<(s->n_groups + 255) / 256, 256, 0, e->stream>>>(s->bounds_dev, s->n_groups, sls::NO_BOUND, true);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    for (int g = 0; g < s->n_groups; g++) s->best_host[g] = make_int2(sls::NO_BOUND, -1);
    s->totals_host[0] = s->totals_host[1] = s->totals_host[2] = 0;
    int rc = sls_build_reach(e, s->rows_dev, n_terrains, s->tabs_dev);
    if (rc) return rc;
    s->dirty = true;                                      // everything here is in-stream: the first reader synchronises
    return sls_init_states(e, s->states, s->n_chains);
}

// dims keys of a platform set: both orientations of every def in defs order, unflipped first (src/encoder.rs:121-130)
static void build_keys(const tss_dims* defs, int n_defs, std::vector<int2>& key_dims, std::vector<tss_platform>& key_proto) {
    key_dims.clear();
    key_proto.clear();
    for (int i = 0; i < n_defs; i++)
        for (int rot = 0; rot < 2; rot++) {
            int2 d = rot ? make_int2(defs[i].h, defs[i].w) : make_int2(defs[i].w, defs[i].h);
            bool seen = false;
            for (auto& kd : key_dims) seen = seen || (kd.x == d.x && kd.y == d.y);
            if (seen) continue;
            key_dims.push_back(d);
            key_proto.push_back(tss_platform{0, 0, defs[i].w, defs[i].h, rot});
        }
}

// keys by area, largest first (stable): the second candidate pass of the placement search draws from the front
static std::vector<int> keys_by_area(const std::vector<int2>& key_dims) {
    std::vector<int> order(key_dims.size());
    for (size_t i = 0; i < order.size(); i++) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key_dims[a].x * key_dims[a].y > key_dims[b].x * key_dims[b].y; });
    return order;
}

// The classes of per-type platform limits (PlatformLimits.card_limits beyond 1x1), as Encoding::with_limits
// (host_model.cpp, encoder.rs:619-667) lowers them: a limit on type d counts one literal per anchor, set by the plat var of
// key d (square d) or implied by those of keys d and its transpose (rectangular d); a platform sets the plat var of every key
// contained in its dims (tss_layout_to_assignment).  So class C_d = the keys q with dims_le(k, q) for some key k in {d, d^T},
// closed under rotation, and a platform counts at most once towards it.  A record with neither d nor d^T among the keys emits
// no constraint, nor does a limit of MAX_ITEMS or more: both are vacuous and skipped.  1x1 records (the platform count, whose
// class is every key) are skipped as well: their callers treat them on their own.  Records with the same class merge into one
// with the smaller limit.  -> key_mask[k] = classes of key k (bit j = class j), class_limit[j]; at most MAX_KEYS classes.
static int card_limit_classes(const std::vector<int2>& key_dims, const int32_t* card, int n_card, std::vector<uint32_t>& key_mask,
                              std::vector<int>& class_limit) {
    key_mask.assign(key_dims.size(), 0u);
    class_limit.clear();
    std::vector<uint32_t> members;   // keys of each class (bit k)
    for (int i = 0; i < n_card; i++) {
        const int dw = card[3 * i], dh = card[3 * i + 1], lim = card[3 * i + 2];
        if (dw <= 0 || dh <= 0 || lim < 0) return TSS_E_INVALID;
        if ((dw == 1 && dh == 1) || lim >= slsm_max_items()) continue;
        uint32_t m = 0;
        for (size_t k = 0; k < key_dims.size(); k++) {
            if (!((key_dims[k].x == dw && key_dims[k].y == dh) || (key_dims[k].x == dh && key_dims[k].y == dw))) continue;
            for (size_t q = 0; q < key_dims.size(); q++)
                if (dims_le(Dims{key_dims[k].x, key_dims[k].y}, Dims{key_dims[q].x, key_dims[q].y})) m |= 1u << q;
        }
        if (!m) continue;
        const size_t j = std::find(members.begin(), members.end(), m) - members.begin();
        if (j < members.size()) { class_limit[j] = std::min(class_limit[j], lim); continue; }
        if ((int)members.size() == slsm_max_keys()) return TSS_E_UNSUPPORTED;
        members.push_back(m);
        class_limit.push_back(lim);
    }
    for (size_t j = 0; j < members.size(); j++)
        for (size_t k = 0; k < key_dims.size(); k++)
            if ((members[j] >> k) & 1u) key_mask[k] |= 1u << j;
    return TSS_OK;
}

static int window_placements_create(tss_engine* e, tss_search* s, const tss_dims* defs, int n_defs, int seeds, const int32_t* card, int n_card);

// Chains that fill the device: 32 warps per SM for the warp kernels (two chains per warp on grids of <= 16 rows),
// 3 CTAs of 128 threads per SM for the thread-per-chain kernels.
static int default_chains(const tss_engine* e, int w, int h, int kernel) {
    const bool thread_default = (sls_t16_fits(w, h) && (kernel == TSS_KERNEL_AUTO || kernel == TSS_KERNEL_THREAD)) ||
                                (sls_p16_fits(w, h) && kernel == TSS_KERNEL_PAIR);
    const int per_sm = thread_default ? 3 * sls_thread_cta_chains() : (h <= 16 ? 64 : 32);
    return e->prop.multiProcessorCount * per_sm;
}

// tss_search_create; card / n_card: per-type limit records for the window placement search (tss_search_create_with_limits)
static int search_create(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                         const tss_search_params* params, const int32_t* card, int32_t n_card, tss_search** out) {
    if (!e) return TSS_E_INVALID;
    if (!grid || !out || w <= 0 || h <= 0 || (!defs && n_defs > 0)) return e->fail(TSS_E_INVALID, "tss_search_create: bad arguments");
    if (int rc = check_defs(e, defs, n_defs, "tss_search_create", nullptr)) return rc;
    if ((size_t)h * ((w + 31) / 32) * 20 > 200 * 1024) return e->fail(TSS_E_UNSUPPORTED, "tss_search: grid %dx%d exceeds the validator's shared-memory planes", w, h);
    TSS_CUDA(e, cudaSetDevice(e->device));
    tss_search* s = new tss_search();
    s->e = e; s->w = w; s->h = h;
    s->grid.assign(grid, grid + (size_t)w * h);
    s->seed = params ? params->seed : 0;
    s->chain_offset = params ? (uint32_t)params->chain_offset : 0;
    s->noise = (params && params->noise_pct >= 0) ? params->noise_pct : sls::DEFAULT_NOISE_PCT;
    s->share = e->comm != nullptr;  // a portfolio created on an engine with a communicator shares its bound every epoch
    if (w > 32 || h > 32) {  // window decomposition: n_chains is read as chains per window (multiple of 4, default 8)
        // default: at most 16 chains per window.  A chain steps at single-warp latency (~1.1 us per step) while the schedulers have
        // spare issue slots; filling the device (56 per window on 256x256) halves the step rate (2.2 us per step) and buys nothing:
        // the count is the same plateau for 4 .. 56 chains per window (profiles/r2_c4_tradeoff.log: 77 ms against 152 ms for
        // 16 phases x 4000 steps, 4 259-4 267 against 4 258-4 268)
        const int n_win = ((w + 31) / 32 + 1) * ((h + 31) / 32 + 1);
        int fill = (e->prop.multiProcessorCount * 32 / n_win) / 4 * 4;
        fill = fill < 8 ? 8 : (fill > 16 ? 16 : fill);
        int seeds = (params && params->n_chains > 0) ? ((params->n_chains + 3) / 4) * 4 : fill;
        if (params && params->kernel == TSS_KERNEL_WINDOW_PLACEMENTS) {
            int rc = window_placements_create(e, s, defs, n_defs, seeds, card, n_card);
            if (rc != TSS_OK) { search_free(s); return rc; }
            *out = s;
            return TSS_OK;
        }
        int rc = lns_create(e, grid, w, h, seeds, s->seed, s->chain_offset, s->noise, &s->lns);
        if (rc != TSS_OK) { delete s; return rc; }
        build_keys(defs, n_defs, s->key_dims, s->key_proto);   // (platform sets beyond {1x1}: the 1x1 layout is merged afterwards, merge_supports)
        s->n_chains = lns_chains(s->lns);
        *out = s;
        return TSS_OK;
    }
    // default: 32 warps per SM (8 CTAs of 4 warps); grids of <= 16 rows run two chains per warp
    // (thread-per-chain kernel: 3 CTAs of 128 chains per SM)
    s->kernel = params ? params->kernel : TSS_KERNEL_AUTO;
    if (s->kernel < TSS_KERNEL_AUTO || s->kernel > TSS_KERNEL_PAIR || (s->kernel == TSS_KERNEL_HALF_WARP && h > 16) ||
        (s->kernel == TSS_KERNEL_THREAD && !sls_t16_fits(w, h)) || (s->kernel == TSS_KERNEL_PAIR && !sls_p16_fits(w, h))) {
        int k = s->kernel;
        delete s;
        if (k == TSS_KERNEL_WINDOW_PLACEMENTS)
            return e->fail(TSS_E_UNSUPPORTED, "tss_search_create: the window placement search needs a grid wider or taller than 32 (got %dx%d)", w, h);
        return e->fail(TSS_E_UNSUPPORTED, "tss_search_create: kernel variant %d does not support a %dx%d grid", k, w, h);
    }
    s->n_chains = (params && params->n_chains > 0) ? params->n_chains : default_chains(e, w, h, s->kernel);
    s->n_groups = 1;
    s->chains_per_terrain = 0;
    uint32_t rows[32];
    pack_rows32(grid, w, h, rows);
    // more than the single 1x1 key -> placement search
    build_keys(defs, n_defs, s->key_dims, s->key_proto);
    bool fits = (int)s->key_dims.size() <= slsm_max_keys();
    for (auto& kd : s->key_dims) fits = fits && kd.x <= 6 && kd.y <= 6;
    if (s->key_dims.size() > 1 && fits) {
        s->multi = true;
        if (!(params && params->n_chains > 0)) s->n_chains = e->prop.multiProcessorCount * 16;
        cudaError_t err = cudaSuccess;
        tss_search* c = e->cached_multi;
        if (c && c->n_chains == s->n_chains) {
            // the workspace of an earlier one-shot solve: its buffers (no allocation) with the host state of this call.  (What is
            // not reset here — n_groups, chains_per_terrain, the 1x1 and window buffers — is the same in every placement search.)
            e->cached_multi = nullptr;
            reuse_for_terrain(c, grid, w, h, s->seed);
            c->chain_offset = s->chain_offset; c->noise = s->noise; c->share = s->share; c->kernel = s->kernel;
            c->key_dims.swap(s->key_dims);
            c->key_proto.swap(s->key_proto);
            c->started = c->timed = c->dirty = false;
            c->n_classes = 0;
            c->greedy_plats.clear();
            c->greedy_done = false;
            delete s;
            s = c;
        } else {
            err = multi_alloc(e, s);
        }
        s->key_costs.assign(s->key_dims.size(), 1);
        s->totals_seen[0] = s->totals_seen[1] = s->totals_seen[2] = 0;
        const int nb = sls::NO_BOUND;
        if (err == cudaSuccess) err = cudaMemcpyAsync(s->rows_dev, rows, sizeof rows, cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) err = cudaMemcpyAsync(s->keys_dev, s->key_dims.data(), sizeof(int2) * s->key_dims.size(), cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) err = cudaMemcpyAsync(s->costs_dev, s->key_costs.data(), sizeof(int) * s->key_costs.size(), cudaMemcpyHostToDevice, e->stream);
        const std::vector<int> order = keys_by_area(s->key_dims);
        if (err == cudaSuccess) err = cudaMemcpyAsync(s->costs_dev + slsm_max_keys(), order.data(), sizeof(int) * order.size(), cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) err = cudaMemcpyAsync(s->bounds_dev, &nb, sizeof nb, cudaMemcpyHostToDevice, e->stream);
        if (err == cudaSuccess) err = cudaMemsetAsync(s->totals_dev, 0, sizeof(unsigned long long) * 3, e->stream);
        int rc = err == cudaSuccess ? slsm_init(e, s->mstates, s->n_chains) : e->fail(TSS_E_CUDA, "tss_search_create: %s", cudaGetErrorString(err));
        if (rc == TSS_OK && cudaStreamSynchronize(e->stream) != cudaSuccess) rc = e->fail(TSS_E_CUDA, "tss_search_create: stream sync failed");
        if (rc != TSS_OK) { search_free(s); return rc; }
        s->best_host[0] = make_int2(sls::NO_BOUND, -1);
        s->totals_host[0] = s->totals_host[1] = s->totals_host[2] = 0;
        *out = s;
        return TSS_OK;
    }
    int rc = search_alloc(e, s, rows, 1);
    if (rc == TSS_OK) rc = search_init_device(e, s, 1);
    if (rc != TSS_OK) { search_free(s); return rc; }
    *out = s;
    return TSS_OK;
}

int tss_search_create(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                      const tss_search_params* params, tss_search** out) {
    return search_create(e, grid, w, h, defs, n_defs, params, nullptr, 0, out);
}

int tss_search_create_with_limits(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, const int32_t* card,
                                  int32_t n_card, const tss_search_params* params, tss_search** out) {
    if (!e) return TSS_E_INVALID;
    if (!grid || !out || w <= 0 || h <= 0 || (!defs && n_defs > 0) || n_card < 0 || (n_card > 0 && !card))
        return e->fail(TSS_E_INVALID, "tss_search_create_with_limits: bad arguments");
    if (int rc = check_defs(e, defs, n_defs, "tss_search_create_with_limits", nullptr)) return rc;
    for (int i = 0; i < n_card; i++) {
        if (card[3 * i] == 1 && card[3 * i + 1] == 1)
            return e->fail(TSS_E_INVALID, "tss_search_create_with_limits: the platform count (1x1) is the search's bound, not a per-type limit");
        if (card[3 * i + 2] < 0) return e->fail(TSS_E_INVALID, "tss_search_create_with_limits: negative limit for %dx%d", card[3 * i], card[3 * i + 1]);
    }
    if (w <= 32 && h <= 32) {
        int rc = tss_search_create(e, grid, w, h, defs, n_defs, params, out);
        if (rc == TSS_OK && (rc = tss_search_set_card_limits(*out, card, n_card)) != TSS_OK) {
            tss_search_destroy(*out);
            *out = nullptr;
        }
        return rc;
    }
    std::vector<int2> kd;
    std::vector<tss_platform> kp;
    std::vector<uint32_t> mask;
    std::vector<int> lim;
    build_keys(defs, n_defs, kd, kp);
    int rc = card_limit_classes(kd, card, n_card, mask, lim);
    if (rc) return e->fail(rc, "tss_search_create_with_limits: bad limit records");
    if (lim.empty()) return tss_search_create(e, grid, w, h, defs, n_defs, params, out);   // every record vacuous
    // the limits are fixed here because the window placement search's start layout depends on them
    tss_search_params p = params ? *params : tss_search_params{0, 0, 0, -1, TSS_KERNEL_AUTO};
    if (p.kernel != TSS_KERNEL_AUTO && p.kernel != TSS_KERNEL_WINDOW_PLACEMENTS)
        return e->fail(TSS_E_UNSUPPORTED, "tss_search_create_with_limits: per-type limits on a %dx%d grid need the window placement search (kernel %d)", w, h, p.kernel);
    p.kernel = TSS_KERNEL_WINDOW_PLACEMENTS;
    return search_create(e, grid, w, h, defs, n_defs, &p, card, n_card, out);
}

void tss_search_destroy(tss_search* s) {
    if (!s) return;
    cudaSetDevice(s->e->device);
    cudaStreamSynchronize(s->e->stream);
    search_free(s);
}

int tss_search_n_chains(const tss_search* s) { return s ? s->n_chains : TSS_E_INVALID; }

void tss_sls_spec_probe(uint32_t* out) {
    if (!out) return;
    out[0] = sls::K1; out[1] = sls::K2; out[2] = sls::noise_q7(20); out[3] = sls::tie_remove(0x12345678u, 3) + 1000u * (uint32_t)(sls::tenure_of(0) + 2 * sls::tenure_of(1) + 3 * sls::tenure_of(2) + 4 * sls::tenure_of(3)) +
             (sls::is_tabu(70000u, sls::stamp_reset(70000u), 20) ? 1u : 0u) + (sls::is_tabu(65540u, (uint16_t)65530u, 12) ? 2u : 0u) +
             100000u * (uint32_t)(sls::effective_tenure(20, 14) + sls::effective_tenure(3, 100) + sls::effective_tenure(6, 2)); out[4] = sls::tie_add(0x12345678u, 7u);
    out[5] = sls::step_hash(1u, 2u); out[6] = sls::tie_remove(3u, 40u) ^ sls::K3; out[7] = sls::chain_base(0x0123456789abcdefull, 5u); out[8] = sls::NO_BOUND;
}

// Which of the four equivalent SLS kernels (same spec, same trajectories) advances this portfolio.
static int search_kernel(const tss_search* s) {
    const int cpt = s->chains_per_terrain;
    const bool t16_ok = sls_t16_fits(s->w, s->h) && (cpt == 0 || cpt % sls_thread_cta_chains() == 0);
    const bool p16_ok = sls_p16_fits(s->w, s->h) && (cpt == 0 || cpt % sls_thread_cta_chains() == 0);
    const bool h16_ok = s->h <= 16 && (cpt == 0 || cpt % 8 == 0);
    if (s->kernel == TSS_KERNEL_PAIR && p16_ok) return TSS_KERNEL_PAIR;
    if (s->kernel == TSS_KERNEL_THREAD && t16_ok) return TSS_KERNEL_THREAD;
    if (s->kernel == TSS_KERNEL_WARP) return TSS_KERNEL_WARP;
    if (s->kernel == TSS_KERNEL_HALF_WARP && h16_ok) return TSS_KERNEL_HALF_WARP;
    // auto: a chain per thread pays off once the device is well filled — a thread-kernel warp steps its 32 chains in
    // ~2.4 us whatever the load, the half-warp kernel steps few chains in ~1.1 us (measured on rect 16x16,
    // profiles/crossover.py: equal at ~7000 chains; 2048 chains 48 vs 25 ms, 16384 chains 49 vs 102 ms per 20000 steps)
    // (grids of at most 16x16: two grid rows per word issue fewer instructions per chain step than one row per word; rect
    // 16x16, 56 832 chains: 30.3 against 24.7 G flips/s, profiles/r3_bench_alternation.jsonl)
    if (s->kernel == TSS_KERNEL_AUTO && p16_ok && s->n_chains >= s->e->prop.multiProcessorCount * 48) return TSS_KERNEL_PAIR;
    if (s->kernel == TSS_KERNEL_AUTO && t16_ok && s->n_chains >= s->e->prop.multiProcessorCount * 48) return TSS_KERNEL_THREAD;
    return h16_ok ? TSS_KERNEL_HALF_WARP : TSS_KERNEL_WARP;
}

int tss_search_kernel(const tss_search* s) {
    return !s ? TSS_E_INVALID : (s->lnsp ? TSS_KERNEL_WINDOW_PLACEMENTS : ((s->lns || s->multi) ? 0 : search_kernel(s)));
}

int tss_search_run(tss_search* s, int64_t steps, int32_t target_count) {
    if (!s) return TSS_E_INVALID;
    tss_engine* e = s->e;
    if (steps <= 0) return e->fail(TSS_E_INVALID, "tss_search_run: steps must be positive");
    TSS_CUDA(e, cudaSetDevice(e->device));
    s->started = true;
    TSS_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    if (s->lns || s->lnsp) {  // one phase of the window decomposition (a phase is one epoch per window: at most MAX_EPOCH_STEPS, see below)
        for (long long left = steps; left > 0; left -= sls::MAX_EPOCH_STEPS) {
            const long long chunk = left < sls::MAX_EPOCH_STEPS ? left : sls::MAX_EPOCH_STEPS;
            int rc = s->lns ? lns_phase(e, s->lns, chunk, s->share) : lnsp_phase(e, s->lnsp, chunk);
            if (rc) return rc;
        }
        TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
        s->dirty = true;
        s->timed = true;
        e->stats.n_solves++;
        return TSS_OK;
    }
    if (s->multi) {
        int rc = slsm_run(e, s->rows_dev, s->w, s->h, s->keys_dev, s->costs_dev, s->costs_dev + slsm_max_keys(), (int)s->key_dims.size(), s->mstates, s->n_chains, s->chain_offset, s->seed, steps,
                          s->bounds_dev, target_count < 0 ? -1 : target_count, s->noise, s->totals_dev, s->best_dev, s->costs_dev + 2 * slsm_max_keys(), s->n_classes);
        if (rc == TSS_OK && e->comm && s->share) rc = comm_allreduce_min(e, e->comm, s->bounds_dev, 1);
        if (rc) return rc;
        TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
        TSS_CUDA(e, cudaMemcpyAsync(s->best_host, s->best_dev, sizeof(int2), cudaMemcpyDeviceToHost, e->stream));
        TSS_CUDA(e, cudaMemcpyAsync(s->totals_host, s->totals_dev, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost, e->stream));
        s->dirty = true;
        s->timed = true;
        e->stats.n_solves++;
        return TSS_OK;
    }
    int chains_per_group = s->n_groups == 1 ? s->n_chains : s->chains_per_terrain;
    const int variant = search_kernel(s);
    if ((variant == TSS_KERNEL_THREAD || variant == TSS_KERNEL_PAIR) && !s->site_lists) TSS_CUDA(e, cudaMalloc(&s->site_lists, sizeof(uint32_t) * sls_t16_list_words(s->n_chains)));
    // an epoch is at most 32768 steps (the tabu stamps are 16 bit, sls_spec.hpp): longer runs are consecutive epochs
    for (long long left = steps; left > 0; left -= sls::MAX_EPOCH_STEPS) {
        const long long chunk = left < sls::MAX_EPOCH_STEPS ? left : sls::MAX_EPOCH_STEPS;
        const int target = target_count < 0 ? -1 : target_count;
        int rc;
        if (variant == TSS_KERNEL_PAIR)
            rc = sls_run_p16(e, s->rows_dev, s->tabs_dev, s->states, s->site_lists, s->n_chains, s->chains_per_terrain, s->chain_offset, s->seed, chunk,
                             s->bounds_dev, target, s->noise, s->totals_dev);
        else if (variant == TSS_KERNEL_THREAD)
            rc = sls_run_t16(e, s->rows_dev, s->tabs_dev, s->states, s->site_lists, s->n_chains, s->chains_per_terrain, s->chain_offset, s->seed, chunk,
                             s->bounds_dev, target, s->noise, s->totals_dev);
        else
            rc = (variant == TSS_KERNEL_HALF_WARP ? sls_run_h16 : sls_run)(e, s->rows_dev, s->tabs_dev, s->states, s->n_chains, s->chains_per_terrain,
                                                                          s->chain_offset, s->seed, chunk, s->bounds_dev, target, s->noise, s->totals_dev);
        if (rc == TSS_OK) rc = sls_best_reduce(e, s->states, chains_per_group, s->n_chains, s->n_groups, s->best_dev, s->bounds_dev, s->reduce_key_dev);
        // multi-GPU portfolio: the one exchange of the path, in-stream on the device-resident bound (no host round trip)
        if (rc == TSS_OK && e->comm && s->share && s->n_groups == 1) rc = comm_allreduce_min(e, e->comm, s->bounds_dev, 1);
        if (rc) return rc;
    }
    TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(s->best_host, s->best_dev, sizeof(int2) * (size_t)s->n_groups, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(s->totals_host, s->totals_dev, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost, e->stream));
    s->dirty = true;
    s->timed = true;
    e->stats.n_solves++;
    return TSS_OK;
}

// the search's running totals (candidates scored, steps, flips) into the engine's counters: what they grew since last seen
static void fold_totals(tss_engine* e, tss_search* s, unsigned long long t0, unsigned long long t1, unsigned long long t2) {
    e->stats.candidates_scored += t0 - s->totals_seen[0];
    e->stats.sls_steps += t1 - s->totals_seen[1];
    e->stats.sls_flips += t2 - s->totals_seen[2];
    s->totals_seen[0] = t0;
    s->totals_seen[1] = t1;
    s->totals_seen[2] = t2;
}

static int search_sync(tss_search* s) {
    tss_engine* e = s->e;
    if (!s->dirty) return TSS_OK;
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    if (s->timed) {  // (an epoch recorded both events; never query unrecorded ones: the error would stick)
        float ms = 0;
        if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) != cudaSuccess) cudaGetLastError();
        e->stats.device_ms = ms;
        s->timed = false;
    }
    auto total = [s](int i) { return s->lns ? lns_total(s->lns, i) : (s->lnsp ? lnsp_total(s->lnsp, i) : s->totals_host[i]); };
    fold_totals(e, s, total(0), total(1), total(2));
    s->dirty = false;
    return TSS_OK;
}

int tss_search_best_count(tss_search* s, int32_t* count) {
    if (!s || !count) return TSS_E_INVALID;
    int rc = search_sync(s);
    if (rc) return rc;
    if (s->lns || s->lnsp) {  // the global layout is always complete; a bound given from outside hides counts that do not beat it
        int c = s->lns ? lns_count(s->lns) : lnsp_value(s->lnsp);
        *count = c < s->external_bound ? c : -1;
        s->e->stats.best_count = *count;
        return TSS_OK;
    }
    int best = sls::NO_BOUND;
    for (int g = 0; g < s->n_groups; g++) best = s->best_host[g].x < best ? s->best_host[g].x : best;
    *count = best >= sls::NO_BOUND ? -1 : best;
    s->e->stats.best_count = *count;
    return TSS_OK;
}

int tss_search_global_best(tss_search* s, int32_t* count) {
    if (!s || !count) return TSS_E_INVALID;
    tss_engine* e = s->e;
    int rc = search_sync(s);
    if (rc) return rc;
    if (s->lns || s->lnsp) return tss_search_best_count(s, count);
    int b = sls::NO_BOUND;
    TSS_CUDA(e, cudaMemcpy(&b, s->bounds_dev, sizeof(int), cudaMemcpyDeviceToHost));
    *count = b >= sls::NO_BOUND ? -1 : b;
    return TSS_OK;
}

int tss_search_set_bound(tss_search* s, int32_t count) {
    if (!s) return TSS_E_INVALID;
    tss_engine* e = s->e;
    if (count < 0) return e->fail(TSS_E_INVALID, "tss_search_set_bound: negative bound");
    int rc = search_sync(s);
    if (rc) return rc;
    if (s->lns || s->lnsp) { s->external_bound = count < s->external_bound ? count : s->external_bound; return TSS_OK; }
    TSS_CUDA(e, cudaSetDevice(e->device));
    bound_min_kernel<<<(s->n_groups + 255) / 256, 256, 0, e->stream>>>(s->bounds_dev, s->n_groups, count, false);   // in-stream, before the next epoch
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    s->dirty = true;
    return TSS_OK;
}

int tss_search_read_chains(tss_search* s, uint32_t* S, uint32_t* best_S, int32_t* k, int32_t* best, uint32_t* step, uint64_t* scored) {
    if (!s) return TSS_E_INVALID;
    tss_engine* e = s->e;
    if (s->lns || s->lnsp || s->multi) return e->fail(TSS_E_UNSUPPORTED, "tss_search_read_chains: only the 1x1 search on grids up to 32x32 exposes per-chain state");
    int rc = search_sync(s);
    if (rc) return rc;
    std::vector<sls::ChainState> st((size_t)s->n_chains);
    TSS_CUDA(e, cudaMemcpy(st.data(), s->states, sizeof(sls::ChainState) * st.size(), cudaMemcpyDeviceToHost));
    for (size_t c = 0; c < st.size(); c++) {
        if (S) std::memcpy(S + c * 32, st[c].S, 128);
        if (best_S) std::memcpy(best_S + c * 32, st[c].bestS, 128);
        if (k) k[c] = st[c].k;
        if (best) best[c] = st[c].best;
        if (step) step[c] = st[c].step;
        if (scored) scored[c] = ((uint64_t)st[c].scored_hi << 32) | st[c].scored_lo;
    }
    return TSS_OK;
}

int tss_search_read_placements(tss_search* s, uint16_t* items, int32_t* k, uint16_t* best_items, int32_t* best_k, int32_t* best, uint32_t* step,
                               tss_dims* key_dims, int32_t* n_keys) {
    if (!s) return TSS_E_INVALID;
    tss_engine* e = s->e;
    if (!s->multi) return e->fail(TSS_E_UNSUPPORTED, "tss_search_read_placements: only the placement search (platform sets beyond 1x1 on grids up to 32x32)");
    int rc = search_sync(s);
    if (rc) return rc;
    if (n_keys) *n_keys = (int32_t)s->key_dims.size();
    if (key_dims)
        for (size_t i = 0; i < s->key_dims.size(); i++) key_dims[i] = tss_dims{s->key_dims[i].x, s->key_dims[i].y};
    return slsm_read_states(e, s->mstates, s->n_chains, items, k, best_items, best_k, best, step);
}

int tss_search_write_chains(tss_search* s, const uint32_t* S) {
    if (!s) return TSS_E_INVALID;
    tss_engine* e = s->e;
    if (!S) return e->fail(TSS_E_INVALID, "tss_search_write_chains: null layout");
    if (s->lns || s->lnsp || s->multi) return e->fail(TSS_E_UNSUPPORTED, "tss_search_write_chains: only the 1x1 search on grids up to 32x32 takes a warm start");
    int rc = search_sync(s);
    if (rc) return rc;
    const uint32_t colmask = s->w >= 32 ? 0xffffffffu : ((1u << s->w) - 1u);
    for (size_t c = 0; c < (size_t)s->n_chains; c++)
        for (int r = 0; r < 32; r++)
            if (S[c * 32 + r] & (r < s->h ? ~colmask : 0xffffffffu)) return e->fail(TSS_E_INVALID, "tss_search_write_chains: chain %zu has a support outside the grid (row %d)", c, r);
    std::vector<sls::ChainState> st((size_t)s->n_chains);
    TSS_CUDA(e, cudaMemcpy(st.data(), s->states, sizeof(sls::ChainState) * st.size(), cudaMemcpyDeviceToHost));
    for (size_t c = 0; c < st.size(); c++) {
        int k = 0;
        for (int r = 0; r < 32; r++) { st[c].S[r] = S[c * 32 + r]; k += __builtin_popcount(S[c * 32 + r]); }
        st[c].k = k;
        st[c].done = 0;
    }
    TSS_CUDA(e, cudaMemcpy(s->states, st.data(), sizeof(sls::ChainState) * st.size(), cudaMemcpyHostToDevice));
    return TSS_OK;
}

// Grids larger than 32x32 are searched with 1x1 supports only (window decomposition).  When the platform set holds larger
// platforms, supports that fit under one footprint are merged into that platform: its reach contains the reach of every
// support under it (validate() dilates from all ceiling tiles under a footprint, platform_layout.rs:116-141), so the
// layout stays complete, and footprints are kept pairwise disjoint and in bounds.  Greedy: larger platforms first, per
// platform size the anchors holding most supports first.  A valid, tighter bound — not a search over placements.
// tiles supported by one platform: validate()'s rule restricted to its own window (footprint + 3 on every side)
static void platform_reach(const std::vector<uint8_t>& grid, int w, int h, const tss_platform& p, std::vector<int>& out) {
    const Dims d = platform_dims(p);
    const int x0 = std::max(p.x - 3, 0), y0 = std::max(p.y - 3, 0), x1 = std::min(p.x + d.w + 3, w), y1 = std::min(p.y + d.h + 3, h);
    const int bw = x1 - x0, bh = y1 - y0;
    std::vector<uint8_t> cur((size_t)bw * bh, 0), nxt;
    for (int y = std::max(p.y, 0); y < std::min(p.y + d.h, h); y++)
        for (int x = std::max(p.x, 0); x < std::min(p.x + d.w, w); x++)
            if (grid[(size_t)y * w + x]) cur[(size_t)(y - y0) * bw + (x - x0)] = 1;
    for (int round = 0; round < kTerrainSupportDistance - 1; round++) {
        nxt = cur;
        for (int y = 0; y < bh; y++)
            for (int x = 0; x < bw; x++) {
                if (!cur[(size_t)y * bw + x]) continue;
                const int nx[4] = {x + 1, x, x - 1, x}, ny[4] = {y, y + 1, y, y - 1};
                for (int k = 0; k < 4; k++)
                    if (nx[k] >= 0 && nx[k] < bw && ny[k] >= 0 && ny[k] < bh && grid[(size_t)(ny[k] + y0) * w + nx[k] + x0]) nxt[(size_t)ny[k] * bw + nx[k]] = 1;
            }
        cur.swap(nxt);
    }
    out.clear();
    for (int y = 0; y < bh; y++)
        for (int x = 0; x < bw; x++)
            if (cur[(size_t)y * bw + x]) out.push_back((y + y0) * w + x + x0);
}

// Drops platforms every tile of whose reach is also supported by another platform (smallest platforms first): the
// merged platforms reach further than the supports they replaced, which makes many neighbours redundant.
static void prune_redundant(const std::vector<uint8_t>& grid, int w, int h, std::vector<tss_platform>& plats) {
    std::vector<std::vector<int>> reach(plats.size());
    std::vector<uint16_t> cover((size_t)w * h, 0);
    for (size_t i = 0; i < plats.size(); i++) {
        platform_reach(grid, w, h, plats[i], reach[i]);
        for (int t : reach[i]) cover[(size_t)t]++;
    }
    std::vector<size_t> order(plats.size());
    for (size_t i = 0; i < order.size(); i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return plats[a].def_w * plats[a].def_h < plats[b].def_w * plats[b].def_h; });
    std::vector<uint8_t> drop(plats.size(), 0);
    for (size_t i : order) {
        bool redundant = true;
        for (int t : reach[i]) redundant = redundant && cover[(size_t)t] >= 2;
        if (!redundant) continue;
        drop[i] = 1;
        for (int t : reach[i]) cover[(size_t)t]--;
    }
    std::vector<tss_platform> kept;
    for (size_t i = 0; i < plats.size(); i++)
        if (!drop[i]) kept.push_back(plats[i]);
    plats.swap(kept);
}

static void merge_supports(int w, int h, const std::vector<int2>& key_dims, const std::vector<tss_platform>& key_proto, std::vector<tss_platform>& plats) {
    if (key_dims.size() <= 1 || plats.empty()) return;
    std::vector<uint8_t> sup((size_t)w * h, 0), occ((size_t)w * h, 0);
    for (auto& p : plats) sup[(size_t)p.y * w + p.x] = 1;
    std::vector<int> order(key_dims.size());
    for (size_t i = 0; i < order.size(); i++) order[i] = (int)i;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return key_dims[a].x * key_dims[a].y > key_dims[b].x * key_dims[b].y; });
    std::vector<tss_platform> merged;
    std::vector<int> pre((size_t)(w + 1) * (h + 1));
    for (int key : order) {
        const int pw = key_dims[key].x, ph = key_dims[key].y;
        if (pw * ph <= 1 || pw > w || ph > h) continue;
        for (;;) {  // rounds: recount after every batch of non-conflicting merges
            std::fill(pre.begin(), pre.end(), 0);
            for (int y = 0; y < h; y++)
                for (int x = 0; x < w; x++)
                    pre[(size_t)(y + 1) * (w + 1) + x + 1] = sup[(size_t)y * w + x] + pre[(size_t)y * (w + 1) + x + 1] + pre[(size_t)(y + 1) * (w + 1) + x] - pre[(size_t)y * (w + 1) + x];
            auto inside = [&](int x, int y) { return pre[(size_t)(y + ph) * (w + 1) + x + pw] - pre[(size_t)y * (w + 1) + x + pw] - pre[(size_t)(y + ph) * (w + 1) + x] + pre[(size_t)y * (w + 1) + x]; };
            std::vector<std::pair<int, int>> cand;  // (supports under the footprint, anchor)
            for (int y = 0; y + ph <= h; y++)
                for (int x = 0; x + pw <= w; x++) {
                    const int c = inside(x, y);
                    if (c >= 2) cand.push_back({c, y * w + x});
                }
            if (cand.empty()) break;
            std::stable_sort(cand.begin(), cand.end(), [](const std::pair<int, int>& a, const std::pair<int, int>& b) { return a.first > b.first; });
            int placed = 0;
            for (auto& [c0, anchor] : cand) {
                const int x = anchor % w, y = anchor / w;
                int c = 0;
                bool free_ = true;
                for (int yy = y; yy < y + ph && free_; yy++)
                    for (int xx = x; xx < x + pw; xx++) {
                        if (occ[(size_t)yy * w + xx]) { free_ = false; break; }
                        c += sup[(size_t)yy * w + xx];
                    }
                if (!free_ || c < 2) continue;   // (an earlier merge of this round took its supports or its tiles)
                for (int yy = y; yy < y + ph; yy++)
                    for (int xx = x; xx < x + pw; xx++) { occ[(size_t)yy * w + xx] = 1; sup[(size_t)yy * w + xx] = 0; }
                tss_platform p = key_proto[key];
                p.x = x; p.y = y;
                merged.push_back(p);
                placed++;
            }
            if (!placed) break;
        }
    }
    if (merged.empty()) return;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            if (sup[(size_t)y * w + x]) merged.push_back(tss_platform{x, y, 1, 1, 0});
    plats.swap(merged);
}

// The greedy placement cover of the terrain (greedy.cu) as platforms, redundant ones pruned (platform sets of at most 16 dims
// keys, each at most 6x6).  greedy.cu emits placements in the order its threads finish and prune_redundant keeps the first of
// equally large redundant platforms, so `anchor_order` sorts the placements row-major first: the same layout on every run.
static int greedy_layout(tss_engine* e, const tss_search* s, bool anchor_order, std::vector<tss_platform>& out) {
    BitGrid bg = BitGrid::from_bytes(s->grid.data(), s->w, s->h);
    std::vector<int4> placed;
    int rc = greedy_cover(e, bg.rows.data(), s->w, s->h, s->key_dims, placed);
    if (rc) return rc;
    if (anchor_order) std::sort(placed.begin(), placed.end(), [](const int4& a, const int4& b) { return a.y != b.y ? a.y < b.y : a.x < b.x; });
    out.clear();
    for (auto& q : placed) {
        tss_platform pl = s->key_proto[(size_t)q.z];
        pl.x = q.x; pl.y = q.y;
        out.push_back(pl);
    }
    prune_redundant(s->grid, s->w, s->h, out);
    return TSS_OK;
}

// The start layout under per-type limits: the platforms of `plats` in row-major anchor order, each kept only while every class
// it belongs to has room, then a 1x1 on every ceiling tile (row-major) that is still unsupported.  Such a tile lies under no
// footprint, and 1x1 is in no class: the layout is complete and keeps every limit.
static void limit_start_layout(const tss_search* s, const std::vector<uint32_t>& mask, const std::vector<int>& lim, std::vector<tss_platform>& plats) {
    std::vector<int> n(lim.size(), 0), reach;
    std::vector<uint8_t> sup((size_t)s->w * s->h, 0);
    std::vector<tss_platform> kept;
    auto add = [&](const tss_platform& p) {
        kept.push_back(p);
        platform_reach(s->grid, s->w, s->h, p, reach);
        for (int t : reach) sup[(size_t)t] = 1;
    };
    for (const tss_platform& p : plats) {
        const Dims d = platform_dims(p);
        uint32_t m = 0;
        for (size_t k = 0; k < s->key_dims.size(); k++)
            if (s->key_dims[k].x == d.w && s->key_dims[k].y == d.h) m = mask[k];
        bool room = true;
        for (size_t j = 0; j < lim.size(); j++) room = room && !(((m >> j) & 1u) && n[j] >= lim[j]);
        if (!room) continue;
        for (size_t j = 0; j < lim.size(); j++) n[j] += (m >> j) & 1u;
        add(p);
    }
    for (int t = 0; t < s->w * s->h; t++)
        if (s->grid[(size_t)t] && !sup[(size_t)t]) add(tss_platform{t % s->w, t / s->w, 1, 1, 0});
    plats.swap(kept);
}

// TSS_KERNEL_WINDOW_PLACEMENTS on a grid larger than 32x32: dims keys, costs and the start layout — the greedy placement cover,
// redundant platforms pruned, as an anchor grid — on the device, then the search (lns_placements.cu).  seeds = chains per window.
// card / n_card: per-type limit records (tss_search_create_with_limits); when they make classes, the start layout is trimmed to
// keep them (limit_start_layout) and the search keeps them in every phase.
static int window_placements_create(tss_engine* e, tss_search* s, const tss_dims* defs, int n_defs, int seeds, const int32_t* card, int n_card) {
    build_keys(defs, n_defs, s->key_dims, s->key_proto);
    bool fits = s->key_dims.size() > 1 && (int)s->key_dims.size() <= slsm_max_keys();
    for (auto& kd : s->key_dims) fits = fits && kd.x <= 6 && kd.y <= 6;
    if (!fits)
        return e->fail(TSS_E_UNSUPPORTED, "tss_search_create: the window placement search needs a platform set beyond {1x1} with at most %d dims keys, each at most 6x6",
                       slsm_max_keys());
    if (e->comm && comm_world(e->comm) > 1) return e->fail(TSS_E_UNSUPPORTED, "tss_search_create: the window placement search runs on a single rank");
    std::vector<uint32_t> mask;
    std::vector<int> lim;
    if (int rc = card_limit_classes(s->key_dims, card, n_card, mask, lim)) return e->fail(rc, "tss_search_create_with_limits: bad limit records");
    s->kernel = TSS_KERNEL_WINDOW_PLACEMENTS;
    s->key_costs.assign(s->key_dims.size(), 1);
    std::vector<tss_platform> start;
    int rc = greedy_layout(e, s, true, start);
    if (rc) return rc;
    if (!lim.empty()) limit_start_layout(s, mask, lim, start);
    std::vector<uint8_t> anchors((size_t)s->w * s->h, 0);
    for (auto& p : start) {
        const Dims d = platform_dims(p);
        for (size_t k = 0; k < s->key_dims.size(); k++)
            if (s->key_dims[k].x == d.w && s->key_dims[k].y == d.h) anchors[(size_t)p.y * s->w + p.x] = (uint8_t)(k + 1);
    }
    const std::vector<int> order = keys_by_area(s->key_dims);
    const size_t nk = s->key_dims.size();
    cudaError_t err = cudaMalloc(&s->keys_dev, sizeof(int2) * (size_t)slsm_max_keys());
    if (err == cudaSuccess) err = cudaMalloc(&s->costs_dev, sizeof(int) * 2 * (size_t)slsm_max_keys());   // costs | keys ordered by area
    if (err == cudaSuccess) err = cudaMemcpy(s->keys_dev, s->key_dims.data(), sizeof(int2) * nk, cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = cudaMemcpy(s->costs_dev, s->key_costs.data(), sizeof(int) * nk, cudaMemcpyHostToDevice);
    if (err == cudaSuccess) err = cudaMemcpy(s->costs_dev + slsm_max_keys(), order.data(), sizeof(int) * nk, cudaMemcpyHostToDevice);
    if (err != cudaSuccess) return e->fail(TSS_E_CUDA, "tss_search_create: %s", cudaGetErrorString(err));
    rc = lnsp_create(e, s->grid.data(), s->w, s->h, anchors.data(), s->keys_dev, s->costs_dev, s->costs_dev + slsm_max_keys(), (int)nk, seeds, s->seed,
                     s->chain_offset, s->noise, mask.data(), lim.data(), (int)lim.size(), &s->lnsp);
    if (rc) return rc;
    s->n_chains = lnsp_chains(s->lnsp);
    return TSS_OK;
}

int tss_layout_merge_supports(const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, tss_platform* plats, int32_t n,
                              int32_t cap) {
    if (!grid || w <= 0 || h <= 0 || n < 0 || (n > 0 && !plats) || (n_defs > 0 && !defs)) return TSS_E_INVALID;
    std::vector<int2> key_dims;
    std::vector<tss_platform> key_proto;
    build_keys(defs, n_defs, key_dims, key_proto);
    std::vector<tss_platform> supports, others;
    for (int i = 0; i < n; i++) {
        const tss_platform& p = plats[i];
        const bool one = p.def_w == 1 && p.def_h == 1;
        if (one && (p.x < 0 || p.y < 0 || p.x >= w || p.y >= h)) return TSS_E_INVALID;
        (one ? supports : others).push_back(p);
    }
    if (!others.empty()) return TSS_E_UNSUPPORTED;   // only layouts of 1x1 supports are merged
    std::vector<uint8_t> g(grid, grid + (size_t)w * h);
    merge_supports(w, h, key_dims, key_proto, supports);
    prune_redundant(g, w, h, supports);
    if ((int)supports.size() > cap) return TSS_E_CAPACITY;
    for (size_t i = 0; i < supports.size(); i++) plats[i] = supports[i];
    return (int)supports.size();
}

// placement codes of the placement search (key << 10 | y << 5 | x, sls_multi.cu) -> platforms
static void codes_to_platforms(const tss_search* s, const uint16_t* codes, int n, tss_platform* out) {
    for (int i = 0; i < n; i++) {
        tss_platform p = s->key_proto[codes[i] >> 10];
        p.x = codes[i] & 31;
        p.y = (codes[i] >> 5) & 31;
        out[i] = p;
    }
}

int tss_search_best_layout(tss_search* s, tss_platform* out, int32_t cap, int32_t* n_out) {
    if (!s || !n_out) return TSS_E_INVALID;
    tss_engine* e = s->e;
    int rc = search_sync(s);
    if (rc) return rc;
    std::vector<tss_platform> plats;
    int2 best;
    if (s->lns) {
        std::vector<uint32_t> rows;
        rc = lns_layout(e, s->lns, rows);
        if (rc) return rc;
        const int wpr = (s->w + 31) / 32;
        for (int y = 0; y < s->h; y++)
            for (int x = 0; x < s->w; x++)
                if ((rows[(size_t)y * wpr + (x >> 5)] >> (x & 31)) & 1u) plats.push_back(tss_platform{x, y, 1, 1, 0});
        if (s->key_dims.size() > 1) {
            // two constructors for a layout with larger platforms, the better one wins: the searched 1x1 layout with supports
            // merged under footprints, and a greedy placement cover of the terrain (greedy.cu)
            merge_supports(s->w, s->h, s->key_dims, s->key_proto, plats);
            prune_redundant(s->grid, s->w, s->h, plats);
            if (!s->greedy_done) {
                bool fits = true;
                for (auto& kd : s->key_dims) fits = fits && kd.x <= 6 && kd.y <= 6;
                if (fits && (int)s->key_dims.size() <= 16) {
                    rc = greedy_layout(e, s, false, s->greedy_plats);
                    if (rc) return rc;
                }
                s->greedy_done = true;
            }
            if (!s->greedy_plats.empty() && s->greedy_plats.size() < plats.size()) plats = s->greedy_plats;
        }
        best = make_int2((int)plats.size(), 0);
    } else if (s->lnsp) {
        std::vector<uint8_t> anchors;
        rc = lnsp_anchors(e, s->lnsp, anchors);
        if (rc) return rc;
        int cost = 0;
        for (int y = 0; y < s->h; y++)
            for (int x = 0; x < s->w; x++) {
                const int a = anchors[(size_t)y * s->w + x];
                if (!a) continue;
                tss_platform p = s->key_proto[(size_t)a - 1];
                p.x = x; p.y = y;
                plats.push_back(p);
                cost += s->key_costs[(size_t)a - 1];
            }
        if (cost != lnsp_value(s->lnsp)) return e->fail(TSS_E_CUDA, "internal error: layout costs %d, the search reported %d", cost, lnsp_value(s->lnsp));
        int n_j = 0, l_j = 0;
        if (const int j = lnsp_over_limit(s->lnsp, &n_j, &l_j); j >= 0)
            return e->fail(TSS_E_CUDA, "internal error: the layout holds %d platforms of limit class %d, its limit is %d", n_j, j, l_j);
        best = make_int2((int)plats.size(), 0);
    } else if (s->multi) {
        best = s->best_host[0];
        if (best.x >= sls::NO_BOUND || best.y < 0) { *n_out = 0; return e->fail(TSS_E_INVALID, "tss_search_best_layout: no complete layout found yet"); }
        std::vector<uint16_t> codes;
        rc = slsm_read_best(e, s->mstates, best.y, codes);
        if (rc) return rc;
        int cost = 0;
        for (uint16_t code : codes) cost += s->key_costs[code >> 10];
        if (cost != best.x) return e->fail(TSS_E_CUDA, "internal error: best layout costs %d, chain reported %d", cost, best.x);
        best.x = (int)codes.size();
        plats.resize(codes.size());
        codes_to_platforms(s, codes.data(), (int)codes.size(), plats.data());
    } else {
        best = s->best_host[0];
        if (best.x >= sls::NO_BOUND || best.y < 0) { *n_out = 0; return e->fail(TSS_E_INVALID, "tss_search_best_layout: no complete layout found yet"); }
        sls::ChainState st;
        TSS_CUDA(e, cudaMemcpy(&st, s->states + best.y, sizeof st, cudaMemcpyDeviceToHost));
        for (int y = 0; y < s->h; y++)
            for (int x = 0; x < s->w; x++)
                if ((st.bestS[y] >> x) & 1u) plats.push_back(tss_platform{x, y, 1, 1, 0});
    }
    *n_out = (int)plats.size();
    // every witness is re-validated by kernel (a) before it leaves the engine
    uint32_t offsets[2] = {0, (uint32_t)plats.size()};
    int32_t res[4] = {0, 0, 0, 0};  // unsupported tiles, platforms, overlapping, out of bounds (platform_layout.rs:187-191)
    rc = tss_eval_platforms(e, s->grid.data(), s->w, s->h, plats.data(), offsets, 1, res);
    if (rc < 0) return rc;
    if (res[0] != 0 || res[2] != 0 || res[3] != 0 || (int)plats.size() != best.x)
        return e->fail(TSS_E_CUDA, "internal error: SLS witness failed validation (%d unsupported tiles, %d overlapping, %d out of bounds, %zu platforms, expected %d)",
                       res[0], res[2], res[3], plats.size(), best.x);
    if ((int)plats.size() > cap || !out) return e->fail(TSS_E_CAPACITY, "tss_search_best_layout: need room for %zu platforms", plats.size());
    std::memcpy(out, plats.data(), sizeof(tss_platform) * plats.size());
    return TSS_OK;
}

int tss_search_set_weights(tss_search* s, const int32_t* weights, int32_t n_weights) {
    if (!s) return TSS_E_INVALID;
    tss_engine* e = s->e;
    if (n_weights < 0 || (n_weights > 0 && !weights)) return e->fail(TSS_E_INVALID, "tss_search_set_weights: bad arguments");
    if (!s->multi && !s->lnsp)
        return e->fail(TSS_E_UNSUPPORTED, "tss_search_set_weights: the weight objective needs a platform set beyond {1x1} on a grid up to 32x32, or the window placement search");
    int rc = search_sync(s);
    if (rc) return rc;
    for (size_t k = 0; k < s->key_dims.size(); k++) {
        const long cost = key_cost(s->key_proto[k], weights, n_weights);
        if (cost <= 0 || cost > 4096)
            return e->fail(TSS_E_UNSUPPORTED, "tss_search_set_weights: platform costs must be in 1..4096 (got %ld for %dx%d)", cost, s->key_proto[k].def_w, s->key_proto[k].def_h);
        s->key_costs[k] = (int)cost;
    }
    TSS_CUDA(e, cudaMemcpy(s->costs_dev, s->key_costs.data(), sizeof(int) * s->key_costs.size(), cudaMemcpyHostToDevice));
    if (s->lnsp) {   // the objective of the current layout under the new costs
        rc = lnsp_objective(e, s->lnsp);
        if (rc) return rc;
        s->dirty = true;
    }
    return TSS_OK;
}

int tss_card_limit_classes(const tss_dims* defs, int32_t n_defs, const int32_t* card, int32_t n_card, int32_t* key_mask, int32_t* class_limit,
                           int32_t* n_keys, int32_t* n_classes) {
    if ((n_defs > 0 && !defs) || n_defs < 0 || n_card < 0 || (n_card > 0 && !card) || !key_mask || !class_limit || !n_keys || !n_classes) return TSS_E_INVALID;
    std::vector<int2> kd;
    std::vector<tss_platform> kp;
    build_keys(defs, n_defs, kd, kp);
    if ((int)kd.size() > slsm_max_keys()) return TSS_E_UNSUPPORTED;
    std::vector<uint32_t> mask;
    std::vector<int> lim;
    const int rc = card_limit_classes(kd, card, n_card, mask, lim);
    if (rc) return rc;
    for (size_t k = 0; k < kd.size(); k++) key_mask[k] = (int32_t)mask[k];
    for (size_t j = 0; j < lim.size(); j++) class_limit[j] = lim[j];
    *n_keys = (int32_t)kd.size();
    *n_classes = (int32_t)lim.size();
    return TSS_OK;
}

int tss_search_set_card_limits(tss_search* s, const int32_t* card, int32_t n_card) {
    if (!s) return TSS_E_INVALID;
    tss_engine* e = s->e;
    if (n_card < 0 || (n_card > 0 && !card)) return e->fail(TSS_E_INVALID, "tss_search_set_card_limits: bad arguments");
    if (s->started) return e->fail(TSS_E_INVALID, "tss_search_set_card_limits: call it before the first tss_search_run");
    for (int i = 0; i < n_card; i++) {
        if (card[3 * i] == 1 && card[3 * i + 1] == 1)
            return e->fail(TSS_E_INVALID, "tss_search_set_card_limits: the platform count (1x1) is the search's bound, not a per-type limit");
        if (card[3 * i + 2] < 0) return e->fail(TSS_E_INVALID, "tss_search_set_card_limits: negative limit for %dx%d", card[3 * i], card[3 * i + 1]);
    }
    std::vector<uint32_t> mask;
    std::vector<int> lim;
    int rc = card_limit_classes(s->key_dims, card, n_card, mask, lim);
    if (rc) return e->fail(rc, "tss_search_set_card_limits: bad limit records");
    if (lim.empty()) return TSS_OK;   // every record vacuous (e.g. on a {1x1}-only set)
    if (!s->multi)
        return e->fail(TSS_E_UNSUPPORTED, "tss_search_set_card_limits: per-type limits need the placement search (a platform set beyond {1x1} on a grid up to 32x32)");
    rc = search_sync(s);
    if (rc) return rc;
    std::vector<int> dev(2 * (size_t)slsm_max_keys(), 0);
    for (size_t k = 0; k < mask.size(); k++) dev[k] = (int)mask[k];
    for (size_t j = 0; j < lim.size(); j++) dev[(size_t)slsm_max_keys() + j] = lim[j];
    TSS_CUDA(e, cudaMemcpy(s->costs_dev + 2 * slsm_max_keys(), dev.data(), sizeof(int) * dev.size(), cudaMemcpyHostToDevice));
    s->n_classes = (int)lim.size();
    return TSS_OK;
}

// The end of a one-shot solve that succeeded: a 1x1 search of one terrain group is kept for the next call (cached_search),
// so is a placement search, without the call's per-type limits (cached_multi: the next solve's fused first epoch runs on it as
// it stands, tss_search_create adopts it).  Everything else, and a workspace whose slot is taken, is destroyed.
static void keep_or_destroy(tss_engine* e, tss_search* s, int rc) {
    if (!s->lns && !s->lnsp && !s->multi && s->n_groups == 1 && !e->cached_search && rc == TSS_OK) {
        cudaStreamSynchronize(e->stream);
        e->cached_search = s;
    } else if (s->multi && !e->cached_multi && rc == TSS_OK) {
        cudaStreamSynchronize(e->stream);
        s->n_classes = 0;
        e->cached_multi = s;
    } else {
        tss_search_destroy(s);
    }
}

// The fused first epoch of a one-shot solve on a cached workspace (sls_h16.cu OneShot, sls_multi.cu OneShotM) between
// fused_epoch_begin and fused_epoch_end: the caller enqueues the one launch in between and reads its result block after.
static int fused_epoch_begin(tss_engine* e, tss_search* s) {
    const int rc = search_sync(s);   // (nothing in flight on a cached workspace; folds counters if there was)
    if (rc == TSS_OK) cudaEventRecord(e->ev0, e->stream);
    return rc;
}

// rc = the launch's: one synchronisation, then the epoch's device time, and the epoch counts as a solve
static int fused_epoch_end(tss_engine* e, int rc) {
    cudaEventRecord(e->ev1, e->stream);
    if (rc == TSS_OK && cudaStreamSynchronize(e->stream) != cudaSuccess)
        rc = e->fail(TSS_E_CUDA, "tss_solve_upper_bound: fused epoch failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc == TSS_OK) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) != cudaSuccess) cudaGetLastError();
        e->stats.device_ms = ms;
        e->stats.n_solves++;
    }
    return rc;
}

int tss_solve_min_weight(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                         const int32_t* weights, int32_t n_weights, int64_t weight_limit, uint64_t seed, int32_t budget_ms,
                         int64_t max_steps, tss_platform* out, int32_t cap, int32_t* n_out, int64_t* out_weight) {
    if (!e) return TSS_E_INVALID;
    if (n_out) *n_out = 0;
    e->stats.interrupted = 0;
    e->stats.best_count = -1;
    tss_search_params p{seed, 0, 0, -1, 0};
    tss_search* s = nullptr;
    int rc = tss_search_create(e, grid, w, h, defs, n_defs, &p, &s);
    if (rc) return rc;
    s->share = false;
    rc = tss_search_set_weights(s, weights, n_weights);
    if (rc == TSS_OK && weight_limit >= 0) rc = tss_search_set_bound(s, (int32_t)(weight_limit + 1 < sls::NO_BOUND ? weight_limit + 1 : sls::NO_BOUND));
    const double t0 = now_ms();
    const bool first_model_only = budget_ms <= 0 && max_steps <= 0;
    if (first_model_only) max_steps = 1 << 16;
    int64_t done_steps = 0, epoch = 64;
    int best = -1;
    while (rc == TSS_OK) {
        if (e->interrupted()) { e->stats.interrupted = 1; break; }
        int64_t steps = epoch;
        if (max_steps > 0 && done_steps + steps > max_steps) steps = max_steps - done_steps;
        if (steps <= 0) break;
        rc = tss_search_run(s, steps, 0);
        if (rc == TSS_OK) rc = tss_search_best_count(s, &best);
        if (rc) break;
        done_steps += steps;
        if (first_model_only && best >= 0) break;
        if (budget_ms > 0 && now_ms() - t0 >= budget_ms) break;
        if (epoch < 4096) epoch *= 2;
    }
    int result = TSS_UNKNOWN;
    if (rc == TSS_OK && best >= 0) {
        int n = 0;
        rc = tss_search_best_layout(s, out, cap, &n);
        if (n_out) *n_out = n;
        if (out_weight) *out_weight = best;
        if (rc == TSS_OK) result = TSS_SAT;
    }
    keep_or_destroy(e, s, rc);   // the GUI tightens weight_limit call after call (app.rs:235-245): the next tss_search_create adopts the workspace
    return rc != TSS_OK ? rc : result;
}

// The one-shot solve behind tss_solve_upper_bound and tss_solve_with_limits: a layout whose objective (platform count, or total
// weight with `weights`) is at most `limit` (< 0: unbounded) and that keeps the per-type limits `card` (records without 1x1,
// see tss_search_set_card_limits).  *out_objective = the objective of the layout returned.
static int solve_search(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, int64_t limit,
                        const int32_t* weights, int32_t n_weights, const int32_t* card, int32_t n_card, uint64_t seed, int32_t budget_ms,
                        int64_t max_steps, tss_platform* out, int32_t cap, int32_t* n_out, int64_t* out_objective) {
    if (!e) return TSS_E_INVALID;
    if (n_out) *n_out = 0;
    const int32_t card_limit = limit < 0 ? -1 : (int32_t)std::min<int64_t>(limit, sls::NO_BOUND - 1);
    // weights and limits live in the search's own buffers: only the plain count objective may take the fused first epochs
    bool limited = false;
    if (n_card > 0) {
        std::vector<int2> kd;
        std::vector<tss_platform> kp;
        std::vector<uint32_t> mask;
        std::vector<int> lim;
        build_keys(defs, n_defs, kd, kp);
        if (card_limit_classes(kd, card, n_card, mask, lim) != TSS_OK) return e->fail(TSS_E_INVALID, "tss_solve_with_limits: bad limit records");
        limited = !lim.empty();
    }
    const bool plain = n_weights <= 0 && !limited;
    // One SAT-like call (no budget, no step count: return the first model within the bound) is latency bound: few
    // chains per SM step fastest (measured on rect 16x16, profiles/tto_sweep.py: 16 chains per SM on the half-warp kernel
    // 0.23 ms, 64 per SM 0.34 ms, 128 per SM 0.50 ms per call).  A call with an effort budget is throughput bound: the
    // engine default (one chain per thread where the grid fits, 384 chains per SM).
    const bool latency_mode = budget_ms <= 0 && max_steps <= 0 && h <= 16;
    const int kernel = latency_mode ? TSS_KERNEL_HALF_WARP : TSS_KERNEL_AUTO;
    const int want_chains = (w > 0 && h > 0) ? (latency_mode ? e->prop.multiProcessorCount * 16 : default_chains(e, w, h, kernel)) : 0;
    bool only_1x1 = true;
    for (int i = 0; i < n_defs; i++) only_1x1 = only_1x1 && defs && defs[i].w == 1 && defs[i].h == 1;
    // (the window-decomposed and the placement search read n_chains differently: leave their defaults)
    // placement search (platform sets beyond {1x1}): 4 chains per SM when only the first model is asked for (measured on
    // test/ex1-3 with the default-8 set, profiles/c1_timing.py: 0.15 / 0.14 / 0.51 ms against 0.21 / 0.19 / 0.88 ms at 16 per SM)
    const int multi_chains = (budget_ms <= 0 && max_steps <= 0 && w <= 32 && h <= 32) ? e->prop.multiProcessorCount * 4 : 0;
    tss_search_params p{seed, (only_1x1 && w <= 32 && h <= 32) ? want_chains : multi_chains, 0, -1, kernel};
    tss_search* s = nullptr;
    e->stats.interrupted = 0;
    e->stats.best_count = -1;
    int rc = TSS_OK;
    if (e->cached_search && only_1x1 && w > 0 && h > 0 && w <= 32 && h <= 32 && e->cached_search->n_chains != want_chains) {  // sized for another grid class / mode
        // (calls that do not use the 1x1 workspace — other platform sets, grids beyond 32x32 — leave it alone: a REPL / GUI that
        // alternates platform sets must not pay a free + cudaMalloc per call)
        search_free(e->cached_search);
        e->cached_search = nullptr;
    }
    int64_t fused_steps = 0;   // steps already executed by the fused first epoch
    int fused_best = -1;
    if (e->cached_search && grid && w > 0 && h > 0 && w <= 32 && h <= 32 && only_1x1 && plain) {
        // reuse the engine's workspace: same buffers, fresh terrain / reach table / chain states (no allocation)
        TSS_CUDA(e, cudaSetDevice(e->device));   // (before the workspace is detached: an early return must not leak it)
        s = e->cached_search;
        e->cached_search = nullptr;
        reuse_for_terrain(s, grid, w, h, seed);
        s->kernel = kernel;
        uint32_t rows_now[32];
        pack_rows32(grid, w, h, rows_now);
        if (latency_mode && s->n_chains % 8 == 0 && !e->interrupted()) {
            // the whole first epoch in ONE launch and ONE synchronisation (sls_h16.cu OneShot): rows travel as kernel
            // parameters, the reach table is derived per CTA, chains start in registers, the last CTA publishes the winner
            // and its validation into mapped host memory
            fused_steps = 32;   // (profiles/steps_to_optimum.py: the fastest of SM x 16 chains needs 16-32 steps on rect 16x16 and test/ex2)
            rc = fused_epoch_begin(e, s);
            if (rc == TSS_OK)
                rc = fused_epoch_end(e, sls_run_h16_oneshot(e, rows_now, card_limit >= 0 ? card_limit + 1 : sls::NO_BOUND, s->rows_dev, s->tabs_dev, s->states,
                                                            s->n_chains, seed, fused_steps, s->bounds_dev, s->best_dev, s->reduce_key_dev, s->ticket_dev,
                                                            card_limit >= 0 ? card_limit : sls::NO_BOUND - 1, s->noise, s->totals_dev, s->oneshot_host_dev));
            if (rc == TSS_OK) {   // (OneShot's result block, sls_h16.cu: [34] best, [35] chain, [36..41] totals)
                const volatile uint32_t* r = s->oneshot_host;
                for (int i = 0; i < 3; i++) s->totals_host[i] = ((unsigned long long)r[37 + 2 * i] << 32) | r[36 + 2 * i];
                fold_totals(e, s, s->totals_host[0], s->totals_host[1], s->totals_host[2]);
                s->best_host[0] = make_int2((int)r[34], (int)r[35]);
                if ((int)r[34] < sls::NO_BOUND) {
                    fused_best = (int)r[34];
                    e->stats.best_count = fused_best;
                    if (r[32] != 0 || (int)r[33] != fused_best)
                        rc = e->fail(TSS_E_CUDA, "internal error: SLS witness failed validation (%u unsupported tiles, %u supports, expected %d)", r[32], r[33], fused_best);
                }
            }
        } else {
            s->totals_seen[0] = s->totals_seen[1] = s->totals_seen[2] = 0;
            s->dirty = false;
            uint32_t* rows = (uint32_t*)e->pin(2, sizeof(uint32_t) * 32);
            if (!rows) rc = TSS_E_CUDA;
            if (rc == TSS_OK) {
                for (int y = 0; y < 32; y++) rows[y] = rows_now[y];
                cudaError_t err = cudaMemcpyAsync(s->rows_dev, rows, sizeof(uint32_t) * 32, cudaMemcpyHostToDevice, e->stream);
                rc = err == cudaSuccess ? search_init_device(e, s, 1) : e->fail(TSS_E_CUDA, "tss_solve_upper_bound: %s", cudaGetErrorString(err));
            }
        }
        if (rc != TSS_OK) { search_free(s); return rc; }
    } else if (!only_1x1 && plain && multi_chains > 0 && grid && defs && w > 0 && h > 0 && e->cached_multi && e->cached_multi->n_chains == multi_chains &&
               !e->interrupted()) {
        // placement search, first-model mode, workspace of the SAME platform set cached (keys, costs and their order are
        // already on the device): the first epoch as one fused launch (sls_multi.cu OneShotM)
        std::vector<int2> kd;
        std::vector<tss_platform> kp;
        build_keys(defs, n_defs, kd, kp);
        tss_search* c = e->cached_multi;
        bool same = kd.size() == c->key_dims.size();
        for (size_t i = 0; same && i < kd.size(); i++) same = kd[i].x == c->key_dims[i].x && kd[i].y == c->key_dims[i].y && c->key_costs[i] == 1;
        if (same) {
            s = c;
            e->cached_multi = nullptr;
            reuse_for_terrain(s, grid, w, h, seed);
            uint32_t rows_now[32];
            pack_rows32(grid, w, h, rows_now);
            fused_steps = 16;
            rc = cudaSetDevice(e->device) == cudaSuccess ? fused_epoch_begin(e, s) : e->fail(TSS_E_CUDA, "tss_solve_upper_bound: cudaSetDevice failed");
            if (rc == TSS_OK)
                rc = fused_epoch_end(e, slsm_run_oneshot(e, rows_now, card_limit >= 0 ? card_limit + 1 : sls::NO_BOUND, s->rows_dev, w, h, s->keys_dev, s->costs_dev,
                                                         s->costs_dev + slsm_max_keys(), (int)s->key_dims.size(), s->mstates, s->n_chains, seed, fused_steps,
                                                         s->bounds_dev, s->best_dev, s->reduce_key_dev, s->ticket_dev, card_limit >= 0 ? card_limit : sls::NO_BOUND - 1,
                                                         s->noise, s->totals_dev, s->oneshot_host_dev));
            if (rc == TSS_OK) {   // (OneShotM's result block, sls_multi.cu: [0] best, [1] chain, [2] n, [3..5] validation, [6..11] totals, codes from word 16)
                const volatile uint32_t* r = s->oneshot_host;
                for (int i = 0; i < 3; i++) s->totals_host[i] = ((unsigned long long)r[7 + 2 * i] << 32) | r[6 + 2 * i];
                fold_totals(e, s, s->totals_host[0], s->totals_host[1], s->totals_host[2]);
                s->best_host[0] = make_int2((int)r[0], (int)r[1]);
                if ((int)r[0] < sls::NO_BOUND) {   // hand the witness to the common tail in the layout of the in-stream witness buffers
                    fused_best = (int)r[0];
                    e->stats.best_count = fused_best;
                    const int n = (int)r[2] < slsm_max_items() ? (int)r[2] : slsm_max_items();
                    const volatile uint16_t* codes = reinterpret_cast<const volatile uint16_t*>(s->oneshot_host + 16);
                    for (int i = 0; i < n; i++) s->mw_codes_host[i] = codes[i];
                    s->mw_misc_host[0] = 0; s->mw_misc_host[1] = r[2];
                    s->mw_misc_host[4] = r[3]; s->mw_misc_host[5] = r[2]; s->mw_misc_host[6] = r[4]; s->mw_misc_host[7] = r[5];
                }
            }
            if (rc != TSS_OK) { search_free(s); return rc; }
        }
    }
    if (!s && limited && (w > 32 || h > 32)) {   // per-type limits on a large grid: the window placement search, limits fixed at creation
        p.kernel = TSS_KERNEL_AUTO;
        rc = tss_search_create_with_limits(e, grid, w, h, defs, n_defs, card, n_card, &p, &s);
        if (rc) return rc;
    }
    if (!s) {
        rc = tss_search_create(e, grid, w, h, defs, n_defs, &p, &s);
        if (rc) return rc;
    }
    s->share = false;  // a one-shot solve runs a rank-local number of epochs: no collective inside
    if (n_weights > 0) rc = tss_search_set_weights(s, weights, n_weights);
    if (rc == TSS_OK && limited && !s->lnsp) rc = tss_search_set_card_limits(s, card, n_card);
    if (rc == TSS_OK && card_limit >= 0 && fused_steps == 0) rc = tss_search_set_bound(s, card_limit + 1);   // (the fused epoch took its bound as a parameter)
    const double t0 = now_ms();
    // no budget given: behave like one SAT call (return the first model within the bound), but give up after a
    // default effort — the engine cannot prove UNSAT, so "no model found" must not turn into an endless search
    const bool windowed = w > 32 || h > 32;  // the window-decomposed search always holds a complete layout: keep improving it
    const bool first_model_only = budget_ms <= 0 && max_steps <= 0 && !(windowed && card_limit < 0);
    if (budget_ms <= 0 && max_steps < 0) max_steps = -max_steps;   // SAT-like call with a caller-chosen give-up point
    else if (budget_ms <= 0 && max_steps == 0) max_steps = windowed ? (1 << 16) : (1 << 18);
    // (a placement-search step costs ~5 us of latency: start with short epochs when the first model is all that is asked for)
    int64_t done_steps = fused_steps, epoch = fused_steps ? 2 * fused_steps : ((s->multi && first_model_only) ? 16 : (first_model_only && !s->lns ? 32 : 64));
    int best = fused_best;
    const bool in_stream_witness = !s->lns && !s->lnsp && !s->multi && s->n_groups == 1;   // 1x1 supports on a grid up to 32x32
    // First-model mode: chains stop at the first layout within the limit (target = card_limit).  (Queueing several epochs
    // per synchronisation — later ones do nothing once the bound is within the target, sls_spec.hpp — was measured and lost:
    // ~20 us of launch / event / copy calls per queued epoch against ~15 us per synchronisation.)
    const int target = first_model_only ? (card_limit >= 0 ? card_limit : sls::NO_BOUND - 1) : 0;
    const bool fused_hit = fused_best >= 0;   // first_model_only holds in latency mode: the fused epoch's layout is the answer
    while (rc == TSS_OK && !fused_hit) {
        if (e->interrupted()) { e->stats.interrupted = 1; break; }
        int64_t steps = epoch;
        if (max_steps > 0 && done_steps + steps > max_steps) steps = max_steps - done_steps;
        if (steps <= 0) break;
        rc = tss_search_run(s, steps, target);
        if (rc) break;
        done_steps += steps;
        if (epoch < 8192) epoch *= 2;
        if (s->multi) {  // placements of the best chain + their validation by the platform evaluator, in-stream
            rc = slsm_witness(e, s->mstates, s->best_dev, s->keys_dev, s->mw_codes_dev, s->mw_plats_dev, s->mw_misc_dev);
            if (rc == TSS_OK) rc = launch_eval_platforms(e, s->rows_dev, w, h, s->mw_plats_dev, s->mw_misc_dev, 1, (int32_t*)(s->mw_misc_dev + 4), nullptr, nullptr, nullptr);
            if (rc) break;
            cudaError_t err = cudaMemcpyAsync(s->mw_codes_host, s->mw_codes_dev, sizeof(uint16_t) * (size_t)slsm_max_items(), cudaMemcpyDeviceToHost, e->stream);
            if (err == cudaSuccess) err = cudaMemcpyAsync(s->mw_misc_host, s->mw_misc_dev, sizeof(uint32_t) * 8, cudaMemcpyDeviceToHost, e->stream);
            if (err != cudaSuccess) { rc = e->fail(TSS_E_CUDA, "tss_solve_upper_bound: %s", cudaGetErrorString(err)); break; }
        }
        if (in_stream_witness) {  // best layout + its validation ride in the same stream: one synchronisation per epoch
            witness_kernel<<<1, 32, 0, e->stream>>>(s->states, s->best_dev, s->rows_dev, s->witness_dev);
            e->stats.kernel_launches++;
            cudaError_t err = cudaMemcpyAsync(s->witness_host, s->witness_dev, sizeof(uint32_t) * 34, cudaMemcpyDeviceToHost, e->stream);
            if (err != cudaSuccess) { rc = e->fail(TSS_E_CUDA, "tss_solve_upper_bound: %s", cudaGetErrorString(err)); break; }
        }
        rc = tss_search_best_count(s, &best);
        if (rc) break;
        if (best == 0) break;
        if (first_model_only && best >= 0) break;
        if (budget_ms > 0 && now_ms() - t0 >= budget_ms) break;
    }
    e->stats.last_solve_steps = done_steps;
    if (rc == TSS_OK && best >= 0 && out_objective) *out_objective = best;
    int result = TSS_UNKNOWN;
    if (rc == TSS_OK && best >= 0 && in_stream_witness) {
        // the witness of the last epoch, already validated on the device (witness_kernel / the fused epoch's last CTA):
        // rows, unsupported tiles, supports
        const uint32_t* wr = fused_hit ? s->oneshot_host : s->witness_host;
        if (wr[32] != 0 || (int)wr[33] != best)
            rc = e->fail(TSS_E_CUDA, "internal error: SLS witness failed validation (%u unsupported tiles, %u supports, expected %d)", wr[32], wr[33], best);
        if (rc == TSS_OK) {
            if (n_out) *n_out = best;
            if (best > cap || !out) rc = e->fail(TSS_E_CAPACITY, "tss_solve_upper_bound: need room for %d platforms", best);
        }
        if (rc == TSS_OK) {
            int n = 0;
            for (int y = 0; y < h; y++)
                for (int x = 0; x < w; x++)
                    if ((wr[y] >> x) & 1u) out[n++] = tss_platform{x, y, 1, 1, 0};
            e->stats.layouts_evaluated++;
            result = TSS_SAT;
        }
    } else if (rc == TSS_OK && best >= 0 && s->multi) {
        // misc = {0, n, -, -, unsupported tiles, platforms, overlapping, out of bounds} (platform_layout.rs:187-191)
        const uint32_t* m = s->mw_misc_host;
        const int n = (int)m[1];
        int cost = 0;
        for (int i = 0; i < n && i < slsm_max_items(); i++) cost += s->key_costs[s->mw_codes_host[i] >> 10];
        if (m[4] != 0 || m[6] != 0 || m[7] != 0 || (int)m[5] != n || cost != best)
            rc = e->fail(TSS_E_CUDA, "internal error: SLS witness failed validation (%u unsupported tiles, %u overlapping, %u out of bounds, %d platforms costing %d, expected %d)",
                         m[4], m[6], m[7], n, cost, best);
        if (rc == TSS_OK) {
            if (n_out) *n_out = n;
            if (n > cap || !out) rc = e->fail(TSS_E_CAPACITY, "tss_solve_upper_bound: need room for %d platforms", n);
        }
        if (rc == TSS_OK) {
            codes_to_platforms(s, s->mw_codes_host, n, out);
            result = TSS_SAT;
        }
    } else if (rc == TSS_OK && best >= 0) {
        int n = 0;
        rc = tss_search_best_layout(s, out, cap, &n);
        if (n_out) *n_out = n;
        if (rc == TSS_OK) result = TSS_SAT;
    }
    keep_or_destroy(e, s, rc);
    return rc != TSS_OK ? rc : result;
}

int tss_solve_upper_bound(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                          int32_t card_limit, uint64_t seed, int32_t budget_ms, int64_t max_steps, tss_platform* out,
                          int32_t cap, int32_t* n_out) {
    return solve_search(e, grid, w, h, defs, n_defs, card_limit, nullptr, 0, nullptr, 0, seed, budget_ms, max_steps, out, cap, n_out, nullptr);
}

int tss_solve_with_limits(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, const int32_t* card,
                          int32_t n_card, const int32_t* weights, int32_t n_weights, int64_t weight_limit, uint64_t seed, int32_t budget_ms,
                          int64_t max_steps, tss_platform* out, int32_t cap, int32_t* n_out, int64_t* out_objective) {
    if (!e) return TSS_E_INVALID;
    if (n_out) *n_out = 0;
    if (!grid || w <= 0 || h <= 0 || n_defs < 0 || (n_defs > 0 && !defs) || n_card < 0 || (n_card > 0 && !card) || n_weights < 0 || (n_weights > 0 && !weights))
        return e->fail(TSS_E_INVALID, "tss_solve_with_limits: bad arguments");
    int32_t count_limit = -1;   // PlatformLimits.card_limits[1x1]: the platform count
    std::vector<int32_t> other;
    for (int i = 0; i < n_card; i++) {
        if (card[3 * i + 2] < 0) return e->fail(TSS_E_INVALID, "tss_solve_with_limits: negative limit for %dx%d", card[3 * i], card[3 * i + 1]);
        if (card[3 * i] == 1 && card[3 * i + 1] == 1) count_limit = count_limit < 0 ? card[3 * i + 2] : std::min(count_limit, card[3 * i + 2]);
        else other.insert(other.end(), card + 3 * i, card + 3 * i + 3);
    }
    if (n_weights > 0 && count_limit >= 0)
        return e->fail(TSS_E_UNSUPPORTED, "tss_solve_with_limits: the search minimises one objective: total weight or the platform count, not both");
    // A limit of 0 removes its class from the platform set, exactly as a smaller --platforms would: the reduced set runs the
    // kernels of that set (down to the 1x1 search), and only positive limits reach the placement search's class counters.
    std::vector<int2> kd;
    std::vector<tss_platform> kp;
    std::vector<uint32_t> mask;
    std::vector<int> lim;
    build_keys(defs, n_defs, kd, kp);
    const int n_other = (int)other.size() / 3;
    int rc = card_limit_classes(kd, other.data(), n_other, mask, lim);
    if (rc) return e->fail(rc, "tss_solve_with_limits: bad limit records");
    uint32_t zero = 0;   // classes with limit 0
    for (size_t j = 0; j < lim.size(); j++) zero |= lim[j] == 0 ? 1u << j : 0u;
    std::vector<tss_dims> kept;
    for (int i = 0; i < n_defs; i++) {
        bool drop = false;
        for (size_t k = 0; k < kd.size(); k++) drop = drop || (kd[k].x == defs[i].w && kd[k].y == defs[i].h && (mask[k] & zero));
        if (!drop) kept.push_back(defs[i]);
    }
    return solve_search(e, grid, w, h, kept.data(), (int32_t)kept.size(), n_weights > 0 ? weight_limit : (int64_t)count_limit, weights, n_weights,
                        other.data(), n_other, seed, budget_ms, max_steps, out, cap, n_out, out_objective);
}

int tss_lower_bound(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, uint64_t seed,
                    int32_t restarts, int32_t* out_xy, int32_t cap, int32_t* n_out) {
    if (!e) return TSS_E_INVALID;
    if (n_out) *n_out = 0;
    if (!grid || !n_out || w <= 0 || h <= 0 || (!defs && n_defs > 0) || cap < 0 || (cap > 0 && !out_xy)) return e->fail(TSS_E_INVALID, "tss_lower_bound: bad arguments");
    bool only_1x1 = true;
    if (int rc = check_defs(e, defs, n_defs, "tss_lower_bound", &only_1x1)) return rc;
    TSS_CUDA(e, cudaSetDevice(e->device));
    if (w > 32 || h > 32) {   // whole-board packing in parallel rounds (lb.cu), 1x1 supports
        if (!only_1x1) return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound: grids larger than 32x32 are supported with 1x1 supports only");
        BitGrid bg = BitGrid::from_bytes(grid, w, h);
        std::vector<uint32_t> pack(bg.rows.size());
        int count = 0;
        int rc = lb_run_big(e, bg.rows.data(), w, h, seed, restarts, pack.data(), &count);
        if (rc) return rc;
        *n_out = count;
        if (count > cap) return cap == 0 ? TSS_OK : e->fail(TSS_E_CAPACITY, "tss_lower_bound: need room for %d tiles", count);
        int n = 0;
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++)
                if ((pack[(size_t)y * bg.wpr + (x >> 5)] >> (x & 31)) & 1u) { out_xy[2 * n] = x; out_xy[2 * n + 1] = y; n++; }
        return TSS_OK;
    }
    std::vector<int2> key_dims;
    std::vector<tss_platform> key_proto;
    const tss_dims one{1, 1};
    build_keys(n_defs ? defs : &one, n_defs ? n_defs : 1, key_dims, key_proto);
    uint32_t rows[32], pack[32];
    pack_rows32(grid, w, h, rows);
    int count = 0;
    int rc = lb_run(e, rows, w, h, key_dims, seed, restarts, pack, &count);
    if (rc) return rc;
    *n_out = count;
    if (count > cap) return cap == 0 ? TSS_OK : e->fail(TSS_E_CAPACITY, "tss_lower_bound: need room for %d tiles", count);
    int n = 0;
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++)
            if ((pack[y] >> x) & 1u) { out_xy[2 * n] = x; out_xy[2 * n + 1] = y; n++; }
    return TSS_OK;
}

// The fractional bound of tss_lower_bound_lp and tss_lower_bound_lp_limits: key_mask / class_limit = classes of per-type limits
// on the keys of `defs` (card_limit_classes; empty: the plain LP, which is all grids larger than 32x32 take).
static int lower_bound_lp(tss_engine* e, const char* fn, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                          const std::vector<uint32_t>& key_mask, const std::vector<int>& class_limit, const int32_t* weights, int32_t n_weights,
                          int32_t max_pivots, int64_t target, int32_t* out_weights, int32_t* out_class_weights, int64_t* out_total,
                          int64_t* out_max_load, int64_t* out_bound, int32_t* out_info) {
    if (int rc = check_defs(e, defs, n_defs, fn, nullptr)) return rc;
    TSS_CUDA(e, cudaSetDevice(e->device));
    std::vector<int2> key_dims;
    std::vector<tss_platform> key_proto;
    const tss_dims one{1, 1};
    build_keys(n_defs ? defs : &one, n_defs ? n_defs : 1, key_dims, key_proto);
    std::vector<int> key_costs(key_dims.size(), 1);   // 1: the platform count
    if (n_weights > 0)
        for (size_t k = 0; k < key_dims.size(); k++) {
            const long cost = key_cost(key_proto[k], weights, n_weights);
            if (cost < 0 || cost > 4096)
                return e->fail(TSS_E_UNSUPPORTED, "%s: platform costs must be in 0..4096 (got %ld for %dx%d)", fn, cost, key_proto[k].def_w, key_proto[k].def_h);
            key_costs[k] = (int)cost;
        }
    if (out_class_weights) std::fill(out_class_weights, out_class_weights + kLpMaxClasses, 0);
    if (w > 32 || h > 32) {   // first-order method on the whole grid (lp_big.cu), the same certificate
        BitGrid bg = BitGrid::from_bytes(grid, w, h);
        std::vector<int> wts((size_t)w * h);
        int info[3];
        unsigned long long totals[3];
        int rc = lp_big_run(e, bg.rows.data(), w, h, key_dims, key_costs, max_pivots, target, wts.data(), totals, info);
        if (rc) return rc;
        if (out_weights) std::copy(wts.begin(), wts.end(), out_weights);
        if (out_total) *out_total = (int64_t)totals[0];
        if (out_max_load) *out_max_load = (int64_t)totals[1];
        if (out_info) { out_info[0] = info[0]; out_info[1] = info[1]; out_info[2] = info[2]; }
        *out_bound = (totals[1] > 0 && totals[2] != ~0ull) ? (int64_t)totals[2] : 0;
        return TSS_OK;
    }
    uint32_t rows[32];
    pack_rows32(grid, w, h, rows);
    int wts[1024 + kLpMaxClasses], info[3];
    unsigned long long totals[3];
    int rc = lp_run(e, rows, w, h, key_dims, key_costs, key_mask, class_limit, max_pivots, target, wts, totals, info);
    if (rc) return rc;
    if (target > 0 && !info[1] && !(totals[1] > 0 && totals[2] != ~0ull && (int64_t)totals[2] >= target)) {
        // stopped early on the floating-point objective, and the integer certificate falls short of the target: run to optimality
        rc = lp_run(e, rows, w, h, key_dims, key_costs, key_mask, class_limit, max_pivots, 0, wts, totals, info);
        if (rc) return rc;
    }
    if (out_weights)
        for (int y = 0; y < h; y++)
            for (int x = 0; x < w; x++) out_weights[(size_t)y * w + x] = wts[y * 32 + x];
    if (out_class_weights) std::copy(wts + 1024, wts + 1024 + kLpMaxClasses, out_class_weights);
    if (out_total) *out_total = (int64_t)totals[0];   // (V: signed, negative when the classes outweigh the tiles)
    if (out_max_load) *out_max_load = (int64_t)totals[1];
    if (out_info) { out_info[0] = info[0]; out_info[1] = info[1]; out_info[2] = info[2]; }
    *out_bound = (totals[1] > 0 && totals[2] != ~0ull) ? (int64_t)totals[2] : 0;   // min over placements of ceil(V * cost / load): exact
    return TSS_OK;
}

int tss_lower_bound_lp(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, const int32_t* weights,
                       int32_t n_weights, int32_t max_pivots, int64_t target, int32_t* out_weights, int64_t* out_total, int64_t* out_max_load,
                       int64_t* out_bound, int32_t* out_info) {
    if (!e) return TSS_E_INVALID;
    if (out_bound) *out_bound = 0;
    if (!grid || !out_bound || w <= 0 || h <= 0 || (!defs && n_defs > 0) || n_weights < 0 || (n_weights > 0 && !weights))
        return e->fail(TSS_E_INVALID, "tss_lower_bound_lp: bad arguments");
    return lower_bound_lp(e, "tss_lower_bound_lp", grid, w, h, defs, n_defs, {}, {}, weights, n_weights, max_pivots, target, out_weights, nullptr,
                          out_total, out_max_load, out_bound, out_info);
}

int tss_lower_bound_lp_limits(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, const int32_t* card,
                              int32_t n_card, const int32_t* weights, int32_t n_weights, int32_t max_pivots, int64_t target, int32_t* out_weights,
                              int32_t* out_class_weights, int64_t* out_total, int64_t* out_max_load, int64_t* out_bound, int32_t* out_info) {
    if (!e) return TSS_E_INVALID;
    if (out_bound) *out_bound = 0;
    if (!grid || !out_bound || w <= 0 || h <= 0 || (!defs && n_defs > 0) || n_card < 0 || (n_card > 0 && !card) || n_weights < 0 || (n_weights > 0 && !weights))
        return e->fail(TSS_E_INVALID, "tss_lower_bound_lp_limits: bad arguments");
    for (int i = 0; i < n_card; i++)
        if (card[3 * i + 2] < 0) return e->fail(TSS_E_INVALID, "tss_lower_bound_lp_limits: negative limit for %dx%d", card[3 * i], card[3 * i + 1]);
    if (int rc = check_defs(e, defs, n_defs, "tss_lower_bound_lp_limits", nullptr)) return rc;
    // the classes on the whole set; a limit of 0 then removes its class from the set, as tss_solve_with_limits does, and the
    // classes are taken again on what is left (the zero-limit records are vacuous there)
    const tss_dims one{1, 1};
    const tss_dims* all = n_defs ? defs : &one;
    const int n_all = n_defs ? n_defs : 1;
    std::vector<int2> kd;
    std::vector<tss_platform> kp;
    std::vector<uint32_t> mask;
    std::vector<int> lim;
    build_keys(all, n_all, kd, kp);
    int rc = card_limit_classes(kd, card, n_card, mask, lim);
    if (rc) return e->fail(rc, "tss_lower_bound_lp_limits: bad limit records");
    if (!lim.empty() && (w > 32 || h > 32))
        return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound_lp_limits: per-type limits on grids larger than 32x32 are not supported (got %dx%d)", w, h);
    uint32_t zero = 0;
    for (size_t j = 0; j < lim.size(); j++) zero |= lim[j] == 0 ? 1u << j : 0u;
    std::vector<tss_dims> kept;
    for (int i = 0; i < n_all; i++) {
        bool drop = false;
        for (size_t k = 0; k < kd.size(); k++) drop = drop || (kd[k].x == all[i].w && kd[k].y == all[i].h && (mask[k] & zero));
        if (!drop) kept.push_back(all[i]);
    }
    if (zero) {
        build_keys(kept.data(), (int)kept.size(), kd, kp);
        rc = card_limit_classes(kd, card, n_card, mask, lim);
        if (rc) return e->fail(rc, "tss_lower_bound_lp_limits: bad limit records");
    }
    return lower_bound_lp(e, "tss_lower_bound_lp_limits", grid, w, h, kept.data(), (int32_t)kept.size(), mask, lim, weights, n_weights, max_pivots, target,
                          out_weights, out_class_weights, out_total, out_max_load, out_bound, out_info);
}

int tss_solve_batch(tss_engine* e, const uint8_t* grids, int32_t w, int32_t h, int64_t n, uint64_t seed, int64_t steps,
                    int32_t chains_per_terrain, int32_t* out_counts, uint32_t* out_layouts) {
    if (!e) return TSS_E_INVALID;
    if (!grids || !out_counts || w <= 0 || h <= 0 || n < 0 || steps <= 0 || chains_per_terrain < 0)
        return e->fail(TSS_E_INVALID, "tss_solve_batch: bad arguments");
    if (w > 32 || h > 32) return e->fail(TSS_E_UNSUPPORTED, "tss_solve_batch: terrains larger than 32x32 are not accelerated yet");
    TSS_CUDA(e, cudaSetDevice(e->device));
    const int per_cta = h <= 16 ? 8 : 4;     // chains of one CTA (two chains per warp when the grid has <= 16 rows)
    const int CPT = chains_per_terrain <= 0 ? per_cta : ((chains_per_terrain + per_cta - 1) / per_cta) * per_cta;
    const int64_t CHUNK = 32768 / (CPT / per_cta) > 256 ? 32768 / (CPT / per_cta) : 256;  // terrains per pass (reach tables: 8 KB each)
    const size_t tiles = (size_t)w * h;
    e->stats.interrupted = 0;
    double dev_ms = 0;
    // one workspace for the whole call, kept on the engine for the next call (allocation dominated the first version)
    const int nt_max = (int)(n < CHUNK ? n : CHUNK);
    tss_search* s = e->cached_batch;
    e->cached_batch = nullptr;
    if (s && (s->cap_terrains < nt_max || s->cap_chains < nt_max * CPT)) { search_free(s); s = nullptr; }
    if (!s && nt_max > 0) {
        s = new tss_search();
        s->e = e;
        s->n_chains = s->cap_chains = nt_max * CPT;
        s->n_groups = s->cap_terrains = nt_max;
        int rc = search_alloc(e, s, nullptr, nt_max);
        if (rc != TSS_OK) { search_free(s); return rc; }
    }
    int rc = TSS_OK;
    for (int64_t base = 0; base < n && rc == TSS_OK; base += CHUNK) {
        if (e->interrupted()) break;
        const int nt = (int)((n - base) < CHUNK ? (n - base) : CHUNK);
        s->w = w; s->h = h; s->seed = seed; s->chain_offset = (uint32_t)(base * CPT);
        s->n_chains = nt * CPT; s->n_groups = nt; s->chains_per_terrain = CPT;
        s->totals_seen[0] = s->totals_seen[1] = s->totals_seen[2] = 0;
        s->dirty = false;
        uint8_t* bytes = (uint8_t*)e->dev(0, tiles * (size_t)nt);
        if (!bytes) { rc = TSS_E_CUDA; break; }
        cudaError_t err = cudaMemcpyAsync(bytes, grids + (size_t)base * tiles, tiles * (size_t)nt, cudaMemcpyHostToDevice, e->stream);
        if (err != cudaSuccess) { rc = e->fail(TSS_E_CUDA, "tss_solve_batch: %s", cudaGetErrorString(err)); break; }
        cudaEventRecord(e->ev2, e->stream);  // device time of the pass: terrains resident in HBM -> counts / layouts ready
        pack_rows32_kernel<<<e->prop.multiProcessorCount * 8, 256, 0, e->stream>>>(bytes, w, h, nt, s->rows_dev);
        e->stats.kernel_launches++;
        rc = search_init_device(e, s, nt);
        // epochs of 1024 steps so the chains of a terrain share their bound and an interrupt is honoured
        for (int64_t done = 0; rc == TSS_OK && done < steps; done += 1024) {
            if (e->interrupted()) break;
            rc = tss_search_run(s, (steps - done) < 1024 ? (steps - done) : 1024, 0);
        }
        uint32_t* rows_dev = nullptr;
        uint32_t* rows_host = nullptr;
        if (rc == TSS_OK && out_layouts) {  // gather the winners' rows on the device: 128 B per terrain instead of every chain state
            rows_dev = (uint32_t*)e->dev(1, sizeof(uint32_t) * 32 * (size_t)nt);
            rows_host = (uint32_t*)e->pin(3, sizeof(uint32_t) * 32 * (size_t)nt);
            if (!rows_dev || !rows_host) { rc = TSS_E_CUDA; break; }
            gather_best_rows_kernel<<<(nt * 32 + 255) / 256, 256, 0, e->stream>>>(s->states, s->best_dev, nt, rows_dev);
            e->stats.kernel_launches++;
            err = cudaMemcpyAsync(rows_host, rows_dev, sizeof(uint32_t) * 32 * (size_t)nt, cudaMemcpyDeviceToHost, e->stream);
            if (err != cudaSuccess) { rc = e->fail(TSS_E_CUDA, "tss_solve_batch: %s", cudaGetErrorString(err)); break; }
        }
        if (rc == TSS_OK) cudaEventRecord(e->ev3, e->stream);
        if (rc == TSS_OK) rc = search_sync(s);
        if (rc == TSS_OK) {
            float pass_ms = 0;
            if (cudaEventElapsedTime(&pass_ms, e->ev2, e->ev3) != cudaSuccess) cudaGetLastError();
            dev_ms += pass_ms;
            for (int t = 0; t < nt; t++) out_counts[base + t] = s->best_host[t].x >= sls::NO_BOUND ? -1 : s->best_host[t].x;
            if (out_layouts)
                for (int t = 0; t < nt; t++)
                    for (int y = 0; y < h; y++) out_layouts[(size_t)(base + t) * h + y] = rows_host[(size_t)t * 32 + y];
        }
    }
    if (s) {
        cudaStreamSynchronize(e->stream);
        s->n_chains = s->cap_chains;
        s->n_groups = s->cap_terrains;
        e->cached_batch = s;
    }
    if (rc != TSS_OK) return rc;
    if (e->interrupted()) e->stats.interrupted = 1;
    e->stats.device_ms = dev_ms;
    return e->interrupted() ? TSS_UNKNOWN : TSS_SAT;
}

int tss_measure_peaks(tss_engine* e, double* out, int32_t n_out) {
    if (!e) return TSS_E_INVALID;
    if (!out || n_out < 5) return e->fail(TSS_E_INVALID, "tss_measure_peaks: need room for 5 values");
    TSS_CUDA(e, cudaSetDevice(e->device));
    return run_peaks(e, out, n_out);
}

}  // extern "C"
