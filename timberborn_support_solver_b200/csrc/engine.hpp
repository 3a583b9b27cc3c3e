// Engine internals shared by the CUDA translation units.  Not part of the ABI (see include/tss.h).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/tss.h"
#include "host_model.hpp"

namespace tss {
struct Comm;
void comm_destroy(Comm* c);
int comm_allreduce_min(tss_engine* e, Comm* c, int* dev, int n);  // in-stream ncclAllReduce(min) on device ints
int comm_allreduce_min_u32(tss_engine* e, Comm* c, const uint32_t* src, uint32_t* dst, int n);
int comm_allreduce_sum_u32(tss_engine* e, Comm* c, const uint32_t* src, uint32_t* dst, int n);
int comm_rank(const Comm* c);
int comm_world(const Comm* c);
}  // namespace tss

// A growable device (or pinned host) scratch buffer owned by the engine.
struct TssBuffer {
    void* ptr = nullptr;
    size_t cap = 0;
    bool pinned = false;
};

struct tss_engine {
    int device = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t stream = nullptr;  // own_stream or a caller-provided one
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;  // bracket the last kernel-level operation (epoch, evaluation)
    cudaEvent_t ev2 = nullptr, ev3 = nullptr;  // bracket a whole multi-epoch pass (tss_solve_batch chunk)
    cudaDeviceProp prop{};
    cudaMemPool_t pool = nullptr;   // stream-ordered allocations that come and go with every solver call (uploaded CNFs): cached, never returned to the OS while the engine lives
    std::string error;
    tss_stats stats{};
    // Interrupt flag polled by the search kernels.  It lives in DEVICE memory (an L2 hit per poll): polling a mapped
    // host flag costs a PCIe round trip per warp and serialises (measured r1: 3.5 ms per poll round of 4736 warps).
    // tss_interrupt() copies a pinned 1 into it on a dedicated non-blocking stream, from any thread.
    volatile int* interrupt_host = nullptr;  // pinned {0, 1} source words
    int* interrupt_dev = nullptr;            // device flag
    cudaStream_t irq_stream = nullptr;
    std::atomic<int> interrupt_flag{0};
    bool certified_unsat = true;             // tss_solve_instance may answer TSS_UNSAT from a certified lower bound (tss_engine_certified_unsat)
    bool limit_bounds = false;               // ... and asks the class-aware LP for instances with per-type limits (tss_engine_limit_bounds)
    bool window_limits = false;              // tss_solve_instance answers per-type instances on grids larger than 32x32 (tss_engine_window_limits)
    struct tss_search* cached_search = nullptr;  // workspace reused by tss_solve_upper_bound (no cudaMalloc per call)
    struct tss_search* cached_batch = nullptr;   // workspace reused by tss_solve_batch
    struct tss_search* cached_multi = nullptr;   // workspace of the placement search (platform sets beyond {1x1}) of a one-shot solve
    struct tss::Comm* comm = nullptr;            // NCCL communicator of a multi-GPU portfolio (comm.cu), or null
    TssBuffer scratch[8];                    // device scratch slots
    TssBuffer staging[6];                    // pinned host staging slots

    int fail(int code, const char* fmt, ...) {
        char buf[512];
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(buf, sizeof buf, fmt, ap);
        va_end(ap);
        error = buf;
        return code;
    }
    // returns nullptr and sets error on failure
    void* dev(int slot, size_t bytes);
    void* pin(int slot, size_t bytes);
    bool interrupted() const { return interrupt_flag.load(std::memory_order_relaxed) != 0; }
};

#define TSS_CUDA(e, call)                                                                              \
    do {                                                                                               \
        cudaError_t err__ = (call);                                                                    \
        if (err__ != cudaSuccess) return (e)->fail(TSS_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(err__), __FILE__, __LINE__); \
    } while (0)

#define TSS_CHECK_LAUNCH(e) TSS_CUDA(e, cudaGetLastError())

// Compact row format (tss.h tss_eval_compact_dev): row stride in bytes and layout stride padded to 4 bytes.
// Grids up to 32x32 use 1/2/4-byte rows; anything larger uses ceil(w/32) u32 words per row.
inline bool tss_is_small(int w, int h) { return w <= 32 && h <= 32; }
inline int tss_row_bits(int w) { return w <= 8 ? 8 : (w <= 16 ? 16 : 32); }
inline size_t tss_row_bytes(int w, int h) { return tss_is_small(w, h) ? (size_t)tss_row_bits(w) / 8 : (size_t)((w + 31) / 32) * 4; }
inline size_t tss_layout_bytes(int w, int h) { return (tss_row_bytes(w, h) * (size_t)h + 3) & ~(size_t)3; }

// ---- kernel launchers (defined in the .cu files), all asynchronous on e->stream
namespace tss {
// eval.cu — kernel (a)
int launch_eval_compact(tss_engine* e, const void* grid_dev, int w, int h, const void* layouts_dev, int64_t n,
                        bool per_layout_terrain, int32_t* out_dev);
// platform layouts: plats_dev records (x,y,w,h) effective dims; offsets_dev[n+1]; out_dev int32[n][4];
// optional single-layout extras: unsupported rows (packed h*wpr) and per-platform flags
int launch_eval_platforms(tss_engine* e, const uint32_t* grid_rows_dev, int w, int h, const int4* plats_dev,
                          const uint32_t* offsets_dev, int64_t n, int32_t* out_dev, uint32_t* unsupported_rows_dev,
                          uint8_t* flags_dev, uint32_t* layers_dev);
// packs u8 masks [n][w*h] into the compact row format on the device
int launch_pack_bytes(tss_engine* e, const uint8_t* bytes_dev, int w, int h, int64_t n, void* compact_dev);
// engine.cu — is this pointer an engine that has not been destroyed (handles that may outlive their engine ask before touching it)
bool engine_alive(const tss_engine* e);
// cnf.cu — one assignment completed (unit propagation, open variables False, every clause checked) in one launch
int cnf_complete_single(tss_engine* e, const struct ::tss_cnf* c, uint8_t* assignment, int32_t* conflict, int32_t* n_falsified);
// host helper: pack one u8 grid into compact rows
void pack_compact_host(const uint8_t* grid, int w, int h, uint8_t* out);
void rows_to_compact_host(const uint32_t* rows, int w, int h, uint8_t* out);
}  // namespace tss
