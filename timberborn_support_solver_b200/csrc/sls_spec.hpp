// Specification constants of the batched stochastic local search (kernel (b)); shared by sls.cu and by the CPU
// model in oracle/sls_model.cpp that the parity tests replay it against (the model re-declares the same values and
// a test compares them — the oracle never includes product headers).
//
// Problem (SURVEY.md §8a E5): with 1x1 supports the encoder's CNF is "choose S, every ceiling tile within geodesic
// distance <= 3 (through ceiling tiles) of a ceiling tile in S, |S| <= n" (src/encoder.rs:500-544, 619-667).
// A site's reach R(s) is the result of validate()'s three masked dilations from {s} (platform_layout.rs:127-141); it
// lives in the 7x7 window around s and is stored as 49 bits (row dy in bits [7*dy, 7*dy+7)).
//
// One chain = one layout = one warp.  Lane r owns grid row r: ceiling C, supports S, and the cover count of every tile
// as five bit-planes c0..c4 (a tile is covered by at most 25 sites).  uncovered U = C & ~(c0|..|c4), covered-once
// O = c0 & ~(c1|..|c4).
//
// A step with bound L (smallest complete count known at the start of the epoch, or the chain's own best):
//   1. k >= L                -> drop the support with the smallest loss (tiles only it covers), random ties
//   2. U empty               -> record (k, S) as the chain's best; done if k <= target
//   3. otherwise, if k == L-1 -> remove the min-loss support (supports added fewer than T steps ago only as a last
//      resort), then pick a random uncovered tile t and add the site v in R(t) with the largest gain |U & R(v)| (random
//      ties; sites removed fewer than T steps ago only as a last resort; with probability ~noise% a uniformly random
//      site of R(t) instead).  T is the chain's tabu tenure, see below.
//
// An epoch whose bound is already <= its target (a layout within the target was found in an earlier epoch, or the caller
// asked for nothing better than what is known) does nothing.
//
// Random numbers are counter based, one hash per step plus one multiply per candidate:
//   hs = fmix32(base ^ step*K1)          one word per (chain, step): bits 0-4 row rotation, 5-9 column rotation,
//                                        10-16 noise draw (7 bits, compared with noise_q7 = round(noise% * 1.28))
//   tie_add(hs, c)    = (hs * ((2c+1)*K2)) >> 16   breaks ties among ADD candidates, c = index in the 25-tile diamond
//   tie_remove(hs, i) = (hs * ((2i+1)*K3)) >> 16   breaks ties among REMOVE candidates, i = index in the site list
//   (multiplicative hashing of the step word by distinct odd constants; candidates that still tie are resolved to the
//   lowest index).  One multiply per candidate keeps the tie-break off the integer-ALU pipe, which bounds the kernels.
// base is keyed by (seed, global chain index), so a run is reproducible for a fixed chain numbering.
#pragma once
#include <cstdint>

namespace tss {
namespace sls {

constexpr uint32_t K1 = 0x9E3779B9u, K2 = 0x85EBCA6Bu, K3 = 0xC2B2AE35u;
constexpr int DEFAULT_NOISE_PCT = 20;
constexpr int MAX_SITES = 1024;   // supports per chain (<= tiles of a 32x32 grid)
constexpr int NO_BOUND = 1 << 20;
constexpr long long MAX_EPOCH_STEPS = 32768;  // steps per epoch (kernel launch): the 16-bit tabu stamps never wrap inside one

#if defined(__CUDACC__)
#define TSS_HD __host__ __device__ __forceinline__
#else
#define TSS_HD inline
#endif

TSS_HD uint32_t fmix32(uint32_t h) {
    h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16;
    return h;
}
TSS_HD uint32_t chain_base(uint64_t seed, uint32_t chain) {
    return fmix32((uint32_t)seed ^ fmix32((uint32_t)(seed >> 32) + chain * K1 + 0x5bd1e995u));
}
TSS_HD uint32_t step_hash(uint32_t base, uint32_t step) { return fmix32(base ^ (step * K1)); }
TSS_HD uint32_t lane_hash(uint32_t hs, uint32_t lane) { return fmix32(hs ^ ((lane + 1u) * K2)); }
TSS_HD uint32_t noise_q7(int noise_pct) { return (uint32_t)((noise_pct * 128 + 50) / 100); }
TSS_HD uint32_t tie_add(uint32_t hs, uint32_t cell) { return (hs * ((2u * cell + 1u) * K2)) >> 16; }
TSS_HD uint32_t tie_remove(uint32_t hs, uint32_t i) { return (hs * ((2u * i + 1u) * K3)) >> 16; }
TSS_HD uint32_t tie_remove_hl(uint32_t hl, uint32_t chunk) { return (hl * (2u * chunk + 1u)) >> 16; }  // placement search (sls_multi.cu)

// Tabu with tenure (the single most effective ingredient on fragmented terrains, see DESIGN.md): a site flipped
// (added or removed) fewer than T steps ago is tabu — a recently added support is not removed, a recently removed site
// not re-added — unless every candidate is tabu.  Implemented as a preference bit in the selection keys, so the fallback
// needs no second pass.  The flip step of every site is kept as a 16-bit stamp per chain (reset at the start of an epoch
// to "half a period ago"); the tenure is a portfolio parameter: chains use T = 3, 6, 12, 20 by global chain index.
constexpr uint32_t TABU_BIT = 0x40000000u;
TSS_HD int tenure_of(uint32_t global_chain) { return (global_chain & 3u) == 0 ? 3 : ((global_chain & 3u) == 1 ? 6 : ((global_chain & 3u) == 2 ? 12 : 20)); }
// ... capped at a third of the current support count (with k = 14 supports a tenure of 20 would freeze the search) but
// never below 2: the support added in the previous step is not removed, the site removed in this step not re-added.
TSS_HD int effective_tenure(int tenure, int k) { int c = k / 3; c = c < 2 ? 2 : c; return tenure < c ? tenure : c; }
TSS_HD uint16_t stamp_reset(uint32_t step) { return (uint16_t)(step - 0x8000u); }
TSS_HD bool is_tabu(uint32_t step, uint16_t stamp, int tenure) { return (uint16_t)((uint16_t)step - stamp) < (uint16_t)tenure; }

// Persistent per-chain state in HBM (one 288-byte record per chain, read once at the start of an epoch and written back at its end).
struct ChainState {
    uint32_t S[32];      // current supports, row r in S[r]
    uint32_t bestS[32];  // best complete layout found by this chain
    int32_t k;           // current number of supports
    int32_t best;        // supports in bestS, NO_BOUND if none yet
    uint32_t step;       // RNG step counter (persists across epochs)
    int32_t done;        // reached the target or nothing left to do
    uint32_t scored_lo, scored_hi;  // candidate layouts scored by this chain (64-bit counter)
    uint32_t steps_done;
    uint32_t reserved;   // (keeps the record a multiple of 16 bytes)
};
static_assert(sizeof(ChainState) == 288, "ChainState layout");

#if defined(__CUDACC__)
// The random uncovered tile of an addition: the first set bit of a row mask (then of the row) at or above offset o,
// wrapping around (bits rotated right by o).
__device__ __forceinline__ int pick_rotated(uint32_t bits, uint32_t o) {
    uint32_t rot = __funnelshift_r(bits, bits, o);
    return (int)((__ffs(rot) - 1 + o) & 31u);
}

// The 25-tile diamond |dx| + |dy| <= 3 of add candidates around t, cell index i in row-major order: window row r = dy + 3
// holds cells cell_start(r) .. cell_start(r + 1) - 1.
__device__ __forceinline__ constexpr int cell_start(int r) { return r <= 4 ? r * r : (r == 5 ? 21 : 24); }
__device__ __forceinline__ void diamond_cell(int i, int& dx, int& dy) {
    const int r = (i >= 1) + (i >= 4) + (i >= 9) + (i >= 16) + (i >= 21) + (i >= 24);
    dy = r - 3;
    dx = i - cell_start(r) - (3 - abs(dy));
}

// Reach window of site v = (x, y) on a terrain given as 32 row words: validate()'s three ceiling-masked dilations
// (src/encoder/platform_layout.rs:127-141) run inside the site's own 7x7 window (geodesic paths of length <= 3 never
// leave it).  Window row dy is grid row y-3+dy, window column 0 is grid column max(x-3, 0).
__device__ __forceinline__ uint2 reach_window(const uint32_t* C, int v) {
    const int x = v & 31, y = v >> 5, ax = x - 3 > 0 ? x - 3 : 0;
    uint32_t c[7], X[7];
#pragma unroll
    for (int j = 0; j < 7; j++) {
        const int yy = y - 3 + j;
        const uint32_t row = (yy >= 0 && yy < 32) ? C[yy] : 0u;
        c[j] = (row >> ax) & 0x7fu;
        X[j] = 0;
    }
    X[3] = c[3] & (1u << (x - ax));  // the site itself, if it is a ceiling tile
    for (int round = 0; round < 3; round++) {  // TERRAIN_SUPPORT_DISTANCE - 1 (src/lib.rs:12)
        uint32_t N[7];
#pragma unroll
        for (int j = 0; j < 7; j++) {
            uint32_t v2 = X[j] | (X[j] << 1) | (X[j] >> 1);
            if (j > 0) v2 |= X[j - 1];
            if (j < 6) v2 |= X[j + 1];
            N[j] = v2 & c[j];
        }
#pragma unroll
        for (int j = 0; j < 7; j++) X[j] = N[j];
    }
    return make_uint2(X[0] | (X[1] << 7) | (X[2] << 14) | (X[3] << 21), X[4] | (X[5] << 7) | (X[6] << 14));
}
#endif

}  // namespace sls
}  // namespace tss
