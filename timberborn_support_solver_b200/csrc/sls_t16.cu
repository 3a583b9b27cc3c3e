// Kernel (b), one chain per THREAD, for grids of at most 16 rows and 26 columns (rect 16x16, test/ex1-3).
//
// ncu on the warp-per-chain kernels (profiles/r1_sls_kernel.md, r1_sls_h16_kernel.md) shows the ALU pipe as the limiter
// with ~276 warp instructions per chain step, most of them cross-lane plumbing (indexed shuffles to fetch window rows,
// ballots, min/max butterflies) and per-chain "uniform" work that all lanes of a (half-)warp repeat.  Here a chain is
// one thread (sls_thread.cuh: the step, the keys, the site list and the removal ring shared with sls_p16.cu): every
// candidate layout is scored by that thread alone (7 row loads, shift/mask/pack, 2 AND+POPC), there are no shuffles,
// ballots or reductions in the step loop, and a warp instruction advances 32 layouts.
//
// The step rule, RNG and tie-breaks are EXACTLY those of sls_spec.hpp: the parity tests replay this kernel against the
// same CPU model as sls.cu / sls_h16.cu (bit-identical trajectories).  The representation:
//   * columns are stored shifted left by 3 and the reach windows re-anchored at x-3 when the table is loaded, so a
//     window row is always `(row >> x) & 0x7f` (no anchor clamp); the boards sit back to back and a row is one LDS at an
//     immediate offset from the site's row: rows outside the grid alias a neighbouring board, which is harmless because
//     they only ever meet zero window bits (reads) or a zero mask (no write);
//   * add candidates: the 13x13 neighbourhood of the uncovered tile is fetched once into registers; per column offset a
//     7-bit slab is masked once and the 25 diamond cells are scored with static shifts, packing on the FMA pipe.
// ncu (profiles/r1_sls_t16_kernel.md): 73 warp instructions per chain step, ALU pipe 75 %, issue slots 72 %, shared-memory
// wavefronts 17.8 per chain step (a third of them bank-conflict replays of the random 8-byte reach-table reads).
// r2: windows as one byte per row assembled with PRMT (the per-row `& 0x7f` and the multiply-packs are gone): 73 -> 65 warp
// instructions per chain step, 23.7 -> 24.6 G flips/s.  The kernel sits at ~75 % of BOTH the ALU pipe and the shared-memory pipe
// (0.75 wavefronts per clock and SM), which is why more resident warps do not help:
// Tried and dropped: the two high count planes in global memory for 4 CTAs per SM (r1: 277 vs 335 G candidates/s; r2, with a
// per-chain "never carried into them" flag so that they are not even read: 22.2 G flips/s at 3 CTAs, 20.4 G at 4 CTAs vs 24.6 G);
// skipping their shared-memory loads until some count reaches 8 (326 vs 334 G: the branches cost more than the loads).
#include "sls_thread.cuh"

namespace tss {
namespace slst {

using namespace tss::slsth;

constexpr int MAXW = 26;         // 3 + w + 3 <= 32 bits

struct Smem {
    uint2 tab[512 + 2 * TAB_PAD];          // reach windows of the 16x32 sites, anchored at x-3; entry of site v at v + TAB_PAD
    uint32_t C[24];                        // terrain rows, columns shifted by 3; row r at C[r + 3], zero outside the grid
    uint32_t rows[N_BOARDS * 16][NT];      // [board][row][thread]: bank = thread, conflict free for any row index
    uint16_t ring[32][NT];                 // site removed at step s in slot s & 31 (NONE if none)
};
constexpr int BOARD = 16 * NT;             // words between the same row of consecutive boards

// adds (ADD) or removes the cover of site v on the five count planes and refreshes U, O and the non-empty-row mask.
// rowmask is kept in padded coordinates: bit r + 3 = row r has an uncovered tile.
template <bool ADD>
__device__ __forceinline__ void flip(Smem& sm, int tid, int v, uint32_t& rowmask) {
    const int x = v & 31, y = v >> 5;
    const uint2 win = sm.tab[v + TAB_PAD];
    uint32_t* p = &sm.rows[0][tid] + y * NT;  // row y of the first board
    uint32_t nz = 0;
#pragma unroll
    for (int j = 0; j < 7; j++) {
        const uint32_t m7 = (j < 4 ? win.x >> (8 * j) : win.y >> (8 * (j - 4))) & 0xffu;
        const uint32_t Un = flip_word<ADD, BOARD>(sm, tid, p, (j - 3) * NT, m7 << x, m7, y + j);  // C[r + 3] = row r
        nz |= Un ? 1u << j : 0u;
    }
    rowmask = (rowmask & ~(0x7fu << y)) | (nz << y);
}

// low bytes of four / three words as one word (the fourth byte of pack3 is a copy of a's: it only ever meets a zero table byte)
__device__ __forceinline__ uint32_t pack4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}
__device__ __forceinline__ uint32_t pack3(uint32_t a, uint32_t b, uint32_t c) { return __byte_perm(__byte_perm(a, b, 0x0040), c, 0x0410); }

// rows of the support bitboard of a site list (rare path: recording a best layout, writing the state back)
__device__ __noinline__ void list_to_rows(const uint32_t* sl, size_t stride, int k, uint32_t* out32) {
    uint32_t rows[16];
    for (int r = 0; r < 16; r++) rows[r] = 0;
    for (int i = 0; i < k; i++) {
        const uint32_t v = sl[(size_t)i * stride] & 0x1ffu;
        rows[v >> 5] |= 1u << (v & 31u);
    }
    for (int r = 0; r < 16; r++) out32[r] = rows[r];
}

// U around the uncovered tile t = (x, y) of an addition: R[j] = row y-6+j, bit b = tile column b + x - 6
struct Nbhd {
    int x, y;
    const uint2* tabt;   // t's table entry
    uint2 wt;            // t's window
    uint32_t R[13];
    // the 7-bit column slab of U for column offset DX: P[j] = columns x+DX-3 .. x+DX+3 of row y-6+j
    using Slab = uint32_t[13];
    template <int DX, int M>
    __device__ __forceinline__ void slab(Slab& P) const {
#pragma unroll
        for (int j = 3 - M; j <= 9 + M; j++) P[j] = R[j] >> (DX + 3);   // (only the low byte is used; its bit 7 meets a zero table bit)
    }
    template <int DY>
    static __device__ __forceinline__ uint32_t gain(const Slab& P, uint2 win) {
        const uint32_t lo = pack4(P[DY + 3], P[DY + 4], P[DY + 5], P[DY + 6]);
        const uint32_t hi = pack3(P[DY + 7], P[DY + 8], P[DY + 9]);
        return (uint32_t)(__popc(lo & win.x) + __popc(hi & win.y));
    }
};

// the board representation of sls_t16_kernel for run_chains (sls_thread.cuh)
struct Rows {
    using Smem = slst::Smem;
    Smem& sm;
    const int tid;
    uint32_t* const sl;
    const size_t stride;
    uint32_t* const Ub;
    const uint32_t* const Ob;

    __device__ __forceinline__ Rows(Smem& sm, int tid, uint32_t* sl, size_t stride)
        : sm(sm), tid(tid), sl(sl), stride(stride), Ub(&sm.rows[B_U * 16][tid]), Ob(&sm.rows[B_O * 16][tid]) {}

    static __device__ __forceinline__ void load(Smem& sm, int tid, const uint32_t* terrain_rows, const uint2* rtabs, int terrain) {
        for (int i = tid; i < 512 + 2 * TAB_PAD; i += NT) {
            const int v = i - TAB_PAD;
            uint2 s = make_uint2(0u, 0u);
            if (v >= 0 && v < 512) {
                s = rtabs[(size_t)terrain * 1024 + v];
                const int x = v & 31, sh = x < 3 ? 3 - x : 0;  // table windows are anchored at max(x-3, 0): re-anchor at x-3
                s = byte_rows(make_uint2(s.x << sh, s.y << sh));
            }
            sm.tab[i] = s;
        }
        if (tid < 24) sm.C[tid] = (tid >= 3 && tid < 19) ? terrain_rows[(size_t)terrain * 32 + tid - 3] << 3 : 0u;
#pragma unroll 8
        for (int r = 0; r < N_BOARDS * 16; r++) sm.rows[r][tid] = 0;
#pragma unroll
        for (int r = 0; r < 32; r++) sm.ring[r][tid] = (uint16_t)NONE;
    }

    __device__ __forceinline__ int start(const uint32_t* S, uint32_t step, uint32_t& rowmask) {
        int k = 0;
        const uint32_t reset = (uint32_t)stamp_reset(step) << 16;
        for (int y = 0; y < 16; y++)
            for (uint32_t bits = S[y]; bits; bits &= bits - 1) sl[(size_t)(k++) * stride] = (uint32_t)(y * 32 + __ffs(bits) - 1) | reset;
        for (int r = 0; r < 16; r++) { const uint32_t c = sm.C[r + 3]; Ub[r * NT] = c; rowmask |= c ? 8u << r : 0u; }
        for (int i = 0; i < k; i++) flip<true>(sm, tid, (int)(sl[(size_t)i * stride] & 0x1ffu), rowmask);
        return k;
    }

    __device__ __forceinline__ void remove(uint32_t hs, uint32_t step, uint32_t stephi, uint32_t young_below, int k, uint32_t& rowmask) {
        uint32_t best_key = 0xffffffffu, mult = K3;                 // mult = (2i+1) * K3
#pragma unroll 4
        for (int i = 0; i < k; i++, mult += 2u * K3) {
            const uint32_t e = sl[(size_t)i * stride];
            const int v = (int)(e & 0x1ffu), x = v & 31;
            const uint2 win = sm.tab[v + TAB_PAD];
            const uint32_t* p = Ob + (v >> 5) * NT;
            uint32_t r7[7];
#pragma unroll
            for (int j = 0; j < 7; j++) r7[j] = ld(sm, p + (j - 3) * NT) >> x;
            const uint32_t lo = pack4(r7[0], r7[1], r7[2], r7[3]);
            const uint32_t hi = pack3(r7[4], r7[5], r7[6]);
            const uint32_t loss = (uint32_t)(__popc(lo & win.x) + __popc(hi & win.y));
            best_key = min(best_key, remove_key(e, i, loss, hs * mult, stephi, young_below));
        }
        const int best_i = (int)(best_key & 0x1ffu);
        const int u = (int)(sl[(size_t)best_i * stride] & 0x1ffu);
        sl[(size_t)best_i * stride] = sl[(size_t)(k - 1) * stride];
        sm.ring[step & 31u][tid] = (uint16_t)u;
        flip<false>(sm, tid, u, rowmask);
    }

    __device__ __forceinline__ Nbhd fetch(uint32_t rowmask, uint32_t hs) const {
        Nbhd N;
        N.y = pick_rotated(rowmask >> 3, hs & 31u);
        const uint32_t* Up = Ub + N.y * NT;
        N.x = pick_rotated(Up[0] >> 3, (hs >> 5) & 31u);
        N.tabt = &sm.tab[N.y * 32 + N.x + TAB_PAD];
        N.wt = N.tabt[0];
#pragma unroll
        for (int j = 0; j < 13; j++) N.R[j] = (ld(sm, Up + (j - 6) * NT) << 3) >> N.x;
        return N;
    }

    __device__ __forceinline__ void add(int v, uint32_t step, int k, uint32_t& rowmask) {
        flip<true>(sm, tid, v, rowmask);
        sl[(size_t)k * stride] = (uint32_t)v | (step << 16);
    }

    __device__ __forceinline__ void list_to_rows(int k, uint32_t* out32) const { slst::list_to_rows(sl, stride, k, out32); }
};

__global__ void __launch_bounds__(NT, 3) sls_t16_kernel(const uint32_t* __restrict__ terrain_rows, const uint2* __restrict__ rtabs,
                                                       ChainState* __restrict__ states, uint32_t* __restrict__ site_lists, size_t stride,
                                                       int n_chains, int chains_per_terrain, uint32_t chain_offset, uint64_t seed,
                                                       long long steps, const int* __restrict__ bounds, int target, int noise_pct,
                                                       const volatile int* interrupt, unsigned long long* __restrict__ totals) {
    run_chains<Rows>(threadIdx.x, terrain_rows, rtabs, states, site_lists, stride, n_chains, chains_per_terrain, chain_offset, seed, steps, bounds, target,
                     noise_pct, interrupt, totals);
}

}  // namespace slst

// violations counted by a -DTSS_CHECKED build since the library was loaded (always 0 in the shipped build, which has no checks)
int sls_t16_smem_violations() { return slst::smem_violations(); }
int sls_t16_checked_build() {
#ifdef TSS_CHECKED
    return 1;
#else
    return 0;
#endif
}
bool sls_t16_fits(int w, int h) { return h <= 16 && w <= slst::MAXW; }
int sls_thread_cta_chains() { return slsth::NT; }
size_t sls_t16_list_words(int n_chains) { return (size_t)16 * slst::MAXW * (((size_t)n_chains + 31) & ~(size_t)31); }

int sls_run_t16(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, uint32_t* site_lists, int n_chains,
                int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
                int noise_pct, unsigned long long* totals_dev) {
    return slsth::launch(slst::sls_t16_kernel, sizeof(slst::Smem), e, rows_dev, tabs_dev, states, site_lists, n_chains, chains_per_terrain,
                         chain_offset, seed, steps, bounds_dev, target, noise_pct, totals_dev);
}

}  // namespace tss
