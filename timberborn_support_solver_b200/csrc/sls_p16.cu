// Kernel (b), one chain per THREAD with two grid rows per word, for grids of at most 16x16 (rect 16x16, test/ex1, test/ex3).
//
// sls_t16.cu sits at ~75 % of both the ALU pipe and the shared-memory pipe (65 warp instructions per chain step), so the
// only way to step faster is to issue fewer instructions per step.  On grids of at most 16 columns one 32-bit word holds
// two grid rows: word p of a board is row 2p in bits 0-15 and row 2p+1 in bits 16-31 (no column padding).  A 7-row
// reach window then spans four words instead of seven rows, and every shift, load and carry of the step works on two rows.
//
// The step rule, RNG and tie-breaks are EXACTLY those of sls_spec.hpp and of sls_t16.cu (bit-identical trajectories, the
// parity tests replay both against the same CPU model); the step, the site list, the removal ring and the selection keys
// are shared with it (sls_thread.cuh).  What differs is the representation:
//   * windows keep the spec's anchor ax = max(x-3, 0) (a 3-column shift would not fit in 16 bits).  `pair >> ax` leaves
//     row 2p's window in byte 0 and row 2p+1's in byte 2; four such words pack into the two table words with one PRMT
//     each.  Columns >= 16 and bit 7 of every byte only ever meet zero table bits, so what bleeds in from the other half
//     is harmless;
//   * a table entry is 8 bytes, one byte per row SLOT: slot i = row 2*p0 + i with p0 = floor((y-3)/2), so the window's
//     seven rows sit in slots s0 .. s0+6 with s0 = (y-3) & 1.  A second table holds every window shifted by one slot
//     (slot 1 - s0): see the addition scoring below;
//   * flips: the cover mask of a pair is the table's two row bytes for it at bits 0 and 16, shifted by ax (cannot spill
//     from row 2p into 2p+1: those columns are off the grid and their bits zero); the carry chain over c0..c4 then
//     updates two rows per instruction.  The uncovered-row mask stays one bit per row, so the row pick is t16's;
//   * addition scoring: the 13 rows around the uncovered tile t = (x, y) are fetched as 7 pairs that START AT ROW y-6
//     (8 loads, 7 PRMT with a selector chosen by y & 1): candidate (DX, DY) then starts at a static pair and half, and
//     one slab per DX (pairs >> max(x+DX-3, 0)) serves all of its DYs.  The table alignment a candidate needs differs
//     from its absolute one exactly when y is odd, hence the second table: the step picks the table base by y & 1.
//     t's own window (candidate validity) and the tabu window stay in t16's byte-per-row format around (x-3, y-3);
//   * the first CAP entries of the site list live in shared memory with their table windows ([slot][thread], bank =
//     thread), so the removal scan reads a scored support with two conflict-free loads at immediate offsets instead of a
//     global load and a bank-conflicting table read.  Entries at index >= CAP stay in the global list (dense warm starts).
#include "sls_thread.cuh"

namespace tss {
namespace slsp {

using namespace tss::slsth;

constexpr int MAXW = 16;         // columns per pair half
constexpr int MAXH = 16;
constexpr int NP = 8;            // pair words per board
constexpr int TAB_N = 512 + 2 * TAB_PAD;

constexpr int CAP = 16;          // site-list entries per chain kept in shared memory (k stays at 14-15 on rect 16x16)

struct Smem {
    uint2 tab[2][TAB_N];                   // [slot shift][site]: reach window of site v at tab[a][v + TAB_PAD], rows in slots s0 ^ a ..
    uint2 cwin[CAP][NT];                   // [slot][thread]: tab[0] window of list entry `slot`
    uint32_t cent[CAP][NT];                // [slot][thread]: list entry `slot` (format of `entry` below)
    uint32_t C[16];                        // terrain pairs; pair p at C[p + 2], zero outside the grid
    uint32_t rows[N_BOARDS * NP][NT];      // [board][pair][thread]: bank = thread, conflict free for any pair index
    uint16_t ring[32][NT];                 // site removed at step s in slot s & 31 (NONE if none)
};
constexpr int BOARD = NP * NT;             // words between the same pair of consecutive boards
// Exactly 3 CTAs per SM (as t16): 444 CTAs of the default portfolio then fill the 148 SMs evenly (the SM has 228 KB, of
// which 1 KB per resident CTA is reserved).
constexpr size_t SMEM_BYTES = sizeof(Smem);
static_assert(3 * (SMEM_BYTES + 1024) <= 228 * 1024 && 4 * (SMEM_BYTES + 1024) > 228 * 1024, "sls_p16 must fit exactly 3 CTAs per SM");

// a support-cache slot index (the slot's column is always the thread's own), bounds-checked in a -DTSS_CHECKED build
__device__ __forceinline__ int slot(int i) {
#ifdef TSS_CHECKED
    if ((unsigned)i >= (unsigned)CAP) { violation(); return 0; }
#endif
    return i;
}

// first pair of site v's window: floor((y - 3) / 2) for v = 32 y + x (x < 32 never carries into the quotient)
__device__ __forceinline__ int first_pair(int v) { return (v - 96) >> 6; }
__device__ __forceinline__ int anchor(int x) { return __viaddmax_s32_relu(x, -3, 0); }   // max(x - 3, 0), one VIADDMNMX
// bytes 0 and 2 of four words as one word (row 2p / 2p+1 windows of four pairs: slots 0..7 -> two table words)
__device__ __forceinline__ uint32_t pack_pairs(uint32_t a, uint32_t b) { return __byte_perm(a, b, 0x6420); }

// site-list entry: site v (bits 0-8), first_pair(v) + 2 (bits 9-12) and the step it was added (bits 16-31).  Bits 9-12
// are the byte offset of the window's first pair within a board, in units of one pair row (NT words = 512 bytes).  The
// tabu test (stephi - e) < ten << 16 only sees bits 16-31: what the low half holds cannot borrow into them.
static_assert(NT * sizeof(uint32_t) == 512, "entry() and removal_loss() take bits 9-12 of an entry as a byte offset of whole pair rows");
__device__ __forceinline__ uint32_t entry(int v, uint32_t stamp) { return (uint32_t)v | (uint32_t)((v + 32) >> 6) << 9 | stamp << 16; }

// removal loss of list entry e with window win: reach tiles that only its support covers
__device__ __forceinline__ uint32_t removal_loss(const Smem& sm, int tid, uint32_t e, uint2 win) {
    const int ax = anchor(e & 31);
    const uint32_t* p = reinterpret_cast<const uint32_t*>(reinterpret_cast<const char*>(&sm.rows[B_O * NP - 2][0]) + ((e & 0x1e00u) | (uint32_t)tid << 2));
    const uint32_t lo = pack_pairs(ld(sm, p) >> ax, ld(sm, p + NT) >> ax);
    const uint32_t hi = pack_pairs(ld(sm, p + 2 * NT) >> ax, ld(sm, p + 3 * NT) >> ax);
    return (uint32_t)(__popc(lo & win.x) + __popc(hi & win.y));
}

// Removal key of list entry e (index i, loss `loss`) in remove_key's order (young, loss, tie, index), one byte per field
// most significant first: young * 64 + loss (a reach window has at most 25 tiles), tie_remove(hs, i) in bytes 1-2, which are bytes 2-3 of
// hsm = hs * (2i+1) * K3, and i (a 16x16 list has at most 256 entries).  One IMAD and one PRMT instead of remove_key's
// shift, mask and merge on the integer-ALU pipe.
static_assert(MAXW * MAXH <= 256, "removal_key keeps a list index in one byte: a list holds at most one entry per site");
__device__ __forceinline__ uint32_t removal_key(uint32_t e, int i, uint32_t loss, uint32_t hsm, uint32_t stephi, uint32_t young_below) {
    const uint32_t x = loss * (1u << 24) + ((stephi - e) < young_below ? TABU_BIT | (uint32_t)i : (uint32_t)i);
    return __byte_perm(hsm, x, 0x7324);
}

// the least of N keys as a tree of mins: log2(N) dependent steps instead of N
template <int N>
__device__ __forceinline__ uint32_t tree_min(const uint32_t* key) {
    if constexpr (N == 1) return key[0];
    else return min(tree_min<N / 2>(key), tree_min<N / 2>(key + N / 2));
}

// adds (ADD) or removes the cover of site v (window win = its tab[0] entry) on the five count planes and refreshes U, O
// and the non-empty-row mask.
// rowmask is kept in padded coordinates: bit r + 4 = row r has an uncovered tile.
template <bool ADD>
__device__ __forceinline__ void flip(Smem& sm, int tid, int v, uint2 win, uint32_t& rowmask) {
    const int ax = anchor(v & 31), p0 = first_pair(v);
    uint32_t* p = &sm.rows[0][tid] + p0 * NT;  // pair p0 of the first board
    uint32_t nz = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t m8 = __byte_perm(j < 2 ? win.x : win.y, 0u, (j & 1) ? 0x4342 : 0x4140);   // slots 2j, 2j+1 at bits 0, 16
        const uint32_t Un = flip_word<ADD, BOARD>(sm, tid, p, j * NT, m8 << ax, m8, p0 + j + 2);
        nz |= ((Un & 0xffffu) ? 1u << (2 * j) : 0u) | ((Un >> 16) ? 2u << (2 * j) : 0u);
    }
    const int sh = 2 * p0 + 4;
    rowmask = (rowmask & ~(0xffu << sh)) | (nz << sh);
}

// rows of the support bitboard of a site list (rare path: recording a best layout, writing the state back)
// (entries below CAP in the thread's cache column `cached`, the rest in the global list)
__device__ __noinline__ void list_to_rows(const uint32_t* cached, const uint32_t* sl, size_t stride, int k, uint32_t* out32) {
    uint32_t rows[16];
    for (int r = 0; r < 16; r++) rows[r] = 0;
    for (int i = 0; i < k; i++) {
        const uint32_t v = (i < CAP ? cached[i * NT] : sl[(size_t)i * stride]) & 0x1ffu;
        rows[v >> 5] |= 1u << (v & 31u);
    }
    for (int r = 0; r < 16; r++) out32[r] = rows[r];
}

// U around the uncovered tile t = (x, y) of an addition: Q[i] = rows y-6+2i (bits 0-15) and y-5+2i (bits 16-31)
struct Nbhd {
    int x, y;
    const uint2* tabt;   // t's entry in the table whose slot alignment matches pairs from y-6 (the candidates' windows)
    uint2 wt;            // t's window
    uint32_t Q[7];
    // L[i] = packed slab of pairs i, i+1 (rows y-6+2i .. y-3+2i, columns from max(x+DX-3, 0)) for column offset DX
    using Slab = uint32_t[6];
    template <int DX, int M>
    __device__ __forceinline__ void slab(Slab& L) const {
        constexpr int ilo = (3 - M) >> 1, ihi = ((3 + M) >> 1) + 2;   // packed slabs L[ilo .. ihi] are used, pairs ilo .. ihi + 1
        const int axc = anchor(x + DX);
        uint32_t P[7];
#pragma unroll
        for (int i = ilo; i <= ihi + 1; i++) P[i] = Q[i] >> axc;
#pragma unroll
        for (int i = ilo; i <= ihi; i++) L[i] = pack_pairs(P[i], P[i + 1]);
    }
    // the candidate's window starts at relative row DY+3, i.e. in pair (DY+3) >> 1
    template <int DY>
    static __device__ __forceinline__ uint32_t gain(const Slab& L, uint2 win) {
        constexpr int i0 = (DY + 3) >> 1;
        return (uint32_t)(__popc(L[i0] & win.x) + __popc(L[i0 + 2] & win.y));
    }
};

// the board representation of sls_p16_kernel for run_chains (sls_thread.cuh)
struct Pairs {
    using Smem = slsp::Smem;
    Smem& sm;
    const int tid;
    uint32_t* const sl;
    const size_t stride;
    uint32_t* const Ub;
    const uint32_t* const cached;

    __device__ __forceinline__ Pairs(Smem& sm, int tid, uint32_t* sl, size_t stride)
        : sm(sm), tid(tid), sl(sl), stride(stride), Ub(&sm.rows[B_U * NP][tid]), cached(&sm.cent[0][tid]) {}

    static __device__ __forceinline__ void load(Smem& sm, int tid, const uint32_t* terrain_rows, const uint2* rtabs, int terrain) {
        for (int i = tid; i < TAB_N; i += NT) {
            const int v = i - TAB_PAD;
            uint2 a = make_uint2(0u, 0u), b = a;
            if (v >= 0 && v < 512) {
                const uint2 s = byte_rows(rtabs[(size_t)terrain * 1024 + v]);   // 7-bit rows, anchored at max(x-3, 0)
                const uint64_t w = (uint64_t)s.x | (uint64_t)s.y << 32;
                // ... placed at row slot s0 = (y-3) & 1 (table 0) and at the other alignment (table 1)
                const int s0 = ((v >> 5) - 3) & 1;
                const uint64_t wa = w << (8 * s0), wb = w << (8 * (s0 ^ 1));
                a = make_uint2((uint32_t)wa, (uint32_t)(wa >> 32));
                b = make_uint2((uint32_t)wb, (uint32_t)(wb >> 32));
            }
            sm.tab[0][i] = a;
            sm.tab[1][i] = b;
        }
        if (tid < 16) {
            const int p = tid - 2;
            sm.C[tid] = (p >= 0 && p < NP) ? (terrain_rows[(size_t)terrain * 32 + 2 * p] & 0xffffu) | (terrain_rows[(size_t)terrain * 32 + 2 * p + 1] << 16) : 0u;
        }
#pragma unroll 8
        for (int r = 0; r < N_BOARDS * NP; r++) sm.rows[r][tid] = 0;
#pragma unroll
        for (int r = 0; r < 32; r++) sm.ring[r][tid] = (uint16_t)NONE;
#pragma unroll
        for (int i = 0; i < CAP; i++) { sm.cent[i][tid] = 0; sm.cwin[i][tid] = make_uint2(0u, 0u); }   // slots past k are loaded (not scored) by the removal scan
    }

    __device__ __forceinline__ int start(const uint32_t* S, uint32_t step, uint32_t& rowmask) {
        for (int p = 0; p < NP; p++) {
            const uint32_t c = sm.C[p + 2];
            Ub[p * NT] = c;
            rowmask |= ((c & 0xffffu) ? 16u << (2 * p) : 0u) | ((c >> 16) ? 32u << (2 * p) : 0u);
        }
        int k = 0;
        const uint32_t reset = stamp_reset(step);
        for (int y = 0; y < MAXH; y++)
            for (uint32_t bits = S[y]; bits; bits &= bits - 1, k++) {
                const int v = y * 32 + __ffs(bits) - 1;
                const uint2 win = ld_tab(sm, &sm.tab[0][v + TAB_PAD]);
                if (k < CAP) { sm.cent[slot(k)][tid] = entry(v, reset); sm.cwin[slot(k)][tid] = win; }
                else sl[(size_t)k * stride] = entry(v, reset);
                flip<true>(sm, tid, v, win, rowmask);
            }
        return k;
    }

    __device__ __forceinline__ void remove(uint32_t hs, uint32_t step, uint32_t stephi, uint32_t young_below, int k, uint32_t& rowmask) {
        uint32_t best_key = 0xffffffffu;
        // cached slots: the warp scans a first group of SCAN slots, then the rest in pairs, up to its largest k (a thread
        // scores only its own k).  No branch inside a group, so the loads of its slots overlap: with 3 warps per scheduler
        // the scan is latency bound when every slot waits for the one before it.  The first group serves grids whose k
        // stays at 8 or below (ex3: 3-5) with one branch; past it, pairs score at most one slot beyond kw (groups of 8 would
        // score 16 slots at the bench's k = 14).
        // kw only has to be >= this thread's own k: threads that arrive here apart from the rest of the warp reduce over a
        // partial mask and scan for their own group, which is still exact
        const int kw = __reduce_max_sync(__activemask(), k);
        constexpr int SCAN = 8;
        uint32_t key[CAP];
#pragma unroll
        for (int i = 0; i < CAP; i++) {
            if ((i < SCAN ? i == 0 : i % 2 == 0) && i >= kw) break;
            const uint32_t e = sm.cent[slot(i)][tid];
            const uint32_t loss = removal_loss(sm, tid, e, sm.cwin[slot(i)][tid]);
            key[i] = i < k ? removal_key(e, i, loss, hs * ((2u * i + 1u) * K3), stephi, young_below) : 0xffffffffu;
            // a group's keys are masked first and then reduced as a tree, not folded into one chain of slot-by-slot mins
            if (i == SCAN - 1) best_key = min(best_key, tree_min<SCAN>(&key[0]));
            else if (i > SCAN && i % 2 == 1) best_key = min(best_key, tree_min<2>(&key[i - 1]));
        }
        if (kw > CAP) {   // the rest of the list (dense warm starts): global entries, windows from the table
            uint32_t mult = (2u * CAP + 1u) * K3;                   // mult = (2i+1) * K3
            for (int i = CAP; i < k; i++, mult += 2u * K3) {
                const uint32_t e = sl[(size_t)i * stride];
                const uint32_t loss = removal_loss(sm, tid, e, ld_tab(sm, &sm.tab[0][(e & 0x1ffu) + TAB_PAD]));
                best_key = min(best_key, removal_key(e, i, loss, hs * mult, stephi, young_below));
            }
        }
        const int best_i = (int)(best_key & 0xffu), last = k - 1;
        int u;
        uint2 win;
        if (best_i < CAP) {
            u = (int)(sm.cent[slot(best_i)][tid] & 0x1ffu);
            win = sm.cwin[slot(best_i)][tid];
        } else {
            u = (int)(sl[(size_t)best_i * stride] & 0x1ffu);
            win = ld_tab(sm, &sm.tab[0][u + TAB_PAD]);
        }
        // swap-remove: entry k-1 (with its window) moves into slot best_i
        if (last < CAP) {
            sm.cent[slot(best_i)][tid] = sm.cent[slot(last)][tid];
            sm.cwin[slot(best_i)][tid] = sm.cwin[slot(last)][tid];
        } else {
            const uint32_t e = sl[(size_t)last * stride];
            if (best_i < CAP) {
                sm.cent[slot(best_i)][tid] = e;
                sm.cwin[slot(best_i)][tid] = ld_tab(sm, &sm.tab[0][(e & 0x1ffu) + TAB_PAD]);
            } else {
                sl[(size_t)best_i * stride] = e;
            }
        }
        sm.ring[step & 31u][tid] = (uint16_t)u;
        flip<false>(sm, tid, u, win, rowmask);
    }

    __device__ __forceinline__ Nbhd fetch(uint32_t rowmask, uint32_t hs) const {
        Nbhd N;
        N.y = pick_rotated(rowmask >> 4, hs & 31u);
        const int odd = N.y & 1;
        // pairs of U from row y-6
        const uint32_t* Up = Ub + ((N.y - 6) >> 1) * NT;
        const uint32_t sel = odd ? 0x5432u : 0x3210u;
        uint32_t A[8];
#pragma unroll
        for (int i = 0; i < 8; i++) A[i] = ld(sm, Up + i * NT);
#pragma unroll
        for (int i = 0; i < 7; i++) N.Q[i] = __byte_perm(A[i], A[i + 1], sel);
        N.x = pick_rotated(N.Q[3] & 0xffffu, (hs >> 5) & 31u);   // Q[3] bits 0-15 = row y
        const int vt = N.y * 32 + N.x + TAB_PAD;
        N.tabt = &sm.tab[odd][vt];
        // t's own window in t16's byte-per-row format around (x-3, y-3): the table whose slot 0 is row y-3, re-anchored
        // from max(x-3, 0) to x-3 (no bit crosses a byte: a window row has no reach bit beyond column x+3)
        const uint2 w0 = ld_tab(sm, &sm.tab[odd ^ 1][vt]);
        const int sh = max(3 - N.x, 0);
        N.wt = make_uint2(w0.x << sh, w0.y << sh);
        return N;
    }

    __device__ __forceinline__ void add(int v, uint32_t step, int k, uint32_t& rowmask) {
        const uint2 win = ld_tab(sm, &sm.tab[0][v + TAB_PAD]);
        flip<true>(sm, tid, v, win, rowmask);
        if (k < CAP) { sm.cent[slot(k)][tid] = entry(v, step); sm.cwin[slot(k)][tid] = win; }
        else sl[(size_t)k * stride] = entry(v, step);
    }

    __device__ __forceinline__ void list_to_rows(int k, uint32_t* out32) const { slsp::list_to_rows(cached, sl, stride, k, out32); }
};

__global__ void __launch_bounds__(NT, 3) sls_p16_kernel(const uint32_t* __restrict__ terrain_rows, const uint2* __restrict__ rtabs,
                                                       ChainState* __restrict__ states, uint32_t* __restrict__ site_lists, size_t stride,
                                                       int n_chains, int chains_per_terrain, uint32_t chain_offset, uint64_t seed,
                                                       long long steps, const int* __restrict__ bounds, int target, int noise_pct,
                                                       const volatile int* interrupt, unsigned long long* __restrict__ totals) {
    run_chains<Pairs>(threadIdx.x, terrain_rows, rtabs, states, site_lists, stride, n_chains, chains_per_terrain, chain_offset, seed, steps,
                      bounds, target, noise_pct, interrupt, totals);
}

}  // namespace slsp

// violations counted by a -DTSS_CHECKED build since the library was loaded (always 0 in the shipped build, which has no checks)
int sls_p16_smem_violations() { return slsp::smem_violations(); }
bool sls_p16_fits(int w, int h) { return h <= slsp::MAXH && w <= slsp::MAXW; }

// site lists: the caller allocates sls_t16_list_words (416 entries per chain >= the 256 sites of a 16x16 grid)
int sls_run_p16(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, uint32_t* site_lists, int n_chains,
                int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
                int noise_pct, unsigned long long* totals_dev) {
    return slsth::launch(slsp::sls_p16_kernel, slsp::SMEM_BYTES, e, rows_dev, tabs_dev, states, site_lists, n_chains, chains_per_terrain,
                         chain_offset, seed, steps, bounds_dev, target, noise_pct, totals_dev);
}

}  // namespace tss
