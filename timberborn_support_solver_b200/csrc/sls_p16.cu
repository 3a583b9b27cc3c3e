// Kernel (b), one chain per THREAD with two grid rows per word, for grids of at most 16x16 (rect 16x16, test/ex1, test/ex3).
//
// sls_t16.cu sits at ~75 % of both the ALU pipe and the shared-memory pipe (65 warp instructions per chain step), so the
// only way to step faster is to issue fewer instructions per step.  On grids of at most 16 columns one 32-bit word holds
// two grid rows: word p of a board is row 2p in bits 0-15 and row 2p+1 in bits 16-31 (no column padding).  A 7-row
// reach window then spans four words instead of seven rows, and every shift, load and carry of the step works on two rows.
//
// The step rule, RNG and tie-breaks are EXACTLY those of sls_spec.hpp and of sls_t16.cu (bit-identical trajectories, the
// parity tests replay both against the same CPU model); the site list, the removal ring and the selection keys are
// t16's.  What differs is the representation:
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
#include "engine.hpp"
#include "sls_spec.hpp"

namespace tss {
namespace slsp {

using namespace tss::sls;

constexpr int NT = 128;          // chains per CTA
constexpr int MAXW = 16;         // columns per pair half
constexpr int MAXH = 16;
constexpr int NP = 8;            // pair words per board
constexpr uint32_t NONE = 0xffffu;
constexpr int TAB_PAD = 128;     // table entries before / after the 512 real ones (candidate sites outside the grid index there)
constexpr int TAB_N = 512 + 2 * TAB_PAD;
// boards of 8 pair words each, back to back: pairs outside [0, 8) of a board alias its neighbours — harmless, because
// out-of-grid rows only ever meet zero window bits (reads) or a zero mask (no write)
enum { B_C0 = 0, B_C1 = 1, B_C2 = 2, B_U = 3, B_O = 4, B_C3 = 5, B_C4 = 6, N_BOARDS = 7 };

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

// ---- bounds-checked build (-DTSS_CHECKED, profiles/checked_build.py), as in sls_t16.cu: every shared-memory access of the
// step loop stays inside the CTA's Smem block, every store lands in a pair of the grid of the board it means.
#ifdef TSS_CHECKED
__device__ unsigned int g_smem_violations = 0;
template <class T>
__device__ __forceinline__ const T* chk_ld(const Smem& sm, const T* p) {
    const size_t off = (size_t)((const char*)p - (const char*)&sm);
    if (off + sizeof(T) > sizeof(Smem) || (off % sizeof(T))) { atomicAdd(&g_smem_violations, 1u); return reinterpret_cast<const T*>(&sm); }
    return p;
}
// a support-cache slot index (the slot's column is always the thread's own)
__device__ __forceinline__ int chk_slot(int i) {
    if ((unsigned)i >= (unsigned)CAP) { atomicAdd(&g_smem_violations, 1u); return 0; }
    return i;
}
__device__ __forceinline__ const uint2* chk_tab(const Smem& sm, const uint2* p) {
    const ptrdiff_t off = p - &sm.tab[0][0];
    if (off < 0 || off >= 2 * TAB_N) { atomicAdd(&g_smem_violations, 1u); return &sm.tab[0][0]; }
    return p;
}
// a store into pair `pair` (0..7) of board `board` for thread tid, and nowhere else
__device__ __forceinline__ uint32_t* chk_st(Smem& sm, uint32_t* p, int board, int tid) {
    const ptrdiff_t off = p - &sm.rows[board * NP][0];
    if (off < 0 || off >= NP * NT || (off % NT) != tid) { atomicAdd(&g_smem_violations, 1u); return &sm.rows[board * NP][tid]; }
    return p;
}
#define LD(p) (*chk_ld(sm, (p)))
#define LDT(p) (*chk_tab(sm, (p)))
#define ST(p, board) (*chk_st(sm, (p), (board), tid))
#define SLOT(arr, i) (sm.arr[chk_slot(i)][tid])
#else
#define LD(p) (*(p))
#define LDT(p) (*(p))
#define ST(p, board) (*(p))
#define SLOT(arr, i) (sm.arr[i][tid])
#endif

__device__ __forceinline__ int pick_rotated(uint32_t bits, uint32_t o) {
    uint32_t rot = __funnelshift_r(bits, bits, o);
    return (int)((__ffs(rot) - 1 + o) & 31u);
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
    const uint32_t lo = pack_pairs(LD(p) >> ax, LD(p + NT) >> ax);
    const uint32_t hi = pack_pairs(LD(p + 2 * NT) >> ax, LD(p + 3 * NT) >> ax);
    return (uint32_t)(__popc(lo & win.x) + __popc(hi & win.y));
}

// adds (ADD) or removes the cover of site v (window win = its tab[0] entry) on the five count planes and refreshes U, O
// and the non-empty-row mask.
// Branch free as in t16: pairs of the window without reach bits (m = 0) recompute what is already there; pairs outside
// the grid read a neighbouring board (never written: the stores are predicated on m != 0) and meet C = 0.
// rowmask is kept in padded coordinates: bit r + 4 = row r has an uncovered tile.
template <bool ADD>
__device__ __forceinline__ void flip(Smem& sm, int tid, int v, uint2 win, uint32_t& rowmask) {
    const int ax = anchor(v & 31), p0 = first_pair(v);
    uint32_t* p = &sm.rows[0][tid] + p0 * NT;  // pair p0 of the first board
    uint32_t nz = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const uint32_t m8 = __byte_perm(j < 2 ? win.x : win.y, 0u, (j & 1) ? 0x4342 : 0x4140);   // slots 2j, 2j+1 at bits 0, 16
        const int off = j * NT;
        uint32_t m = m8 << ax;
        uint32_t a0 = LD(p + B_C0 * BOARD + off), a1 = LD(p + B_C1 * BOARD + off), a2 = LD(p + B_C2 * BOARD + off), t;
        uint32_t a3 = LD(p + B_C3 * BOARD + off), a4 = LD(p + B_C4 * BOARD + off);
        if (ADD) {
            t = a0 & m; a0 ^= m; m = t;
            t = a1 & m; a1 ^= m; m = t;
            t = a2 & m; a2 ^= m; m = t;
        } else {
            t = ~a0 & m; a0 ^= m; m = t;
            t = ~a1 & m; a1 ^= m; m = t;
            t = ~a2 & m; a2 ^= m; m = t;
        }
        if (m) {  // a count crossing 7 <-> 8: rare
            if (ADD) { t = a3 & m; a3 ^= m; a4 ^= t; } else { t = ~a3 & m; a3 ^= m; a4 ^= t; }
            ST(p + B_C3 * BOARD + off, B_C3) = a3; ST(p + B_C4 * BOARD + off, B_C4) = a4;
        }
        const uint32_t hi = a1 | a2 | a3 | a4, C = sm.C[p0 + j + 2];
        const uint32_t Un = C & ~(a0 | hi);
        if (m8) {
            ST(p + B_C0 * BOARD + off, B_C0) = a0; ST(p + B_C1 * BOARD + off, B_C1) = a1; ST(p + B_C2 * BOARD + off, B_C2) = a2;
            ST(p + B_U * BOARD + off, B_U) = Un;
            ST(p + B_O * BOARD + off, B_O) = a0 & ~hi & C;
        }
        nz |= ((Un & 0xffffu) ? 1u << (2 * j) : 0u) | ((Un >> 16) ? 2u << (2 * j) : 0u);
    }
    const int sh = 2 * p0 + 4;
    rowmask = (rowmask & ~(0xffu << sh)) | (nz << sh);
}

__device__ __forceinline__ uint32_t shl_clamped(uint32_t v, int n) {  // PTX shl: shift counts above 31 (incl. "negative" ones) give 0
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
    return r;
}

__device__ __forceinline__ constexpr int cell_start(int r) { return r <= 4 ? r * r : (r == 5 ? 21 : 24); }   // first diamond cell of window row r
__device__ __forceinline__ constexpr int iabs(int a) { return a < 0 ? -a : a; }
__device__ __forceinline__ constexpr int cell_index(int dx, int dy) { return cell_start(dy + 3) + dx + (3 - iabs(dy)); }
__device__ __forceinline__ uint32_t shift_static(uint32_t v, int s) { return s >= 0 ? v << s : v >> (-s); }

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

// One ADD candidate: the site at offset (DX, DY) from the uncovered tile.  L[i] = packed slab of pairs i, i+1 (rows
// y-6+2i .. y-3+2i, columns from max(x+DX-3, 0)); the candidate's window starts at relative row DY+3, i.e. in pair
// (DY+3) >> 1, and tabt is the table whose slot alignment matches that (chosen per step by y & 1).  Keys are t16's.
template <int DX, int DY>
__device__ __forceinline__ uint32_t add_key(const Smem& sm, const uint32_t (&L)[6], const uint2* tabt, uint2 wt, uint32_t fresh_lo, uint32_t fresh_hi,
                                            uint32_t hs, uint32_t gmul) {
    constexpr int cell = cell_index(DX, DY), bit = 8 * (DY + 3) + DX + 3;   // position in t's byte-per-row window (rows 0-3 / 4-6)
    constexpr int i0 = (DY + 3) >> 1;
    const uint2 win = LDT(tabt + DY * 32 + DX);
    const uint32_t g = (uint32_t)(__popc(L[i0] & win.x) + __popc(L[i0 + 2] & win.y));
    const uint32_t tie = ((hs * ((2u * cell + 1u) * K2)) >> 11) & 0x1fffe0u;             // tie_add(hs, cell) << 5
    const uint32_t fresh = shift_static(bit < 32 ? fresh_lo : fresh_hi, 30 - (bit < 32 ? bit : bit - 32)) & TABU_BIT;  // (all zero in a noise step)
    const uint32_t key = (fresh | tie) + g * gmul + ((1u << 21) | (31u - cell));   // gmul = 1 << 21, or 0 in a noise step
    const bool valid = ((bit < 32 ? wt.x >> bit : wt.y >> (bit - 32)) & 1u) != 0;
    return valid ? key : 0u;
}

template <int DX>
__device__ __forceinline__ uint32_t add_column(const Smem& sm, const uint32_t (&Q)[7], int x, const uint2* tabt, uint2 wt, uint32_t fresh_lo,
                                               uint32_t fresh_hi, uint32_t hs, uint32_t gmul) {
    constexpr int M = 3 - iabs(DX);
    constexpr int ilo = (3 - M) >> 1, ihi = ((3 + M) >> 1) + 2;   // packed slabs L[ilo .. ihi] are used, pairs ilo .. ihi + 1
    const int axc = anchor(x + DX);
    uint32_t P[7], L[6];
#pragma unroll
    for (int i = ilo; i <= ihi + 1; i++) P[i] = Q[i] >> axc;
#pragma unroll
    for (int i = ilo; i <= ihi; i++) L[i] = pack_pairs(P[i], P[i + 1]);
    uint32_t mx = add_key<DX, 0>(sm, L, tabt, wt, fresh_lo, fresh_hi, hs, gmul);
    if (M >= 1) {
        mx = max(mx, add_key<DX, (M >= 1 ? -1 : 0)>(sm, L, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
        mx = max(mx, add_key<DX, (M >= 1 ? 1 : 0)>(sm, L, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
    }
    if (M >= 2) {
        mx = max(mx, add_key<DX, (M >= 2 ? -2 : 0)>(sm, L, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
        mx = max(mx, add_key<DX, (M >= 2 ? 2 : 0)>(sm, L, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
    }
    if (M >= 3) {
        mx = max(mx, add_key<DX, (M >= 3 ? -3 : 0)>(sm, L, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
        mx = max(mx, add_key<DX, (M >= 3 ? 3 : 0)>(sm, L, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
    }
    return mx;
}

__global__ void __launch_bounds__(NT, 3) sls_p16_kernel(const uint32_t* __restrict__ terrain_rows, const uint2* __restrict__ rtabs,
                                                       ChainState* __restrict__ states, uint32_t* __restrict__ site_lists, size_t stride,
                                                       int n_chains, int chains_per_terrain, uint32_t chain_offset, uint64_t seed,
                                                       long long steps, const int* __restrict__ bounds, int target, int noise_pct,
                                                       const volatile int* interrupt, unsigned long long* __restrict__ totals) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const int tid = threadIdx.x;
    const int chain = blockIdx.x * NT + tid;
    const int terrain = chains_per_terrain > 0 ? (blockIdx.x * NT) / chains_per_terrain : 0;
    // a layout within the target is already known for this terrain: nothing to do (as t16)
    if (target >= 0 && bounds[chains_per_terrain > 0 ? terrain : 0] <= target) return;
    for (int i = tid; i < TAB_N; i += NT) {
        const int v = i - TAB_PAD;
        uint2 a = make_uint2(0u, 0u), b = a;
        if (v >= 0 && v < 512) {
            const uint2 s = rtabs[(size_t)terrain * 1024 + v];   // 7-bit rows, anchored at max(x-3, 0)
            // one BYTE per window row (rows 0-3 in .x, rows 4-6 in .y) ...
            const uint64_t w = (uint64_t)((s.x & 0x7fu) | ((s.x & 0x3f80u) << 1) | ((s.x & 0x1fc000u) << 2) | ((s.x & 0xfe00000u) << 3)) |
                               (uint64_t)((s.y & 0x7fu) | ((s.y & 0x3f80u) << 1) | ((s.y & 0x1fc000u) << 2)) << 32;
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
    __syncthreads();

    const bool exists = chain < n_chains;
    ChainState& st = states[exists ? chain : 0];
    int done = exists ? st.done : 1;
    const bool run = !done;
    unsigned long long scored = 0;
    long long my_steps = 0;
    uint32_t flips = 0;   // supports added + removed

    if (run) {
        const int epoch_bound = bounds[chains_per_terrain > 0 ? terrain : 0];
        const uint32_t base = chain_base(seed, chain_offset + (uint32_t)chain);
        const uint32_t nq7 = noise_q7(noise_pct);
        const int tenure = tenure_of(chain_offset + (uint32_t)chain);
        uint32_t* sl = site_lists + chain;
        uint32_t* const Ub = &sm.rows[B_U * NP][tid];
        const uint32_t* const cached = &sm.cent[0][tid];
        int best = st.best, k = 0;
        uint32_t step = st.step, rowmask = 0;

        {   // site list in row-major order (spec), stamps "half a period ago"; cover planes from the list
            for (int p = 0; p < NP; p++) {
                const uint32_t c = sm.C[p + 2];
                Ub[p * NT] = c;
                rowmask |= ((c & 0xffffu) ? 16u << (2 * p) : 0u) | ((c >> 16) ? 32u << (2 * p) : 0u);
            }
            const uint32_t reset = stamp_reset(step);
            for (int y = 0; y < MAXH; y++)
                for (uint32_t bits = st.S[y]; bits; bits &= bits - 1, k++) {
                    const int v = y * 32 + __ffs(bits) - 1;
                    const uint2 win = LDT(&sm.tab[0][v + TAB_PAD]);
                    if (k < CAP) { SLOT(cent, k) = entry(v, reset); SLOT(cwin, k) = win; }
                    else sl[(size_t)k * stride] = entry(v, reset);
                    flip<true>(sm, tid, v, win, rowmask);
                }
        }

        for (long long it = 0; it < steps; it++) {
            if ((it & 1023) == 1023 && *interrupt) break;
            const int limit = min(epoch_bound, best);
            const uint32_t hs = step_hash(base, step);
            const int ten = effective_tenure(tenure, k);
            const bool drop = k >= limit;
            if (drop && k == 0) { done = 1; break; }
            sm.ring[step & 31u][tid] = (uint16_t)NONE;  // every consumed step owns its slot (stale entries are 32 steps old)
            if (!drop && rowmask == 0) {  // complete layout with k < limit supports
                best = k;
                list_to_rows(cached, sl, stride, k, st.bestS);
                step++; my_steps++;
                if (k <= target || k == 0) { done = 1; break; }
                continue;
            }
            if (drop || (k == limit - 1 && k > 0)) {
                // ---- removal: min-loss support, random ties; supports younger than the tenure only as a last resort (not when
                // dropping).  key = young | loss | tie | list index: unique, so the minimum is the spec's (lowest index wins ties)
                const uint32_t stephi = (step << 16) | 0xffffu;             // stephi - entry = (age << 16) + (0xffff - site): no borrow
                const uint32_t young_below = drop ? 0u : (uint32_t)ten << 16;
                uint32_t best_key = 0xffffffffu;
                // cached slots: the warp scans them in groups of SCAN up to its largest k (a thread scores only its own k).  No
                // branch inside a group, so the loads of its slots overlap: with 3 warps per scheduler the scan is latency bound
                // when every slot waits for the one before it.
                // kw only has to be >= this thread's own k: threads that arrive here apart from the rest of the warp reduce over a
                // partial mask and scan for their own group, which is still exact
                const int kw = __reduce_max_sync(__activemask(), k);
                constexpr int SCAN = 8;
#pragma unroll
                for (int i = 0; i < CAP; i++) {
                    if (i % SCAN == 0 && i >= kw) break;
                    const uint32_t e = SLOT(cent, i);
                    const uint32_t loss = removal_loss(sm, tid, e, SLOT(cwin, i));
                    const uint32_t tie = ((hs * ((2u * i + 1u) * K3)) >> 7) & 0x1fffe00u;  // tie_remove(hs, i) << 9
                    const uint32_t young = (stephi - e) < young_below ? TABU_BIT : 0u;
                    const uint32_t key = (young | tie | (uint32_t)i) + loss * (1u << 25);
                    best_key = i < k ? min(best_key, key) : best_key;   // compiles to a select: no branch inside a group
                }
                if (kw > CAP) {   // the rest of the list (dense warm starts): global entries, windows from the table
                    uint32_t mult = (2u * CAP + 1u) * K3;                   // mult = (2i+1) * K3
                    for (int i = CAP; i < k; i++, mult += 2u * K3) {
                        const uint32_t e = sl[(size_t)i * stride];
                        const uint32_t loss = removal_loss(sm, tid, e, LDT(&sm.tab[0][(e & 0x1ffu) + TAB_PAD]));
                        const uint32_t tie = ((hs * mult) >> 7) & 0x1fffe00u;
                        const uint32_t young = (stephi - e) < young_below ? TABU_BIT : 0u;
                        best_key = min(best_key, (young | tie | (uint32_t)i) + loss * (1u << 25));
                    }
                }
                const int best_i = (int)(best_key & 0x1ffu), last = k - 1;
                int u;
                uint2 win;
                if (best_i < CAP) {
                    u = (int)(SLOT(cent, best_i) & 0x1ffu);
                    win = SLOT(cwin, best_i);
                } else {
                    u = (int)(sl[(size_t)best_i * stride] & 0x1ffu);
                    win = LDT(&sm.tab[0][u + TAB_PAD]);
                }
                // swap-remove: entry k-1 (with its window) moves into slot best_i
                if (last < CAP) {
                    SLOT(cent, best_i) = SLOT(cent, last);
                    SLOT(cwin, best_i) = SLOT(cwin, last);
                } else {
                    const uint32_t e = sl[(size_t)last * stride];
                    if (best_i < CAP) {
                        SLOT(cent, best_i) = e;
                        SLOT(cwin, best_i) = LDT(&sm.tab[0][(e & 0x1ffu) + TAB_PAD]);
                    } else {
                        sl[(size_t)best_i * stride] = e;
                    }
                }
                sm.ring[step & 31u][tid] = (uint16_t)u;
                flip<false>(sm, tid, u, win, rowmask);
                scored += (unsigned)k;
                k--;
                flips++;
            }
            if (!drop) {
                // ---- addition at a random uncovered tile t: best-gain site of R(t)
                const int y = pick_rotated(rowmask >> 4, hs & 31u);
                const int odd = y & 1;
                // pairs of U from row y-6: Q[i] = rows y-6+2i (bits 0-15) and y-5+2i (bits 16-31)
                const uint32_t* Up = Ub + ((y - 6) >> 1) * NT;
                const uint32_t sel = odd ? 0x5432u : 0x3210u;
                uint32_t A[8], Q[7];
#pragma unroll
                for (int i = 0; i < 8; i++) A[i] = LD(Up + i * NT);
#pragma unroll
                for (int i = 0; i < 7; i++) Q[i] = __byte_perm(A[i], A[i + 1], sel);
                const int x = pick_rotated(Q[3] & 0xffffu, (hs >> 5) & 31u);   // Q[3] bits 0-15 = row y
                const int vt = y * 32 + x + TAB_PAD;
                const uint2* tabt = &sm.tab[odd][vt];                // candidates' windows in the slot alignment of pairs from y-6
                // t's own window in t16's byte-per-row format around (x-3, y-3): the table whose slot 0 is row y-3, re-anchored
                // from max(x-3, 0) to x-3 (no bit crosses a byte: a window row has no reach bit beyond column x+3)
                const uint2 w0 = LDT(&sm.tab[odd ^ 1][vt]);
                const int sh = max(3 - x, 0);
                const uint2 wt = make_uint2(w0.x << sh, w0.y << sh);
                const bool noise = ((hs >> 10) & 127u) < nq7;
                uint32_t tw_lo = 0, tw_hi = 0;  // sites removed fewer than `ten` steps ago, as a byte-per-row window around t (rows 0-3 / 4-6)
                for (int j = 0; j < ten; j++) {
                    const uint32_t e = sm.ring[(step - (uint32_t)j) & 31u][tid];
                    const int dx3 = (int)(e & 31u) - x + 3, dy3 = (int)(e >> 5) - y + 3;
                    if ((unsigned)dx3 < 7u && (unsigned)dy3 < 7u) {
                        const int bit = 8 * dy3 + dx3;       // byte-per-row window, like wt
                        tw_lo |= shl_clamped(1u, bit);
                        tw_hi |= shl_clamped(1u, bit - 32);
                    }
                }
                const uint32_t fresh_lo = noise ? 0u : ~tw_lo, fresh_hi = noise ? 0u : ~tw_hi;
                const uint32_t gmul = noise ? 0u : 1u << 21;
                uint32_t mx = add_column<0>(sm, Q, x, tabt, wt, fresh_lo, fresh_hi, hs, gmul);
                mx = max(mx, add_column<-1>(sm, Q, x, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
                mx = max(mx, add_column<1>(sm, Q, x, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
                mx = max(mx, add_column<-2>(sm, Q, x, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
                mx = max(mx, add_column<2>(sm, Q, x, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
                mx = max(mx, add_column<-3>(sm, Q, x, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
                mx = max(mx, add_column<3>(sm, Q, x, tabt, wt, fresh_lo, fresh_hi, hs, gmul));
                // the winning cell from the key's low bits
                const int cell = 31 - (int)(mx & 31u);
                const int r = (cell >= 1) + (cell >= 4) + (cell >= 9) + (cell >= 16) + (cell >= 21) + (cell >= 24);
                const int dy = r - 3, dx = cell - cell_start(r) - (3 - abs(dy));
                const int v = (y + dy) * 32 + x + dx;
                const uint2 win = LDT(&sm.tab[0][v + TAB_PAD]);
                flip<true>(sm, tid, v, win, rowmask);
                if (k < CAP) { SLOT(cent, k) = entry(v, step); SLOT(cwin, k) = win; }
                else sl[(size_t)k * stride] = entry(v, step);
                if (!noise) scored += (unsigned)(__popc(wt.x) + __popc(wt.y));
                k++;
                flips++;
            }
            step++; my_steps++;
        }

        list_to_rows(cached, sl, stride, k, st.S);
        st.k = k; st.best = best; st.step = step; st.done = done;
        const unsigned long long tot = ((unsigned long long)st.scored_hi << 32 | st.scored_lo) + scored;
        st.scored_lo = (uint32_t)tot; st.scored_hi = (uint32_t)(tot >> 32);
        st.steps_done += (uint32_t)my_steps;
    }
    // one pair of atomics per warp
    unsigned long long a = scored, b = (unsigned long long)my_steps, c = (unsigned long long)flips;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); c += __shfl_xor_sync(0xffffffffu, c, o); }
    if ((tid & 31) == 0 && (a | b)) { atomicAdd(&totals[0], a); atomicAdd(&totals[1], b); atomicAdd(&totals[2], c); }
}

}  // namespace slsp

// violations counted by a -DTSS_CHECKED build since the library was loaded (always 0 in the shipped build, which has no checks)
int sls_p16_smem_violations() {
#ifdef TSS_CHECKED
    unsigned int v = 0;
    if (cudaMemcpyFromSymbol(&v, slsp::g_smem_violations, sizeof v) != cudaSuccess) return -1;
    return (int)v;
#else
    return 0;
#endif
}
bool sls_p16_fits(int w, int h) { return h <= slsp::MAXH && w <= slsp::MAXW; }
int sls_p16_cta_chains() { return slsp::NT; }

// site lists: the caller allocates sls_t16_list_words (416 entries per chain >= the 256 sites of a 16x16 grid)
int sls_run_p16(tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, sls::ChainState* states, uint32_t* site_lists, int n_chains,
                int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
                int noise_pct, unsigned long long* totals_dev) {
    TSS_CUDA(e, cudaFuncSetAttribute(slsp::sls_p16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)slsp::SMEM_BYTES));
    const size_t stride = ((size_t)n_chains + 31) & ~(size_t)31;
    const int blocks = (n_chains + slsp::NT - 1) / slsp::NT;
    slsp::sls_p16_kernel<<<blocks, slsp::NT, slsp::SMEM_BYTES, e->stream>>>(rows_dev, tabs_dev, states, site_lists, stride, n_chains,
                                                                           chains_per_terrain, chain_offset, seed, steps, bounds_dev, target,
                                                                           noise_pct, e->interrupt_dev, totals_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}

}  // namespace tss
