// The thread-per-chain SLS kernels (sls_t16.cu: one grid row per word, sls_p16.cu: two grid rows per word) share
// everything but their board representation: the step rule, RNG and tie-breaks of sls_spec.hpp, the selection keys, the
// site-list format, the removal ring, the kernel frame and the launch.  That part lives here, once; a kernel supplies a
// representation struct K (its Smem layout, table load, list start-up, removal scan, addition fetch and flips) and a
// __global__ entry point that calls run_chains<K>.
//
// A chain is one thread: its boards live in shared memory as [row][thread] words (bank = thread, conflict free for any row
// index), every candidate layout is scored by that thread alone, and a warp instruction advances 32 layouts.
//   * the site list lives in global memory as [index][chain] words (coalesced across the warp, L1 resident): site v in bits
//     0-8 (sls_p16.cu packs the site into the low half its own way, see its entry()), the step at which the support was
//     added in bits 16-31 — for a current support that IS its last flip, so the "young support" test of the spec needs no
//     per-site stamp array;
//   * "recently removed" (the tabu test of add candidates, which are never current supports) is answered from a ring of
//     the sites removed in the last 32 steps (one slot per step), folded once per step into a 7x7 window mask around the
//     chosen uncovered tile.  Equivalent to the spec's 16-bit stamps for epochs of at most 32768 steps — the engine never
//     launches longer ones (tss_search_run splits them);
//   * selection keys carry the candidate's index in their low bits, so min / max are single instructions, independent of
//     the evaluation order, and ties go to the lowest index as the spec demands.
#pragma once
#include "engine.hpp"
#include "sls_spec.hpp"

namespace tss {
namespace slsth {

using namespace tss::sls;

constexpr int NT = 128;          // chains per CTA
constexpr uint32_t NONE = 0xffffu;
constexpr int TAB_PAD = 128;     // table entries before / after the 512 real ones (candidate sites outside the grid index there)
// boards back to back: rows outside the grid of a board alias its neighbours — harmless, because out-of-grid rows only ever
// meet zero window bits (reads) or a zero mask (no write)
enum { B_C0 = 0, B_C1 = 1, B_C2 = 2, B_U = 3, B_O = 4, B_C3 = 5, B_C4 = 6, N_BOARDS = 7 };

// ---- bounds-checked build (-DTSS_CHECKED, profiles/checked_build.py): compute-sanitizer is closed on the B200 pool, and these
// kernels alias neighbouring boards on purpose, so the claim "every access stays inside the CTA's Smem block, every STORE
// lands in a row of the grid of the board it means" is checked by the kernel itself: each shared-memory access of the step
// loop goes through ld / ld_tab / st, violations are counted in a device global (tss_debug_smem_violations()).  The counter
// is static: the library is compiled without -rdc, so each kernel's .cu has its own, read by its sls_*_smem_violations().
#ifdef TSS_CHECKED
static __device__ unsigned int g_smem_violations = 0;
static __device__ __forceinline__ void violation() { atomicAdd(&g_smem_violations, 1u); }
#endif

template <class Smem, class T>
__device__ __forceinline__ T ld(const Smem& sm, const T* p) {
#ifdef TSS_CHECKED
    const size_t off = (size_t)((const char*)p - (const char*)&sm);
    if (off + sizeof(T) > sizeof(Smem) || (off % sizeof(T))) { violation(); return *reinterpret_cast<const T*>(&sm); }
#endif
    return *p;
}
// a reach-table entry
template <class Smem>
__device__ __forceinline__ uint2 ld_tab(const Smem& sm, const uint2* p) {
#ifdef TSS_CHECKED
    const ptrdiff_t off = p - reinterpret_cast<const uint2*>(&sm.tab);
    if (off < 0 || off >= (ptrdiff_t)(sizeof(sm.tab) / sizeof(uint2))) { violation(); return *reinterpret_cast<const uint2*>(&sm.tab); }
#endif
    return *p;
}
// a store into a row of the grid of board `board` for thread tid, and nowhere else
template <class Smem>
__device__ __forceinline__ uint32_t& st(Smem& sm, uint32_t* p, int board, int tid) {
#ifdef TSS_CHECKED
    constexpr int ROWS = sizeof(sm.rows) / sizeof(sm.rows[0]) / N_BOARDS;   // words of one thread per board
    const ptrdiff_t off = p - &sm.rows[board * ROWS][0];
    if (off < 0 || off >= ROWS * NT || (off % NT) != tid) { violation(); return sm.rows[board * ROWS][tid]; }
#endif
    return *p;
}
#ifdef TSS_CHECKED
static inline int smem_violations() {
    unsigned int v = 0;
    if (cudaMemcpyFromSymbol(&v, g_smem_violations, sizeof v) != cudaSuccess) return -1;
    return (int)v;
}
#else
static inline int smem_violations() { return 0; }   // the shipped build has no checks
#endif

// ---- phase-profiling build (-DTSS_SLS_PROF, profiles/sls_phases.py): clock64() between the parts of a step, summed per
// thread and added into a device global once per warp at the end of the launch (read by the kernel file's
// sls_*_phases()).  A load is charged to the phase that first waits for it, so the figures say where a warp waits, not
// where an instruction was issued.  In the shipped build Prof is empty and every mark compiles to nothing.
enum { PH_SCAN, PH_RFLIP, PH_FETCH, PH_CAND, PH_AFLIP, PH_FRAME, N_PHASES };
#ifdef TSS_SLS_PROF
static __device__ unsigned long long g_phases[N_PHASES + 1];   // cycles per phase summed over threads, then thread steps
struct Prof {
    unsigned long long c[N_PHASES] = {};
    long long t = 0;
    __device__ __forceinline__ void start() { t = clock64(); }
    __device__ __forceinline__ void mark(int ph) { const long long n = clock64(); c[ph] += (unsigned long long)(n - t); t = n; }
    __device__ __forceinline__ void flush(unsigned long long steps) {
#pragma unroll
        for (int i = 0; i <= N_PHASES; i++) {
            unsigned long long a = i < N_PHASES ? c[i] : steps;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
            if ((threadIdx.x & 31) == 0) atomicAdd(&g_phases[i], a);
        }
    }
};
// copies the totals to out[0 .. N_PHASES] and clears them
static inline int read_phases(unsigned long long* out) {
    static const unsigned long long zero[N_PHASES + 1] = {};
    if (cudaMemcpyFromSymbol(out, g_phases, sizeof zero) != cudaSuccess) return -1;
    return cudaMemcpyToSymbol(g_phases, zero, sizeof zero) == cudaSuccess ? N_PHASES : -1;
}
#else
struct Prof {
    __device__ __forceinline__ void start() {}
    __device__ __forceinline__ void mark(int) {}
    __device__ __forceinline__ void flush(unsigned long long) {}
};
#endif

__device__ __forceinline__ uint32_t shl_clamped(uint32_t v, int n) {  // PTX shl: shift counts above 31 (incl. "negative" ones) give 0
    uint32_t r;
    asm("shl.b32 %0, %1, %2;" : "=r"(r) : "r"(v), "r"(n));
    return r;
}
// a & b as one AND that the compiler keeps: a product or a test of the result does not get the AND folded into it
__device__ __forceinline__ uint32_t and_b32(uint32_t a, uint32_t b) {
    uint32_t r;
    asm("and.b32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b));
    return r;
}
__device__ __forceinline__ constexpr int iabs(int a) { return a < 0 ? -a : a; }
__device__ __forceinline__ constexpr int cell_index(int dx, int dy) { return cell_start(dy + 3) + dx + (3 - iabs(dy)); }

// a reach-table window (7-bit rows, sls_spec.hpp) spread to one BYTE per row: rows 0-3 in .x, rows 4-6 in .y.  Windows cut
// out of the boards are then assembled with byte permutes, and bit 7 of every byte (zero here) masks whatever the cut left there.
__device__ __forceinline__ uint2 byte_rows(uint2 s) {
    return make_uint2((s.x & 0x7fu) | ((s.x & 0x3f80u) << 1) | ((s.x & 0x1fc000u) << 2) | ((s.x & 0xfe00000u) << 3),
                      (s.y & 0x7fu) | ((s.y & 0x3f80u) << 1) | ((s.y & 0x1fc000u) << 2));
}

// The five count planes of one board word at p + off (a row or a pair of rows of the first board): adds (ADD) or removes the
// cover mask m and refreshes U and O there; returns the new U word.  Branch free: words of the window without reach bits
// (cover = 0) recompute what is already there; words outside the grid read a neighbouring board (never written: the stores
// are predicated on cover != 0) and meet C = 0 (terrain word sm.C[c]).
template <bool ADD, int BOARD, class Smem>
__device__ __forceinline__ uint32_t flip_word(Smem& sm, int tid, uint32_t* p, int off, uint32_t m, uint32_t cover, int c) {
    uint32_t a0 = ld(sm, p + B_C0 * BOARD + off), a1 = ld(sm, p + B_C1 * BOARD + off), a2 = ld(sm, p + B_C2 * BOARD + off), t;
    uint32_t a3 = ld(sm, p + B_C3 * BOARD + off), a4 = ld(sm, p + B_C4 * BOARD + off);
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
        st(sm, p + B_C3 * BOARD + off, B_C3, tid) = a3; st(sm, p + B_C4 * BOARD + off, B_C4, tid) = a4;
    }
    const uint32_t hi = a1 | a2 | a3 | a4, C = sm.C[c];
    const uint32_t Un = C & ~(a0 | hi);
    if (cover) {
        st(sm, p + B_C0 * BOARD + off, B_C0, tid) = a0; st(sm, p + B_C1 * BOARD + off, B_C1, tid) = a1; st(sm, p + B_C2 * BOARD + off, B_C2, tid) = a2;
        st(sm, p + B_U * BOARD + off, B_U, tid) = Un;
        st(sm, p + B_O * BOARD + off, B_O, tid) = a0 & ~hi & C;
    }
    return Un;
}

// Removal key of list entry e (index i, loss `loss`): young | loss | tie | index, unique, so the minimum is the spec's
// (lowest index wins ties).  hsm = hs * (2i+1) * K3; stephi - e = (age << 16) + (0xffff - low half): no borrow.
// sls_p16.cu encodes the same order with one byte per field (its removal_key): its lists have at most 256 entries.
__device__ __forceinline__ uint32_t remove_key(uint32_t e, int i, uint32_t loss, uint32_t hsm, uint32_t stephi, uint32_t young_below) {
    const uint32_t tie = (hsm >> 7) & 0x1fffe00u;  // tie_remove(hs, i) << 9
    const uint32_t young = (stephi - e) < young_below ? TABU_BIT : 0u;
    return (young | tie | (uint32_t)i) + loss * (1u << 25);
}

// One ADD candidate: the site at offset (DX, DY) from the uncovered tile.  S = the kernel's slab of U for this DX, from
// which Nbhd::gain takes the candidate's gain with its reach window; tabt = the table entry of the tile; vf = validity and
// freshness of the 25 candidates (add_site).  Keys are unique per cell (the cell index sits in the low bits), so the
// maximum is independent of the evaluation order and ties go to the lowest cell as the spec demands.
// One byte per field, most significant first: fresh * 64 + gain + 1 (a gain is at most 25 tiles; 1 in a noise step),
// tie_add(hs, cell) in bytes 1-2, which are bytes 2-3 of the tie product, and (3 - DY) * 32 + (3 - DX) in byte 0: it falls
// as the cell index grows (cells are numbered by DY, then DX), and the site is (y + 3) * 32 + x + 3 minus it, with no
// decode of the cell.  The fields are built on the FMA pipe (IMADs) and merged with one PRMT, off the integer-ALU pipe
// that bounds both kernels: one AND picks the candidate's two bits of vf, valid at bit a (lands in byte 1, which the PRMT
// drops) and fresh at bit a + 16 (lands at bit 30, the 64 of byte 3), and the same AND decides validity.
template <int DX, int DY, class Nbhd, class Smem>
__device__ __forceinline__ uint32_t add_key(const Smem& sm, const typename Nbhd::Slab& S, const uint2* tabt, const uint32_t (&vf)[4],
                                            uint32_t hs, uint32_t gmul) {
    constexpr int cell = cell_index(DX, DY), a = 8 * ((DY + 3) & 1) + DX + 3;   // a: the candidate's validity bit in vf[(DY + 3) >> 1]
    const uint2 win = ld_tab(sm, tabt + DY * 32 + DX);
    const uint32_t g = Nbhd::template gain<DY>(S, win);
    const uint32_t q = and_b32(vf[(DY + 3) >> 1], 1u << a | 1u << (a + 16));
    const uint32_t lo = 0x01000000u | (uint32_t)((3 - DY) * 32 + 3 - DX);
    const uint32_t key = __byte_perm(hs * ((2u * cell + 1u) * K2), g * gmul + lo + q * (1u << (14 - a)), 0x7324);   // gmul = 1 << 24, or 0 in a noise step
    return q ? key : 0u;
}

// the best key of the candidates in column DX of the diamond: one slab of U serves all of them
template <int DX, class Smem, class Nbhd>
__device__ __forceinline__ uint32_t add_column(const Smem& sm, const Nbhd& N, const uint32_t (&vf)[4], uint32_t hs, uint32_t gmul) {
    constexpr int M = 3 - iabs(DX);
    typename Nbhd::Slab S;
    N.template slab<DX, M>(S);
    uint32_t mx = add_key<DX, 0, Nbhd>(sm, S, N.tabt, vf, hs, gmul);
    if (M >= 1) {
        mx = max(mx, add_key<DX, (M >= 1 ? -1 : 0), Nbhd>(sm, S, N.tabt, vf, hs, gmul));
        mx = max(mx, add_key<DX, (M >= 1 ? 1 : 0), Nbhd>(sm, S, N.tabt, vf, hs, gmul));
    }
    if (M >= 2) {
        mx = max(mx, add_key<DX, (M >= 2 ? -2 : 0), Nbhd>(sm, S, N.tabt, vf, hs, gmul));
        mx = max(mx, add_key<DX, (M >= 2 ? 2 : 0), Nbhd>(sm, S, N.tabt, vf, hs, gmul));
    }
    if (M >= 3) {
        mx = max(mx, add_key<DX, (M >= 3 ? -3 : 0), Nbhd>(sm, S, N.tabt, vf, hs, gmul));
        mx = max(mx, add_key<DX, (M >= 3 ? 3 : 0), Nbhd>(sm, S, N.tabt, vf, hs, gmul));
    }
    return mx;
}

// Removal-ring slots of the steps before this one that every step reads: a tenure is at least 2, and at most 4 at k <= 14
// (effective_tenure), the 16x16 optimum plateau.  They do not depend on the step's own results, so the step loads them first.
constexpr int RECENT = 3;

// site e (NONE: none) into the tabu window around t = (x, y): a byte-per-row window like wt (rows 0-3 in lo, 4-6 in hi)
__device__ __forceinline__ void tabu_bit(uint32_t e, int x, int y, uint32_t& lo, uint32_t& hi) {
    const int dx3 = (int)(e & 31u) - x + 3, dy3 = (int)(e >> 5) - y + 3;
    if ((unsigned)dx3 < 7u && (unsigned)dy3 < 7u) {
        const int bit = 8 * dy3 + dx3;
        lo |= shl_clamped(1u, bit);
        hi |= shl_clamped(1u, bit - 32);
    }
}

// The addition at the uncovered tile (N.x, N.y) that the kernel's fetch picked: the site of the best of the 25 candidates.
// Sites removed fewer than `ten` steps ago are tabu: `removed` in this step, recent[j] j + 1 steps ago, older ones in the
// ring.  In a noise step every valid candidate ties on gain and freshness.
template <class Smem, class Nbhd>
__device__ __forceinline__ int add_site(const Smem& sm, int tid, const Nbhd& N, uint32_t hs, uint32_t step, int ten, bool noise, uint32_t removed,
                                        const uint32_t (&recent)[RECENT], Prof& pf) {
    const int x = N.x, y = N.y;
    uint32_t tw_lo = 0, tw_hi = 0;
    tabu_bit(removed, x, y, tw_lo, tw_hi);
#pragma unroll
    for (int j = 0; j < RECENT; j++)
        if (j + 1 < ten) tabu_bit(recent[j], x, y, tw_lo, tw_hi);
#pragma unroll 1
    for (int j = RECENT + 1; j < ten; j++) tabu_bit(sm.ring[(step - (uint32_t)j) & 31u][tid], x, y, tw_lo, tw_hi);
    pf.mark(PH_FETCH);
    // vf[i]: rows 2i, 2i+1 of t's window N.wt (byte-per-row, validity) in bytes 0-1, the same rows of its valid and fresh
    // candidates (not tabu; none in a noise step) in bytes 2-3
    const uint32_t fv_lo = noise ? 0u : N.wt.x & ~tw_lo, fv_hi = noise ? 0u : N.wt.y & ~tw_hi;
    const uint32_t vf[4] = {__byte_perm(N.wt.x, fv_lo, 0x5410), __byte_perm(N.wt.x, fv_lo, 0x7632), __byte_perm(N.wt.y, fv_hi, 0x5410),
                            __byte_perm(N.wt.y, fv_hi, 0x7632)};
    const uint32_t gmul = noise ? 0u : 1u << 24;
    uint32_t mx = add_column<0>(sm, N, vf, hs, gmul);
    mx = max(mx, add_column<-1>(sm, N, vf, hs, gmul));
    mx = max(mx, add_column<1>(sm, N, vf, hs, gmul));
    mx = max(mx, add_column<-2>(sm, N, vf, hs, gmul));
    mx = max(mx, add_column<2>(sm, N, vf, hs, gmul));
    mx = max(mx, add_column<-3>(sm, N, vf, hs, gmul));
    mx = max(mx, add_column<3>(sm, N, vf, hs, gmul));
    return (y + 3) * 32 + x + 3 - (int)(mx & 0xffu);   // the winning site from the key's low byte
}

// The kernel body.  K is the board representation:
//   K::Smem, K::load(sm, tid, terrain_rows, rtabs, terrain)  shared memory and its set-up (table, terrain, boards, ring)
//   K(sm, tid, sl, stride)                                    the chain's view of it and of its global site list `sl`
//   start(S, step, rowmask) -> k                              site list and cover planes of the layout S
//   remove(hs, stephi, young_below, k, rowmask, pf)           the removal: scan, swap-remove, flip; returns the removed site
//   fetch(rowmask, hs) -> Nbhd                                the uncovered tile of an addition and U around it
//   add(v, step, k, rowmask)                                  the addition of site v as list entry k
//   list_to_rows(k, out)                                      the support rows of the list (rare path)
// K::Smem has the members tab, C, rows and ring.  tid = threadIdx.x, read by the __global__ entry point: there
// __launch_bounds__ tells the compiler that it is below NT.
template <class K>
__device__ __forceinline__ void run_chains(const int tid, const uint32_t* __restrict__ terrain_rows, const uint2* __restrict__ rtabs,
                                           ChainState* __restrict__ states, uint32_t* __restrict__ site_lists, size_t stride,
                                           int n_chains, int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps,
                                           const int* __restrict__ bounds, int target, int noise_pct, const volatile int* interrupt,
                                           unsigned long long* __restrict__ totals) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typename K::Smem& sm = *reinterpret_cast<typename K::Smem*>(smem_raw);
    const int chain = blockIdx.x * NT + tid;
    const int terrain = chains_per_terrain > 0 ? (blockIdx.x * NT) / chains_per_terrain : 0;
    // a layout within the target is already known for this terrain (found in an earlier epoch): nothing to do.  Lets a host
    // queue several epochs back to back without a round trip in between (one-shot solves, sls_spec.hpp).
    if (target >= 0 && bounds[chains_per_terrain > 0 ? terrain : 0] <= target) return;
    K::load(sm, tid, terrain_rows, rtabs, terrain);
    __syncthreads();

    const bool exists = chain < n_chains;
    ChainState& st = states[exists ? chain : 0];
    int done = exists ? st.done : 1;
    const bool run = !done;
    unsigned long long scored = 0;
    long long my_steps = 0;
    uint32_t flips = 0;   // supports added + removed
    Prof pf;
    pf.start();

    if (run) {
        const int epoch_bound = bounds[chains_per_terrain > 0 ? terrain : 0];
        const uint32_t base = chain_base(seed, chain_offset + (uint32_t)chain);
        const uint32_t nq7 = noise_q7(noise_pct);
        const int tenure = tenure_of(chain_offset + (uint32_t)chain);
        K R(sm, tid, site_lists + chain, stride);
        int best = st.best;
        uint32_t step = st.step, rowmask = 0;
        int k = R.start(st.S, step, rowmask);   // site list in row-major order (spec), stamps "half a period ago"
        int limit = min(epoch_bound, best);
        uint32_t hs = step_hash(base, step);

        for (long long it = 0; it < steps; it++) {
            if ((it & 1023) == 1023 && *interrupt) break;
            const int ten = effective_tenure(tenure, k);
            const bool drop = k >= limit;
            if (drop && k == 0) { done = 1; break; }
            // the ring slots of earlier steps and the next step's hash depend on nothing this step computes: issued first, their
            // latency overlaps the removal scan instead of waiting in the addition's (and the next step's) dependent chain
            uint32_t recent[RECENT];
#pragma unroll
            for (int j = 0; j < RECENT; j++) recent[j] = sm.ring[(step - 1u - (uint32_t)j) & 31u][tid];
            const uint32_t hs_next = step_hash(base, step + 1u);
            if (!drop && rowmask == 0) {  // complete layout with k < limit supports
                sm.ring[step & 31u][tid] = (uint16_t)NONE;  // every consumed step owns its slot (stale entries are 32 steps old)
                best = k;
                limit = min(epoch_bound, best);
                R.list_to_rows(k, st.bestS);
                step++; my_steps++;
                hs = hs_next;
                if (k <= target || k == 0) { done = 1; break; }
                continue;
            }
            uint32_t removed = NONE;
            if (drop || (k > 0 && k == limit - 1)) {
                // ---- removal: min-loss support, random ties; supports younger than the tenure only as a last resort (not when
                // dropping)
                const uint32_t stephi = (step << 16) | 0xffffu;
                const uint32_t young_below = drop ? 0u : (uint32_t)ten << 16;
                pf.mark(PH_FRAME);
                removed = (uint32_t)R.remove(hs, stephi, young_below, k, rowmask, pf);
                pf.mark(PH_RFLIP);
                scored += (unsigned)k;
                k--;
                flips++;
            }
            sm.ring[step & 31u][tid] = (uint16_t)removed;
            if (!drop) {
                // ---- addition at a random uncovered tile t: best-gain site of R(t)
                pf.mark(PH_FRAME);
                const auto N = R.fetch(rowmask, hs);
                const bool noise = ((hs >> 10) & 127u) < nq7;
                const int v = add_site(sm, tid, N, hs, step, ten, noise, removed, recent, pf);
                pf.mark(PH_CAND);
                R.add(v, step, k, rowmask);
                pf.mark(PH_AFLIP);
                if (!noise) scored += (unsigned)(__popc(N.wt.x) + __popc(N.wt.y));
                k++;
                flips++;
            }
            step++; my_steps++;
            hs = hs_next;
        }

        R.list_to_rows(k, st.S);
        st.k = k; st.best = best; st.step = step; st.done = done;
        const unsigned long long tot = ((unsigned long long)st.scored_hi << 32 | st.scored_lo) + scored;
        st.scored_lo = (uint32_t)tot; st.scored_hi = (uint32_t)(tot >> 32);
        st.steps_done += (uint32_t)my_steps;
    }
    pf.flush((unsigned long long)my_steps);
    // one pair of atomics per warp
    unsigned long long a = scored, b = (unsigned long long)my_steps, c = (unsigned long long)flips;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); c += __shfl_xor_sync(0xffffffffu, c, o); }
    if ((tid & 31) == 0 && (a | b)) { atomicAdd(&totals[0], a); atomicAdd(&totals[1], b); atomicAdd(&totals[2], c); }
}

// the launch of a thread-per-chain kernel with its whole shared-memory block
template <class Kernel>
int launch(Kernel kernel, size_t smem_bytes, tss_engine* e, const uint32_t* rows_dev, const uint2* tabs_dev, ChainState* states, uint32_t* site_lists,
           int n_chains, int chains_per_terrain, uint32_t chain_offset, uint64_t seed, long long steps, const int* bounds_dev, int target,
           int noise_pct, unsigned long long* totals_dev) {
    // (idempotent and cheap; several engines / host threads may get here at once, so no "already set" cache)
    TSS_CUDA(e, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes));
    const size_t stride = ((size_t)n_chains + 31) & ~(size_t)31;
    const int blocks = (n_chains + NT - 1) / NT;
    kernel<<<blocks, NT, smem_bytes, e->stream>>>(rows_dev, tabs_dev, states, site_lists, stride, n_chains, chains_per_terrain, chain_offset, seed,
                                                   steps, bounds_dev, target, noise_pct, e->interrupt_dev, totals_dev);
    TSS_CHECK_LAUNCH(e);
    e->stats.kernel_launches++;
    return TSS_OK;
}

}  // namespace slsth
}  // namespace tss
