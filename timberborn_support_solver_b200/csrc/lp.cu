// FRACTIONAL packing lower bound (the LP dual of the support-placement relaxation), solved on the GPU and certified in
// integer arithmetic.  Not in the reference; it is the strengthening of lb.cu's integral packing that closes the proof on
// test/ex2.toml and the README terrain with 1x1 supports (LP optimum 13.2 / 13.13 -> bound 14 = the optimum), where the
// reference spends "minutes (or even hours)" (README.md:31) and the exact solver here ~10 s on the UNSAT call alone.
//
//     maximise  sum_t y_t   subject to   sum_{t in reach(p)} y_t <= 1  for every in-bounds placement p,   y >= 0
//
// reach(p) = validate()'s rule for the single platform p: the ceiling under its footprint plus three ceiling-masked
// 4-neighbour dilations (src/encoder/platform_layout.rs:104-141).  Any complete layout L satisfies
// |L| >= sum_{p in L} sum_{t in reach(p)} y_t >= sum_t y_t, so ceil(sum y) bounds the platform count from below (an integral
// y is lb.cu's packing).  Weak duality needs y to be FEASIBLE, nothing else, so the certificate never trusts the floating
// point solve: the solution is rounded to integer weights k_t = floor(y_t * 2^20), a second kernel recomputes every
// placement's load sum_{t in reach(p)} k_t from the reach bitboards in 64-bit integers, and the bound is
// ceil(sum k / max load) — exact, whatever the simplex did (a primal simplex iterate is feasible at every pivot, so an
// iteration cap only weakens the bound).
//
// Kernels: lp_reach_kernel (one warp per placement: footprint, dilations -> 32 row words), lp_init_kernel (dense condensed
// tableau [m + 1][n + 1] in doubles: constraints x ceiling tiles, right-hand side, objective row), lp_simplex_kernel (ONE CTA
// of 1024 threads: Devex pricing, ratio test, rank-1 update with the pivot row staged in shared memory; the
// instances are a few hundred columns, launch-free pivoting beats a multi-CTA update with grid syncs), lp_simplex_cluster_kernel
// (tableaus up to ~1.6 MB: rows resident in the shared memory of an 8-CTA thread-block cluster, exchange over distributed
// shared memory), lp_certify_kernel (integer loads).
#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>

#include "engine.hpp"

namespace cg = cooperative_groups;

namespace tss {
namespace lp {

constexpr uint32_t FULL = 0xffffffffu;
constexpr int MAX_KEYS = 16;
constexpr int THREADS = 1024;
constexpr int MAX_COLS = 1024;                 // ceiling tiles of a 32x32 grid
constexpr double EPS = 1e-9;
// integer weights k_t = floor(y_t * scale); scale = 2^20 for costs up to 1024, smaller powers of two above (k_t fits an int)

struct Keys {
    int n;
    int w[MAX_KEYS], h[MAX_KEYS];
    int cost[MAX_KEYS];   // what a platform of this key costs: 1 for the platform count, the GUI's total_weight otherwise
};

__device__ __forceinline__ uint32_t dilate(uint32_t X, uint32_t C, int lane) {
    uint32_t up = __shfl_up_sync(FULL, X, 1), down = __shfl_down_sync(FULL, X, 1);
    if (lane == 0) up = 0;
    if (lane == 31) down = 0;
    return (X | (X << 1) | (X >> 1) | up | down) & C;
}

// reach rows of every placement (key, anchor): out[(key * 1024 + y * 32 + x) * 32 + row]; all zero if the footprint leaves
// the grid (forbidden, src/encoder.rs:601-609) or covers no ceiling.  nonempty[placement] = 1 if it supports anything.
__global__ void __launch_bounds__(128) lp_reach_kernel(const uint32_t* __restrict__ rows, int W, int H, Keys keys, uint32_t* __restrict__ out,
                                                       uint8_t* __restrict__ nonempty) {
    const int lane = threadIdx.x & 31, p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= keys.n * 1024) return;
    const int k = p >> 10, x = p & 31, y = (p >> 5) & 31, w = keys.w[k], h = keys.h[k];
    const uint32_t C = rows[lane];
    uint32_t X = 0;
    if (x + w <= W && y + h <= H && lane >= y && lane < y + h) X = ((w >= 32 ? FULL : ((1u << w) - 1u)) << x) & C;
#pragma unroll
    for (int r = 0; r < kTerrainSupportDistance - 1; r++) X = dilate(X, C, lane);
    out[(size_t)p * 32 + lane] = X;
    const bool any = __any_sync(FULL, X != 0);
    if (lane == 0) nonempty[p] = any ? 1 : 0;
}

// condensed tableau, row-major with leading dimension ld = n + 1: rows 0..m-1 = constraints (column j = tile col_site[j],
// column n = right-hand side), row m = objective (-1 per tile, value 0)
__global__ void lp_init_kernel(const uint32_t* __restrict__ reach, const int* __restrict__ cons, int m, const int* __restrict__ col_site, int n,
                               double* __restrict__ T, double perturb, Keys keys) {
    const int ld = n + 1;
    const long long total = (long long)(m + 1) * ld;
    for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(idx / ld), j = (int)(idx % ld);
        double v;
        if (i == m) v = j < n ? -1.0 : 0.0;
        else if (j == n) v = (double)keys.cost[cons[i] >> 10] * (1.0 + perturb * (double)((i * 37) % 101) / 101.0);   // cost of the placement; tiny perturbation against degenerate ties (the certificate is exact anyway)
        else {
            const int s = col_site[j];
            v = (double)((reach[(size_t)cons[i] * 32 + (s >> 5)] >> (s & 31)) & 1u);
        }
        T[idx] = v;
    }
}

struct ArgD { double v; int i; };
__device__ __forceinline__ ArgD better_min(ArgD a, ArgD b) { return (b.v < a.v || (b.v == a.v && b.i < a.i)) ? b : a; }

// block-wide argmin with lowest-index ties (1024 threads); result valid in every thread
__device__ ArgD block_argmin(ArgD a, ArgD* red) {
    for (int o = 16; o > 0; o >>= 1) {
        ArgD b{__shfl_xor_sync(FULL, a.v, o), __shfl_xor_sync(FULL, a.i, o)};
        a = better_min(a, b);
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();
    if (lane == 0) red[warp] = a;
    __syncthreads();
    ArgD r = red[lane < (int)(blockDim.x >> 5) ? lane : 0];
    for (int o = 16; o > 0; o >>= 1) {
        ArgD b{__shfl_xor_sync(FULL, r.v, o), __shfl_xor_sync(FULL, r.i, o)};
        r = better_min(r, b);
    }
    return r;
}

// Primal simplex on the condensed tableau, all-slack start (y = 0 is feasible).  basis[i] = label of row i, nonbasis[j] =
// label of column j; labels 0..n-1 are tiles, n.. are slacks.  info[0] = pivots, info[1] = 1 if optimal.
__global__ void __launch_bounds__(THREADS) lp_simplex_kernel(double* __restrict__ T, int m, int n, int* __restrict__ basis, int* __restrict__ nonbasis,
                                                            int max_pivots, double stop_at, int* __restrict__ info) {
    __shared__ double prow[MAX_COLS + 1];
    __shared__ double devex[MAX_COLS + 1];   // Devex reference weights of the non-basic columns (see the cluster kernel)
    __shared__ ArgD red[32];
    const int ld = n + 1, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, n_warps = blockDim.x >> 5;
    for (int i = tid; i < m; i += blockDim.x) basis[i] = n + i;
    for (int j = tid; j < n; j += blockDim.x) { nonbasis[j] = j; devex[j] = 1.0; }
    __syncthreads();
    int pivots = 0, optimal = 0;
    for (; pivots < max_pivots; pivots++) {
        // entering column: Devex pricing, largest d_j^2 / w_j among the improving columns, lowest index on ties
        ArgD e{0.0, 0x7fffffff};
        for (int j = tid; j < n; j += blockDim.x) {
            const double d = T[(size_t)m * ld + j];
            if (d < -EPS) e = better_min(e, ArgD{-d * d / devex[j], j});
        }
        e = block_argmin(e, red);
        if (e.i == 0x7fffffff) { optimal = 1; break; }
        const int q = e.i;
        // ratio test over the rows with a positive entry in column q
        ArgD r{1e300, 0x7fffffff};
        for (int i = tid; i < m; i += blockDim.x) {
            const double a = T[(size_t)i * ld + q];
            if (a > EPS) r = better_min(r, ArgD{T[(size_t)i * ld + n] / a, i});
        }
        r = block_argmin(r, red);
        if (r.i == 0x7fffffff) break;   // unbounded: cannot happen (every tile lies in its own site's reach), never spin on it
        const int pr = r.i;
        const double piv = T[(size_t)pr * ld + q], inv = 1.0 / piv;
        __syncthreads();
        for (int j = tid; j <= n; j += blockDim.x) prow[j] = j == q ? inv : T[(size_t)pr * ld + j] * inv;   // the new pivot row
        __syncthreads();
        // rank-1 update: a warp per row, lanes across the columns (coalesced); the objective row is row m
        for (int i = warp; i <= m; i += n_warps) {
            double* row = T + (size_t)i * ld;
            if (i == pr) {
                for (int j = lane; j <= n; j += 32) row[j] = prow[j];
                continue;
            }
            const double f = row[q];
            __syncwarp();               // every lane has read the multiplier before lane q % 32 overwrites it
            if (f == 0.0) continue;     // (0/1 rows: most rows do not touch the entering column)
            for (int j = lane; j <= n; j += 32) row[j] = j == q ? -f * inv : row[j] - f * prow[j];
        }
        const double wq = devex[q];
        __syncthreads();
        for (int j = tid; j < n; j += blockDim.x) devex[j] = j == q ? fmax(wq * inv * inv, 1.0) : fmax(devex[j], prow[j] * prow[j] * wq);
        if (tid == 0) { const int t = basis[pr]; basis[pr] = nonbasis[q]; nonbasis[q] = t; }
        __syncthreads();
        if (stop_at > 0.0 && T[(size_t)m * ld + n] >= stop_at) { pivots++; break; }   // the bound the caller asked about is reached
    }
    if (tid == 0) { info[0] = pivots; info[1] = optimal; }
}

// ---- the same simplex for tableaus that fit the shared memory of a thread-block CLUSTER (8 CTAs: up to ~1.6 MB) --------------
// The single-CTA kernel above is bound by what ONE SM can move to and from L2: a pivot rewrites the whole tableau (450 KB for
// test/ex2.toml with 1x1 supports), ~20 us per pivot (ncu: long-scoreboard stalls 11 of 17, issue slots 35 %).  Here the
// constraint rows are dealt out to the 8 CTAs of one cluster and never leave shared memory; what every CTA needs of the others
// travels over distributed shared memory: the local winners of the ratio test are written into every CTA's slot array, the
// pivot row is pulled from its owner's shared memory.  Objective row, basis labels and the choice of the entering column are
// replicated (every CTA computes them from identical inputs in identical order, so they agree bit for bit).  Two cluster
// barriers per pivot.
constexpr int CLUSTER = 8;
constexpr int CL_THREADS = 512;

// 1 / x for the pivot arithmetic: single-precision reciprocal refined by two Newton steps in double precision (error ~1 ulp).  An
// IEEE double division is a chain of ~20 dependent FP64 operations (~800 cycles measured here, and every pivot has three of them on
// its critical path); this is 5.  The certificate does not depend on it: it is recomputed in integers (lp_certify_kernel).
__device__ __forceinline__ double fast_rcp(double x) {
    double r = (double)(1.0f / (float)x);
    r = r * (2.0 - x * r);
    r = r * (2.0 - x * r);
    return r;
}

// Devex pricing key d^2 / w.  The reference weights only grow (past 2^120 on full rectangles of 16x16 and more).  Beyond that the single-precision
// seed of fast_rcp flushes to zero (--use_fast_math), which priced improving columns at 0 and ended the simplex short of the optimum
// with the optimal flag set (full 32x32 grid, 1x1 supports: 45.70 of 46.90).  Such weights take an exact division.
__device__ __forceinline__ double devex_key(double d, double w) { return d * d * (w < 0x1p120 ? fast_rcp(w) : 1.0 / w); }

// Exact warp argmin over non-negative doubles (lowest index on ties) in three 32-bit REDUX instructions instead of five shuffle
// rounds on (double, int) pairs: non-negative doubles order like their bit patterns, so reduce the high words, then the low words
// among the lanes that hold the minimum high word, then the indices among the lanes that hold both.  Lanes without a candidate
// pass v = +inf, i = 0x7fffffff.  Every lane gets the result.
__device__ __forceinline__ ArgD warp_argmin_nonneg(ArgD a) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(a.v);
    const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
    const unsigned mhi = __reduce_min_sync(FULL, hi);
    const unsigned mlo = __reduce_min_sync(FULL, hi == mhi ? lo : 0xffffffffu);
    const bool mine = hi == mhi && lo == mlo;
    const unsigned mi = __reduce_min_sync(FULL, mine ? (unsigned)a.i : 0xffffffffu);
    return ArgD{__longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo)), (int)mi};
}
// The same for a maximum (pricing: largest Devex ratio, lowest column on ties).  Lanes without a candidate pass v = 0, i = 0x7fffffff.
__device__ __forceinline__ ArgD warp_argmax_nonneg(ArgD a) {
    const unsigned long long bits = (unsigned long long)__double_as_longlong(a.v);
    const unsigned hi = (unsigned)(bits >> 32), lo = (unsigned)bits;
    const unsigned mhi = __reduce_max_sync(FULL, hi);
    const unsigned mlo = __reduce_max_sync(FULL, hi == mhi ? lo : 0u);
    const bool mine = hi == mhi && lo == mlo;
    const unsigned mi = __reduce_min_sync(FULL, mine ? (unsigned)a.i : 0xffffffffu);
    return ArgD{__longlong_as_double((long long)(((unsigned long long)mhi << 32) | mlo)), (int)mi};
}

__device__ __forceinline__ ArgD warp_argmin(ArgD a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ArgD b{__shfl_xor_sync(FULL, a.v, o), __shfl_xor_sync(FULL, a.i, o)};
        a = better_min(a, b);
    }
    return a;
}

// One pivot = one cluster barrier.  Measured on the first version (clock64 per stage, TSS_LP_PROF=1; 11 400 cycles per pivot on
// test/ex2.toml): the rank-1 update took 5 000 (an integer division per cell to find its row), pricing and the ratio test 1 700 +
// 1 500 (two block-wide reductions with two barriers each for 236 columns / 30 rows), pulling the pivot row out of its owner's
// shared memory 1 700 (dependent remote reads) and the two cluster barriers 650-850 each.  Now:
//   * warp 0 alone prices (8 columns per lane) and runs the ratio test over this CTA's rows (one per lane): shuffles only;
//   * every CTA then PUSHES its candidate — ratio and the whole candidate pivot row — into the shared memory of all eight CTAs
//     (remote stores do not stall; buffers alternate with the pivot's parity, so one barrier per pivot is enough: nobody can be two
//     barriers ahead of a CTA that still reads);
//   * after the barrier everybody picks the winner among the eight local copies and scales its row; the update walks rows by warp
//     (no divisions) and skips the rows that do not touch the entering column.
// Decisions are unchanged (same keys, same tie-breaks): the same pivot sequence and certificate as before.
__global__ void __cluster_dims__(CLUSTER, 1, 1) __launch_bounds__(CL_THREADS)
lp_simplex_cluster_kernel(const double* __restrict__ T, int m, int n, const int* __restrict__ col_site, int max_pivots, double stop_at, int* __restrict__ info,
                          int* __restrict__ weights /* [1024] zeroed */, double scale, long long* __restrict__ prof /* optional [8]: clock cycles per pivot stage */) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank(), tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, ld = n + 1;
    const int rows_per = (m + CLUSTER - 1) / CLUSTER, row0 = rank * rows_per, my_rows = max(0, min(rows_per, m - row0));
    extern __shared__ __align__(16) unsigned char dyn[];
    double* Tl = reinterpret_cast<double*>(dyn);            // [rows_per][ld] my constraint rows (right-hand side at [n])
    double* obj = Tl + (size_t)rows_per * ld;               // [ld] objective row (replicated)
    double* devex = obj + ld;                               // [ld] Devex reference weights of the non-basic columns (replicated)
    double* pcol = devex + ld;                              // [rows_per] my part of the entering column
    double* cand = pcol + rows_per;                         // [2][CLUSTER][ld] candidate pivot rows of all CTAs, by pivot parity
    ArgD* slots = reinterpret_cast<ArgD*>(cand + (size_t)2 * CLUSTER * ld);   // [2][CLUSTER] local winners of the ratio test
    int* basis = reinterpret_cast<int*>(slots + 2 * CLUSTER);                 // [m] (replicated)
    int* nonbasis = basis + m;                              // [n] (replicated)
    __shared__ ArgD red[CL_THREADS / 32];                   // per-warp pricing candidates of the next pivot (Devex ratio, column)
    for (int idx = tid; idx < my_rows * ld; idx += blockDim.x) Tl[idx] = T[(size_t)row0 * ld + idx];
    for (int j = tid; j <= n; j += blockDim.x) { obj[j] = T[(size_t)m * ld + j]; devex[j] = 1.0; }
    for (int i = tid; i < m; i += blockDim.x) basis[i] = n + i;
    for (int j = tid; j < n; j += blockDim.x) nonbasis[j] = j;
    __syncthreads();
    // Devex pricing (Forrest & Goldfarb): largest d_j^2 / w_j among the improving columns, the reference weights w_j approximating
    // the steepest-edge norms at the price of one pass over the pivot row (Dantzig's rule needs ~1 500 pivots on the 21x16
    // terrains, this ~760).  Every thread prices the columns it has just updated (one division each, all in parallel) and the
    // warps leave their candidates in `red`; the barrier that ends the pivot publishes them.
    auto price = [&]() {
        ArgD e{0.0, 0x7fffffff};
        for (int j = tid; j < n; j += blockDim.x) {
            const double d = obj[j];
            if (d < -EPS) {
                const double key = devex_key(d, devex[j]);
                // (columns ascend: the first of equal keys stays; every improving column is a candidate, even at key 0, so that
                // "no candidate" means no reduced cost below -EPS)
                if (key > e.v || e.i == 0x7fffffff) e = ArgD{key, j};
            }
        }
        e = warp_argmax_nonneg(e);
        if (lane == 0) red[warp] = e;
    };
    price();
    cluster.sync();
    int pivots = 0, optimal = 0;
    long long tprev = clock64(), acc[6] = {0, 0, 0, 0, 0, 0};
#define LP_LAP(i) do { if (prof && rank == 0 && tid == 0) { const long long t_ = clock64(); acc[i] += t_ - tprev; tprev = t_; } } while (0)
    for (; pivots < max_pivots; pivots++) {
        const int par = pivots & 1;
        const ArgD ent = warp_argmax_nonneg(red[lane & (CL_THREADS / 32 - 1)]);   // the entering column: every warp folds the 16 candidates itself
        if (ent.i == 0x7fffffff) { optimal = 1; break; }    // (identical in every CTA: nobody is left waiting at a barrier)
        const int q = ent.i;
        const double fo = obj[q], wq = devex[q];            // (read before the barrier below; rewritten after it)
        // ratio test over my rows, one per lane — by EVERY warp for itself (identical results, no block barrier to publish them)
        ArgD r{__longlong_as_double(0x7ff0000000000000ll), 0x7fffffff};   // +inf: no candidate
        for (int li = lane; li < my_rows; li += 32) {
            const double a = Tl[(size_t)li * ld + q];
            pcol[li] = a;                                   // (all warps store the same values)
            if (a > EPS) r = better_min(r, ArgD{fmax(Tl[(size_t)li * ld + n] * fast_rcp(a), 0.0), row0 + li});
        }
        r = warp_argmin_nonneg(r);
        __syncwarp();
        LP_LAP(0);
        if (r.i != 0x7fffffff) {                            // my candidate row into everybody's buffer
            const double* mine = Tl + (size_t)(r.i - row0) * ld;
            for (int j = tid; j <= n; j += blockDim.x) {
                const double v = mine[j];
#pragma unroll
                for (int c = 0; c < CLUSTER; c++) cluster.map_shared_rank(cand, c)[((size_t)par * CLUSTER + rank) * ld + j] = v;
            }
        }
        if (tid < CLUSTER) cluster.map_shared_rank(slots, tid)[par * CLUSTER + rank] = r;
        LP_LAP(1);
        cluster.sync();
        LP_LAP(2);
        const ArgD g = warp_argmin_nonneg(slots[par * CLUSTER + (lane & (CLUSTER - 1))]);   // the winner among the eight candidates
        if (g.i == 0x7fffffff) break;                       // unbounded: cannot happen, never spin on it
        const int pr = g.i, owner = pr / rows_per;
        const double* crow = cand + ((size_t)par * CLUSTER + owner) * ld;   // the pivot row before scaling: a local copy
        const double inv = fast_rcp(crow[q]);
        auto prow_at = [&](int j) { return j == q ? inv : crow[j] * inv; };   // element j of the new pivot row
        LP_LAP(3);
        // rank-1 update: a thread owns one column (two threads share it, even / odd rows) and walks down the rows, eight at a time with
        // all reads first; rows that do not touch the entering column (0/1 rows: most) cost one broadcast read
        for (int j = tid & (CL_THREADS / 2 - 1); j <= n; j += CL_THREADS / 2) {
            const double pj = prow_at(j);
            for (int li = tid / (CL_THREADS / 2); li < my_rows; li += 2) {
                const double f = pcol[li];                  // (uniform across the warp: no divergence)
                double* cell = Tl + (size_t)li * ld + j;
                if (row0 + li == pr) *cell = pj;
                else if (f != 0.0) *cell = j == q ? -f * inv : *cell - f * pj;
            }
        }
        LP_LAP(4);
        for (int j = tid; j <= n; j += blockDim.x) {        // objective row and Devex weights: prow[j] = alpha_rj / alpha_rq for j != q, prow[q] = 1 / alpha_rq
            const double pj = prow_at(j);
            obj[j] = j == q ? -fo * inv : obj[j] - fo * pj;
            if (j < n) devex[j] = j == q ? fmax(wq * inv * inv, 1.0) : fmax(devex[j], pj * pj * wq);
        }
        if (tid == 0) { const int t = basis[pr]; basis[pr] = nonbasis[q]; nonbasis[q] = t; }
        price();                                            // (each thread prices exactly the columns it has just written)
        __syncthreads();
        LP_LAP(5);
        if (stop_at > 0.0 && obj[n] >= stop_at) { pivots++; break; }   // the bound the caller asked about is reached (obj is replicated: every CTA leaves here)
    }
    for (int li = tid; li < my_rows; li += blockDim.x) {    // y -> integer weights: floor(y * SCALE) for my basic tiles
        const int label = basis[row0 + li];
        if (label >= n) continue;
        const double y = Tl[(size_t)li * ld + n];
        const long long k = y > 0.0 ? (long long)floor(y * scale) : 0ll;
        weights[col_site[label]] = (int)(k > (1ll << 30) ? (1ll << 30) : k);
    }
    if (rank == 0 && tid == 0) { info[0] = pivots; info[1] = optimal; }
    if (prof && rank == 0 && tid == 0)
        for (int i = 0; i < 6; i++) prof[i] = acc[i];
    cluster.sync();                                         // nobody exits while its shared memory may still be written remotely
}

// ---- the same simplex for tableaus beyond the cluster's shared memory: the whole device, one grid barrier per pivot ------------
// (default-8 platform sets: thousands of constraints; 1x1 supports on 24x24 .. 32x32 terrains — the GUI's default grid is 24x24,
// crates/gui/src/app.rs: tens of MB that stay in the 126 MB L2.)  The single-CTA kernel moves all of it through ONE SM, 50-130 us
// per pivot.  Here the constraint rows are dealt out to one CTA per SM (cooperative launch); objective row and Devex weights are
// replicated in every CTA's shared memory exactly as in the cluster kernel, so the entering column needs no exchange; every CTA
// publishes its ratio-test winner AND a copy of its candidate row in global memory (buffers alternate with the pivot's parity),
// one grid barrier, then everybody picks the winner among the slots, reads that row from L2 and updates its own rows in place.
constexpr int GRID_THREADS = 512;

__global__ void __launch_bounds__(GRID_THREADS, 1)
lp_simplex_grid_kernel(double* __restrict__ T, int m, int n, const int* __restrict__ col_site, int max_pivots, double stop_at, int* __restrict__ info,
                       int* __restrict__ weights /* [1024] zeroed */, double scale, int* __restrict__ basis /* [m] */, int* __restrict__ nonbasis /* [n] */,
                       double* __restrict__ cand /* [2][gridDim.x][ld] */, ArgD* __restrict__ slots /* [2][gridDim.x] */) {
    cg::grid_group grid = cg::this_grid();
    const int G = (int)gridDim.x, rank = (int)blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, ld = n + 1;
    const int rows_per = (m + G - 1) / G, row0 = rank * rows_per, my_rows = max(0, min(rows_per, m - row0));
    extern __shared__ __align__(16) unsigned char dyn[];
    double* obj = reinterpret_cast<double*>(dyn);           // [ld] objective row (replicated)
    double* devex = obj + ld;                               // [ld] Devex reference weights (replicated)
    double* pcol = devex + ld;                              // [rows_per] my part of the entering column
    __shared__ ArgD red[GRID_THREADS / 32];                 // per-warp pricing candidates of the next pivot
    __shared__ ArgD rred[GRID_THREADS / 32];                // per-warp ratio-test candidates
    for (int j = tid; j <= n; j += blockDim.x) { obj[j] = T[(size_t)m * ld + j]; devex[j] = 1.0; }
    if (rank == 0) {
        for (int i = tid; i < m; i += blockDim.x) basis[i] = n + i;
        for (int j = tid; j < n; j += blockDim.x) nonbasis[j] = j;
    }
    __syncthreads();
    auto price = [&]() {
        ArgD e{0.0, 0x7fffffff};
        for (int j = tid; j < n; j += blockDim.x) {
            const double d = obj[j];
            if (d < -EPS) {
                const double key = devex_key(d, devex[j]);
                if (key > e.v || e.i == 0x7fffffff) e = ArgD{key, j};
            }
        }
        e = warp_argmax_nonneg(e);
        if (lane == 0) red[warp] = e;
    };
    price();
    __syncthreads();
    int pivots = 0, optimal = 0;
    for (; pivots < max_pivots; pivots++) {
        const int par = pivots & 1;
        const ArgD ent = warp_argmax_nonneg(red[lane & (GRID_THREADS / 32 - 1)]);
        if (ent.i == 0x7fffffff) { optimal = 1; break; }    // (identical in every CTA: nobody is left waiting at the barrier)
        const int q = ent.i;
        const double fo = obj[q], wq = devex[q];
        ArgD r{__longlong_as_double(0x7ff0000000000000ll), 0x7fffffff};
        for (int li = tid; li < my_rows; li += blockDim.x) {   // ratio test over my rows (tableau in L2)
            const double a = T[(size_t)(row0 + li) * ld + q];
            pcol[li] = a;
            if (a > EPS) r = better_min(r, ArgD{fmax(T[(size_t)(row0 + li) * ld + n] * fast_rcp(a), 0.0), row0 + li});
        }
        r = warp_argmin_nonneg(r);
        if (lane == 0) rred[warp] = r;
        __syncthreads();
        r = warp_argmin_nonneg(rred[lane & (GRID_THREADS / 32 - 1)]);
        if (r.i != 0x7fffffff) {                            // my candidate row, copied out before anybody may rewrite it
            const double* mine = T + (size_t)r.i * ld;
            double* dst = cand + ((size_t)par * G + rank) * ld;
            for (int j = tid; j <= n; j += blockDim.x) dst[j] = mine[j];
        }
        if (tid == 0) slots[par * G + rank] = r;
        grid.sync();
        ArgD g{__longlong_as_double(0x7ff0000000000000ll), 0x7fffffff};
        for (int c = lane; c < G; c += 32) g = better_min(g, ArgD{__ldcg(&slots[par * G + c].v), __ldcg(&slots[par * G + c].i)});   // (L2 reads: written by other SMs)
        g = warp_argmin_nonneg(g);
        if (g.i == 0x7fffffff) break;                       // unbounded: cannot happen, never spin on it
        const int pr = g.i, owner = pr / rows_per;
        const double* crow = cand + ((size_t)par * G + owner) * ld;   // the pivot row before scaling
        const double inv = fast_rcp(__ldcg(&crow[q]));
        for (int j = tid & (GRID_THREADS / 2 - 1); j <= n; j += GRID_THREADS / 2) {   // rank-1 update of my rows: a thread owns a column, even / odd rows
            const double pj = j == q ? inv : __ldcg(&crow[j]) * inv;
            for (int li = tid / (GRID_THREADS / 2); li < my_rows; li += 2) {
                const double f = pcol[li];
                double* cell = T + (size_t)(row0 + li) * ld + j;
                if (row0 + li == pr) *cell = pj;
                else if (f != 0.0) *cell = j == q ? -f * inv : *cell - f * pj;
            }
        }
        for (int j = tid; j <= n; j += blockDim.x) {
            const double pj = j == q ? inv : __ldcg(&crow[j]) * inv;
            obj[j] = j == q ? -fo * inv : obj[j] - fo * pj;
            if (j < n) devex[j] = j == q ? fmax(wq * inv * inv, 1.0) : fmax(devex[j], pj * pj * wq);
        }
        if (rank == 0 && tid == 0) { const int t = basis[pr]; basis[pr] = nonbasis[q]; nonbasis[q] = t; }
        price();
        __syncthreads();
        if (stop_at > 0.0 && obj[n] >= stop_at) { pivots++; break; }
    }
    grid.sync();                                            // basis labels (written by CTA 0) and every row are final
    for (int li = tid; li < my_rows; li += blockDim.x) {    // y -> integer weights: floor(y * SCALE) for my basic tiles
        const int label = basis[row0 + li];
        if (label >= n) continue;
        const double y = T[(size_t)(row0 + li) * ld + n];
        const long long k = y > 0.0 ? (long long)floor(y * scale) : 0ll;
        weights[col_site[label]] = (int)(k > (1ll << 30) ? (1ll << 30) : k);
    }
    if (rank == 0 && tid == 0) { info[0] = pivots; info[1] = optimal; }
}

// y -> integer weights per site (floor(y * SCALE), never negative), zero for non-basic tiles
__global__ void lp_weights_kernel(const double* __restrict__ T, int m, int n, const int* __restrict__ basis, const int* __restrict__ col_site,
                                  int* __restrict__ weights /* [1024] zeroed */, double scale) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int label = basis[i];
    if (label >= n) return;
    const double y = T[(size_t)i * (n + 1) + n];
    const long long k = y > 0.0 ? (long long)floor(y * scale) : 0ll;
    weights[col_site[label]] = (int)(k > (1ll << 30) ? (1ll << 30) : k);
}

// exact certificate, all in 64-bit integers.  out[0] = sum of the weights k_t (lp_total_kernel).  For every in-bounds placement p (ALL
// of them, not only the tableau's rows) with load(p) = sum of the weights in its reach: a layout L costs sum_{p in L} cost(p) and
// covers every tile, so  total <= sum_{p in L} load(p) <= (max_p load(p) / cost(p)) * cost(L):  cost(L) >= total * cost(p) / load(p)
// for the placement with the worst ratio.  out[1] = max load, out[2] = min over placements of ceil(total * cost(p) / load(p)) — the
// bound.  With unit costs that is ceil(total / max load).
__global__ void lp_total_kernel(const int* __restrict__ weights, unsigned long long* __restrict__ out) {
    long long s = 0;
    for (int t = threadIdx.x; t < 1024; t += 32) s += weights[t];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
    if (threadIdx.x == 0) out[0] = (unsigned long long)s;
}
__global__ void __launch_bounds__(128) lp_certify_kernel(const uint32_t* __restrict__ reach, int n_placements, const int* __restrict__ weights, Keys keys,
                                                         unsigned long long* __restrict__ out) {
    const int lane = threadIdx.x & 31, p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= n_placements) return;
    long long load = 0;
    for (uint32_t bits = reach[(size_t)p * 32 + lane]; bits; bits &= bits - 1) load += weights[lane * 32 + __ffs(bits) - 1];
    for (int o = 16; o > 0; o >>= 1) load += __shfl_xor_sync(FULL, load, o);
    if (lane == 0 && load > 0) {
        const unsigned long long total = out[0], num = total * (unsigned long long)keys.cost[p >> 10];
        atomicMax(&out[1], (unsigned long long)load);
        atomicMin(&out[2], (num + (unsigned long long)load - 1ull) / (unsigned long long)load);
    }
}

}  // namespace lp

// rows32_host: terrain rows; key_dims: effective (w, h) per dims key.  out_weights (host, 1024 ints, index y * 32 + x),
// key_costs: cost of a platform per key.  totals[0] = sum of the weights, totals[1] = largest placement load, totals[2] = the bound
// (min over placements of ceil(total * cost / load); ~0 if no placement carries load), info[0] = pivots, info[1] = optimal, info[2] = constraints.
int lp_run(tss_engine* e, const uint32_t* rows32_host, int W, int H, const std::vector<int2>& key_dims, const std::vector<int>& key_costs, int max_pivots,
           long long target, int* out_weights, unsigned long long* totals, int* info) {
    if ((int)key_dims.size() > lp::MAX_KEYS) return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound_lp: more than %d dims keys", lp::MAX_KEYS);
    lp::Keys keys;
    keys.n = (int)key_dims.size();
    int max_cost = 1;
    for (int i = 0; i < keys.n; i++) {
        keys.w[i] = key_dims[(size_t)i].x; keys.h[i] = key_dims[(size_t)i].y; keys.cost[i] = key_costs[(size_t)i];
        max_cost = key_costs[(size_t)i] > max_cost ? key_costs[(size_t)i] : max_cost;
    }
    double scale = (double)(1 << 20);            // y_t <= the largest cost: keep floor(y * scale) below 2^30
    while (scale * (double)max_cost > (double)(1 << 30)) scale *= 0.5;
    const int n_place = keys.n * 1024;
    std::vector<int> col_site;
    for (int s = 0; s < 1024; s++)
        if ((rows32_host[s >> 5] >> (s & 31)) & 1u) col_site.push_back(s);
    const int n = (int)col_site.size();
    totals[0] = totals[1] = totals[2] = 0;
    info[0] = info[1] = info[2] = 0;
    for (int i = 0; i < 1024; i++) out_weights[i] = 0;
    if (n == 0) return TSS_OK;
    // scratch slot 6: rows [32] | reach [n_place][32] | nonempty [n_place] bytes ; slot 7 is lb.cu's
    const size_t reach_words = (size_t)n_place * 32;
    uint32_t* buf = (uint32_t*)e->dev(6, sizeof(uint32_t) * (32 + reach_words) + (size_t)n_place);
    if (!buf) return TSS_E_CUDA;
    uint32_t *rows_dev = buf, *reach = buf + 32;
    uint8_t* nonempty = (uint8_t*)(reach + reach_words);
    TSS_CUDA(e, cudaMemcpyAsync(rows_dev, rows32_host, sizeof(uint32_t) * 32, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaEventRecord(e->ev0, e->stream));
    lp::lp_reach_kernel<<<(n_place + 3) / 4, 128, 0, e->stream>>>(rows_dev, W, H, keys, reach, nonempty);
    TSS_CHECK_LAUNCH(e);
    std::vector<uint8_t> ne((size_t)n_place);
    TSS_CUDA(e, cudaMemcpyAsync(ne.data(), nonempty, (size_t)n_place, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    std::vector<int> cons;
    for (int p = 0; p < n_place; p++)
        if (ne[(size_t)p]) cons.push_back(p);
    const int m = (int)cons.size();
    info[2] = m;
    const size_t cells = (size_t)(m + 1) * (n + 1);
    if (cells > ((size_t)1 << 27)) return e->fail(TSS_E_UNSUPPORTED, "tss_lower_bound_lp: tableau of %d x %d exceeds the supported size", m, n);
    // scratch slot 5: tableau doubles | cons [m] | col_site [n] | basis [m] | nonbasis [n] | weights [1024] | info [4] | totals [2] u64
    const size_t ints = (size_t)m + n + m + n + 1024 + 4;
    double* T = (double*)e->dev(5, sizeof(double) * cells + sizeof(int) * ints + 16 + 24);
    if (!T) return TSS_E_CUDA;
    int* cons_dev = (int*)(T + cells);
    int *col_dev = cons_dev + m, *basis = col_dev + n, *nonbasis = basis + m, *weights = nonbasis + n, *info_dev = weights + 1024;
    unsigned long long* totals_dev = (unsigned long long*)(((uintptr_t)(info_dev + 4) + 15) & ~(uintptr_t)15);
    TSS_CUDA(e, cudaMemcpyAsync(cons_dev, cons.data(), sizeof(int) * (size_t)m, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(col_dev, col_site.data(), sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    TSS_CUDA(e, cudaMemsetAsync(weights, 0, sizeof(int) * (1024 + 4), e->stream));
    TSS_CUDA(e, cudaMemsetAsync(totals_dev, 0, sizeof(unsigned long long) * 2, e->stream));
    TSS_CUDA(e, cudaMemsetAsync(totals_dev + 2, 0xff, sizeof(unsigned long long), e->stream));   // running minimum
    const int init_blocks = (int)((cells + 255) / 256 < (size_t)e->prop.multiProcessorCount * 8 ? (cells + 255) / 256 : (size_t)e->prop.multiProcessorCount * 8);
    // (the size of the perturbation does not matter: 0 .. 1e-3 all need 1 300 - 1 800 pivots on the 21x16 terrains — the pivot count is
    // Dantzig pricing on this LP, not degenerate stalling)
    lp::lp_init_kernel<<<init_blocks, 256, 0, e->stream>>>(reach, cons_dev, m, col_dev, n, T, 1e-7, keys);
    const int pivots_cap = max_pivots > 0 ? max_pivots : 8 * (m + n);
    // target > 0: the caller only asks whether the bound reaches `target`.  Every iterate is feasible and the objective only grows,
    // so the simplex may stop once it exceeds target - 1 by more than the certificate loses to rounding (floor(y * scale) per
    // tile: < n / scale in total; right-hand sides perturbed by 1e-7): the loop's question "nothing within target - 1?" is usually
    // settled after 60-80 % of the pivots (ex2 / README terrain with 1x1 supports: 13.0 is passed long before the optimum 13.2 / 13.13)
    const double stop_at = target > 0 ? (double)(target - 1) + 4.0 * (double)n / scale + 2e-3 : 0.0;
    const int rows_per = (m + lp::CLUSTER - 1) / lp::CLUSTER, ld = n + 1;
    const size_t cl_smem = sizeof(double) * ((size_t)rows_per * ld + 2 * (size_t)ld + rows_per + 2 * (size_t)lp::CLUSTER * ld) + sizeof(lp::ArgD) * 2 * lp::CLUSTER +
                           sizeof(int) * ((size_t)m + n);
    const char* force = getenv("TSS_LP_SINGLE_CTA");       // (A/B switch for profiles/lb_stream.py)
    // TSS_LP_PROF=1: clock cycles of CTA 0 per pivot stage on stderr (pricing, ratio test, slot exchange + barrier, pivot row pull, barrier, update)
    long long* prof_dev = nullptr;
    if (getenv("TSS_LP_PROF")) prof_dev = (long long*)e->dev(7, sizeof(long long) * 8);
    if (cl_smem <= 200 * 1024 && !(force && force[0] == '1')) {
        // the tableau fits the shared memory of one 8-CTA cluster: rows resident in shared memory, exchange over DSMEM
        TSS_CUDA(e, cudaFuncSetAttribute(lp::lp_simplex_cluster_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cl_smem));
        if (lp::CLUSTER > 8) TSS_CUDA(e, cudaFuncSetAttribute(lp::lp_simplex_cluster_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
        lp::lp_simplex_cluster_kernel<<<lp::CLUSTER, lp::CL_THREADS, cl_smem, e->stream>>>(T, m, n, col_dev, pivots_cap, stop_at, info_dev, weights, scale, prof_dev);
    } else {
        // beyond the cluster: one CTA per SM, cooperative launch, one grid barrier per pivot (TSS_LP_SINGLE_CTA=1: the one-CTA kernel)
        int coop = 0;
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, e->device);
        const int G = std::max(1, std::min(e->prop.multiProcessorCount, (m + 3) / 4));
        const size_t g_smem = sizeof(double) * (2 * (size_t)ld + (size_t)((m + G - 1) / G));
        double* cand = nullptr;
        if (coop && !(force && force[0] == '1') && g_smem <= 200 * 1024) cand = (double*)e->dev(4, sizeof(double) * 2 * (size_t)G * ld + sizeof(lp::ArgD) * 2 * (size_t)G + 64);
        if (cand) {
            lp::ArgD* slots = reinterpret_cast<lp::ArgD*>(cand + 2 * (size_t)G * ld);
            int m_ = m, n_ = n, cap_ = pivots_cap;
            double stop_ = stop_at, scale_ = scale;
            const int* col_ = col_dev;
            void* args[] = {&T, &m_, &n_, &col_, &cap_, &stop_, &info_dev, &weights, &scale_, &basis, &nonbasis, &cand, &slots};
            TSS_CUDA(e, cudaFuncSetAttribute(lp::lp_simplex_grid_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g_smem));
            TSS_CUDA(e, cudaLaunchCooperativeKernel((const void*)lp::lp_simplex_grid_kernel, dim3(G), dim3(lp::GRID_THREADS), args, g_smem, e->stream));
        } else {
            lp::lp_simplex_kernel<<<1, lp::THREADS, 0, e->stream>>>(T, m, n, basis, nonbasis, pivots_cap, stop_at, info_dev);
            lp::lp_weights_kernel<<<(m + 255) / 256, 256, 0, e->stream>>>(T, m, n, basis, col_dev, weights, scale);
        }
    }
    lp::lp_total_kernel<<<1, 32, 0, e->stream>>>(weights, totals_dev);
    lp::lp_certify_kernel<<<(n_place + 3) / 4, 128, 0, e->stream>>>(reach, n_place, weights, keys, totals_dev);
    TSS_CHECK_LAUNCH(e);
    TSS_CUDA(e, cudaEventRecord(e->ev1, e->stream));
    e->stats.kernel_launches += 5;
    TSS_CUDA(e, cudaMemcpyAsync(out_weights, weights, sizeof(int) * 1024, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(info, info_dev, sizeof(int) * 2, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaMemcpyAsync(totals, totals_dev, sizeof(unsigned long long) * 3, cudaMemcpyDeviceToHost, e->stream));
    TSS_CUDA(e, cudaStreamSynchronize(e->stream));
    float ms = 0;
    if (cudaEventElapsedTime(&ms, e->ev0, e->ev1) != cudaSuccess) cudaGetLastError();
    e->stats.device_ms = ms;
    if (prof_dev && info[0] > 0 && cl_smem <= 200 * 1024) {
        long long prof[6];
        TSS_CUDA(e, cudaMemcpy(prof, prof_dev, sizeof prof, cudaMemcpyDeviceToHost));
        static const char* const names[6] = {"fold pricing + ratio test", "push candidate rows", "cluster barrier", "pick pivot row", "row update", "objective / devex / pricing"};
        for (int i = 0; i < 6; i++) std::fprintf(stderr, "[lp prof] %-30s %8.0f cycles per pivot\n", names[i], (double)prof[i] / info[0]);
    }
    return TSS_OK;
}

}  // namespace tss
