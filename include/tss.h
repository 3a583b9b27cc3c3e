/* tss.h — C ABI of libtss, the B200 (sm_100a) upper-bound engine for Timberborn ceiling-support placement.
 *
 * Drop-in boundary for ONE path of MetaflameDragon/timberborn_support_solver: the feasibility-and-bound loop
 * (encode -> bound -> CNF -> solve -> decode -> validate -> tighten).  Every entry point cites the reference
 * interface (file:line, relative to the reference tree) it stands behind; INTEGRATION.md shows the Rust
 * `extern "C"` block + safe wrapper a maintainer would add.
 *
 * Conventions (SURVEY.md §8b)
 *   - grids are row-major u8, index x + y*width, non-zero = ceiling           (src/math/grid.rs:66-68, src/world.rs:19)
 *   - a platform is (x, y) of its min-x/min-y corner + CANONICAL def dims (w <= h as in PLATFORMS_DEFAULT)
 *     + `rotated` (effective dims flipped)                                      (src/platform.rs:64-70,111-113)
 *   - literals are DIMACS-signed int32 over 1-based variables (rustsat Var idx + 1)
 *   - assignments are u8 per variable, index = variable (slot 0 unused): 0 False, 1 True, 2 DontCare (rustsat TernaryVal)
 *   - bit-packed grids ("rows"): each grid row is ceil(width/32) little-endian u32 words, bit (x & 31) of word
 *     (x >> 5) = tile (x, y); unused high bits are zero
 *   - all buffers are caller-allocated HOST memory unless the name ends in `_dev`; the engine never keeps a
 *     caller pointer after the call returns; outputs that do not fit return TSS_E_CAPACITY
 *   - no exceptions / aborts cross this boundary; every call returns a status (>= 0 ok, < 0 error) and
 *     tss_last_error() describes the last failure on that engine
 *   - the GPU path has NO CPU fallback: without a usable CUDA device tss_engine_create fails with TSS_E_CUDA
 */
#ifndef TSS_H
#define TSS_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TSS_VERSION 103

/* status codes; solve results follow IPASIR / rustsat SolverResult (crates/repl/src/main.rs:326-339) */
#define TSS_OK 0
#define TSS_UNKNOWN 0       /* budget exhausted or interrupted: no layout within the bound was found (NOT a proof) */
#define TSS_SAT 10          /* a validated layout within the bound was found */
#define TSS_UNSAT 20        /* never produced by a SEARCH (the exact solver proves UNSAT); tss_solve_instance returns it when the limit lies
                               below a certified lower bound (tss_lower_bound / tss_lower_bound_lp) */
#define TSS_E_INVALID (-1)  /* bad argument (null pointer, zero-sized grid, platform set without 1x1, ...) */
#define TSS_E_CAPACITY (-2) /* an output buffer is too small; the required size is reported where documented */
#define TSS_E_CUDA (-3)     /* CUDA runtime failure or no device */
#define TSS_E_UNSUPPORTED (-4) /* valid input outside what this build accelerates (e.g. grid larger than 256x256 for SLS) */
#define TSS_E_PARSE (-5)    /* project file rejected (src/world.rs:49-79) */

typedef struct tss_engine tss_engine;     /* one per GPU / CUDA stream; single caller except tss_interrupt */
typedef struct tss_encoding tss_encoding; /* host-side Encoding (src/encoder.rs:428-432) */
typedef struct tss_cnf tss_cnf;           /* a CNF resident on the device in CSR form */
typedef struct tss_search tss_search;     /* a device-resident SLS portfolio on one terrain */

/* src/platform.rs:64-70 Platform {point, def, rotated} */
typedef struct tss_platform {
    int32_t x, y;         /* anchor = min corner */
    int32_t def_w, def_h; /* canonical def dims */
    int32_t rotated;
} tss_platform;

/* src/platform.rs:11-15 PlatformDef */
typedef struct tss_dims {
    int32_t w, h;
} tss_dims;

/* rustsat SolveStats (crates/repl/src/main.rs:363) + engine counters */
typedef struct tss_stats {
    uint64_t layouts_evaluated;   /* full evaluations by the coverage kernel (a) */
    uint64_t candidates_scored;   /* candidate layouts scored incrementally by the SLS kernel (b) */
    uint64_t sls_steps;           /* swap / drop steps executed over all chains */
    uint64_t clauses_checked;     /* clause x assignment evaluations by the CNF kernel (c) */
    uint64_t kernel_launches;     /* kernels launched by this engine */
    uint64_t n_solves;            /* tss_solve_upper_bound / tss_search_run calls */
    double   device_ms;           /* device time of the kernels of the last call (CUDA events on the engine stream) */
    int32_t  best_count;          /* best platform count of the last solve (-1 if none) */
    int32_t  interrupted;         /* last solve ended by tss_interrupt */
    int64_t  last_solve_steps;    /* SLS steps per chain the last tss_solve_upper_bound call ran before it returned */
    uint64_t sls_flips;           /* supports (platforms) added + removed by the SLS kernels: one flip = one candidate layout
                                     evaluated incrementally (the unit of SURVEY.md §8(d)); candidates_scored counts the neighbour
                                     layouts scored to CHOOSE those flips */
} tss_stats;

/* ------------------------------------------------------------------------------------------------ engine */
int tss_version(void);
/* Bounds-checked build only (nvcc -DTSS_CHECKED, profiles/checked_build.py): shared-memory accesses of the thread-per-chain SLS kernels
 * that left their board since the library was loaded; -1 in the shipped build, which carries no checks. */
int tss_debug_smem_violations(void);
/* device < 0: current device.  Fails with TSS_E_CUDA when no CUDA device is usable (no CPU fallback). */
int tss_engine_create(int device, tss_engine** out);
void tss_engine_destroy(tss_engine* e);
/* Run the engine's kernels on a caller-owned cudaStream_t (e.g. the host framework's current stream) instead of
 * the engine's own stream.  NULL restores the engine stream. */
int tss_engine_set_stream(tss_engine* e, void* cuda_stream);
const char* tss_last_error(const tss_engine* e);
/* rustsat InterruptSolver::interrupt (crates/repl/src/main.rs:310-317, crates/gui/src/solver_backend.rs:47-49):
 * callable from any thread while a solve runs on `e`; the running call returns TSS_UNKNOWN with stats.interrupted. */
void tss_interrupt(tss_engine* e);
void tss_clear_interrupt(tss_engine* e);
int tss_get_stats(const tss_engine* e, tss_stats* out);
/* name[<=cap], SM count, max SM clock in kHz */
int tss_device_info(const tss_engine* e, char* name, int cap, int* sm_count, int* clock_khz);

/* ---------------------------------------------------------------------------- multi-GPU portfolio (SURVEY.md §8e) */
/* One process per GPU.  Rank 0 makes an id (tss_comm_unique_id), the host passes its 128 bytes to the other ranks, every
 * rank calls tss_comm_init.  From then on a search created with tss_search_create on this engine all-reduce-mins its
 * device-resident bound over NCCL/NVLink after every tss_search_run — 4 bytes, in-stream, no host round trip — so all
 * ranks must call tss_search_run the same number of times.  On grids larger than 32x32 (window decomposition) every rank
 * additionally adopts the best LAYOUT of all ranks after each phase (a second all-reduce-min over the bit-packed layout
 * in which only the winner contributes its bits).  The one-shot tss_solve_* calls never communicate.
 * NCCL is bound at run time (dlopen libnccl.so.2); TSS_E_UNSUPPORTED if it is not installed. */
int tss_comm_unique_id(tss_engine* e, uint8_t* out_id128);
int tss_comm_init(tss_engine* e, const uint8_t* id128, int32_t rank, int32_t world);
int tss_comm_world(const tss_engine* e);

/* --------------------------------------------------------------------------------- world (src/world.rs:49-79) */
/* Parses `[world] grid = ["XX ", ...]`.  Ragged rows are left-aligned and padded false as world.rs:82-86 documents
 * (the reference's copy_from_slice at :73 would panic instead; *ragged reports that case).  err gets a message. */
int tss_world_parse_toml(const char* text, uint8_t* grid, size_t cap, int32_t* w, int32_t* h, int32_t* ragged,
                         char* err, size_t err_cap);
/* world.rs:21-40 serialiser; returns bytes written (excl. NUL) or TSS_E_CAPACITY */
int tss_world_to_toml(const uint8_t* grid, int32_t w, int32_t h, char* out, size_t cap);
/* SURVEY.md §8(d) synthetic terrain: ceiling iff (splitmix64(seed*0x9E3779B97F4A7C15 + (t<<20) + y*w + x) >> 40) < density_q24 */
int tss_world_synthetic(int32_t w, int32_t h, uint64_t seed, uint64_t t, uint32_t density_q24, uint8_t* grid);

/* --------------------------------------------------------------- encoder (src/encoder.rs:435-667), host side */
/* Encoding::encode(&[PlatformDef], &WorldGrid) (encoder.rs:435).  Rejects a platform set without 1x1 with
 * TSS_E_INVALID (the reference unwraps, encoder.rs:564-566). */
int tss_encoding_create(const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, tss_encoding** out);
void tss_encoding_destroy(tss_encoding* enc);
/* sizes of the base instance: vars, clauses, literals, number of dims keys K (encoder.rs:121-130) */
int tss_encoding_sizes(const tss_encoding* enc, int32_t* n_vars, int32_t* n_clauses, int64_t* n_lits, int32_t* n_dims);
/* dims keys in variable order (deterministic replacement for the reference's HashMap order, encoder.rs:191-194) */
int tss_encoding_dims(const tss_encoding* enc, tss_dims* out_dims /* [K] */);
/* Encoding::vars() (encoder.rs:615): plat_var[tile*K + k], terr_var[tile*4 + layer]; 0 = absent */
int tss_encoding_var_maps(const tss_encoding* enc, int32_t* plat_var, int32_t* terr_var);
/* the base CNF in CSR form: lits[n_lits], offsets[n_clauses+1] */
int tss_encoding_cnf(const tss_encoding* enc, int32_t* lits, uint32_t* offsets);
/* Encoding::with_limits(&PlatformLimits) + SatInstance::into_cnf() (encoder.rs:619-667, crates/repl/src/main.rs:292-293).
 * card / weights are records (def_w, def_h, value); weight_limit is ignored unless has_weight_limit.
 * Two-call protocol: with lits == NULL only the sizes are returned. */
int tss_encoding_with_limits(const tss_encoding* enc, const int32_t* card, int32_t n_card, const int32_t* weights,
                             int32_t n_weights, int32_t has_weight_limit, int64_t weight_limit, int32_t* n_vars,
                             int32_t* n_clauses, int64_t* n_lits, int32_t* lits, uint32_t* offsets);
/* PlatformLayout::from_assignment (src/encoder/platform_layout.rs:26-52): largest platform per anchor.
 * returns the number of platforms (may exceed cap -> TSS_E_CAPACITY). */
int tss_layout_from_assignment(const tss_encoding* enc, const uint8_t* assignment, int32_t n_assignment,
                               tss_platform* out, int32_t cap, int32_t* n_out);
/* The inverse used to hand a GPU witness to the exact solver / CNF check: platform vars from the layout (every dims
 * key <= the platform's dims at its anchor, per the DAG implications encoder.rs:449-458), terrain-layer vars from
 * the support layers (T_l(p) = p within 3-l steps of a directly supported tile).  Runs the coverage kernel (a). */
int tss_layout_to_assignment(tss_engine* e, const tss_encoding* enc, const tss_platform* plats, int32_t n_plats,
                             uint8_t* assignment /* [n_vars_base + 1] */);
/* run_trivial_optimization (platform_layout.rs:151-172): drop platforms under no ceiling tile; returns new count */
int tss_layout_trivial_optimization(const uint8_t* grid, int32_t w, int32_t h, tss_platform* plats, int32_t n);
/* Host-side post-pass for layouts of 1x1 supports when the platform set holds larger platforms (what the engine applies to
 * its window-decomposed search on grids larger than 32x32): supports that fit under one footprint are merged into that
 * platform — validate() supports everything a platform's footprint covers plus three dilations, so its reach contains
 * theirs (platform_layout.rs:116-141) — footprints stay in bounds and pairwise disjoint (encoder.rs:546-609), then
 * platforms whose reach the others already cover are dropped.  A complete layout stays complete.  plats: n platforms in,
 * result out (capacity cap); returns the new count, TSS_E_CAPACITY if it does not fit (cannot happen for cap >= n). */
int tss_layout_merge_supports(const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, tss_platform* plats, int32_t n,
                              int32_t cap);
/* total_weight (platform_layout.rs:174-183); weights are records (def_w, def_h, weight) */
int64_t tss_layout_total_weight(const tss_platform* plats, int32_t n, const int32_t* weights, int32_t n_weights);
/* Platform::overlaps (src/platform.rs:86-97) */
int tss_platform_overlaps(const tss_platform* a, const tss_platform* b);

/* ------------------------------------------------------- kernel (a): coverage evaluator == PlatformLayout::validate */
/* validate() of ONE layout (platform_layout.rs:85-149), on the GPU.  out_unsupported: u8[w*h] mask of unsupported
 * terrain; out_flags[n]: bit0 overlapping, bit1 out of bounds.  Returns the number of unsupported tiles. */
int tss_validate(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_platform* plats, int32_t n,
                 uint8_t* out_unsupported, uint8_t* out_flags);
/* Batched validate of 1x1-only layouts given as u8 site masks [n][w*h] (non-zero = support) on one terrain. */
int tss_eval_sites(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const uint8_t* sites, int64_t n,
                   int32_t* out_uncovered, int32_t* out_count);
/* Same with bit-packed inputs: grid_rows[h*wpr], layouts[n][h*wpr] (wpr = ceil(w/32)).  Host buffers. */
int tss_eval_packed(tss_engine* e, const uint32_t* grid_rows, int32_t w, int32_t h, const uint32_t* layouts, int64_t n,
                    int32_t* out_uncovered, int32_t* out_count);
/* Device-resident variant (inputs/outputs already in HBM; async on the engine stream).  `layouts_dev` uses the
 * compact row format: for grids up to 32x32 the row stride is 1, 2 or 4 bytes for w <= 8, 16, 32 and a layout is
 * padded to a multiple of 4 bytes; larger grids use 4*wpr bytes per row.  out_dev: int32[n][2] =
 * (uncovered, count).  per_layout_terrain != 0: grid_dev holds n terrains (one per layout, same format). */
int tss_eval_compact_dev(tss_engine* e, const void* grid_dev, int32_t w, int32_t h, const void* layouts_dev, int64_t n,
                         int32_t per_layout_terrain, int32_t* out_dev);
size_t tss_compact_row_bytes(int32_t w, int32_t h);
size_t tss_compact_layout_bytes(int32_t w, int32_t h);
/* Batched validate of general platform layouts: layout i = plats[offsets[i] .. offsets[i+1]).  out[n][4] =
 * (unsupported tiles, platforms, overlapping platforms, out-of-bounds platforms). */
int tss_eval_platforms(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_platform* plats,
                       const uint32_t* offsets, int64_t n, int32_t* out);

/* -------------------------------------------- kernel (c): clause evaluation + unit propagation over the encoder's CNF */
/* Solve::add_cnf analogue (crates/repl/src/solver_runner.rs:12): uploads lits/offsets (CSR) once. */
int tss_cnf_upload(tss_engine* e, const int32_t* lits, const uint32_t* offsets, int32_t n_clauses, int32_t n_vars, tss_cnf** out);
void tss_cnf_destroy(tss_cnf* c);
/* Evaluates every clause under n assignments [n][n_vars+1] (0 F / 1 T / 2 DontCare; a DontCare literal satisfies
 * nothing).  out_n_falsified[n], out_first_falsified[n] (clause index or -1). */
int tss_cnf_check(tss_engine* e, const tss_cnf* c, const uint8_t* assignments, int64_t n, int32_t* out_n_falsified,
                  int32_t* out_first_falsified);
/* Unit propagation to fixpoint from n partial assignments (in/out).  out_conflict[n] = index of a clause falsified
 * at the fixpoint, or -1.  out_rounds (optional) = propagation rounds executed. */
int tss_cnf_propagate(tss_engine* e, const tss_cnf* c, uint8_t* assignments, int64_t n, int32_t* out_conflict, int32_t* out_rounds);

/* --------------------------------------------------- kernel (b): batched stochastic local search (upper bounds) */
typedef struct tss_search_params {
    uint64_t seed;         /* counter-based RNG key; results are reproducible for (seed, n_chains, chain_offset) */
    int32_t n_chains;      /* independent layouts searched in parallel (one per warp); 0 = fill the device */
    int32_t chain_offset;  /* global index of this engine's first chain (rank * n_chains in a multi-GPU portfolio) */
    int32_t noise_pct;     /* probability (percent) of a random instead of greedy add move; < 0 = default */
    int32_t kernel;        /* TSS_KERNEL_*: which of the equivalent SLS kernels runs (same step rule, same trajectories); 0 = auto.
                            * TSS_KERNEL_WINDOW_PLACEMENTS selects a different search on grids larger than 32x32 (see there) */
} tss_search_params;

/* SLS kernel variants for grids up to 32x32 with 1x1 supports.  All four execute the published step rule bit for bit
 * (tests replay each against the CPU model); they differ in how a chain is mapped to the hardware. */
#define TSS_KERNEL_AUTO 0
#define TSS_KERNEL_WARP 1      /* one chain per warp, any grid up to 32x32 */
#define TSS_KERNEL_HALF_WARP 2 /* two chains per warp, grids of at most 16 rows */
#define TSS_KERNEL_THREAD 3    /* one chain per thread, grids of at most 16 rows x 26 columns */
#define TSS_KERNEL_PAIR 4      /* one chain per thread, two grid rows per word, grids of at most 16x16 */
/* The window-decomposed placement search: grids wider or taller than 32 with a platform set beyond {1x1} (at most 16 dims
 * keys, each at most 6x6), on one rank.  The global layout starts as the greedy placement cover and only improves: each
 * tss_search_run phase (MAX_EPOCH_STEPS steps at most, longer runs are several phases) runs the placement search on 32x32
 * windows with the platforms near window borders frozen, and keeps each window's best (its target_count is not used:
 * the windows search without a target).  n_chains = chains per window
 * (rounded up to a multiple of 4; 0 = 8..16).  Otherwise (AUTO) those grids run the 1x1 window decomposition with a
 * host post-pass.  tss_search_create answers TSS_E_UNSUPPORTED where it does not apply. */
#define TSS_KERNEL_WINDOW_PLACEMENTS 5

/* Creates a portfolio on one terrain.  defs must contain 1x1 (encoder.rs:564-566). */
int tss_search_create(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                      const tss_search_params* params, tss_search** out);
void tss_search_destroy(tss_search* s);
/* Runs `steps` SLS steps per chain (one epoch, one kernel launch + a best-reduce), asynchronously on the engine
 * stream.  Chains stop early once a layout with <= target_count platforms is found (target < 0: never). */
int tss_search_run(tss_search* s, int64_t steps, int32_t target_count);
/* Best validated platform count found so far (synchronises the stream); -1 if no complete layout yet. */
int tss_search_best_count(tss_search* s, int32_t* count);
/* Shares an externally known bound (e.g. the all-reduce-min over GPUs): chains only look for layouts with fewer
 * than `count` platforms from now on. */
int tss_search_set_bound(tss_search* s, int32_t count);
/* The bound the next epoch searches below: min(best counts of this search, bounds set from outside, and — with a
 * communicator on the engine — the best counts of every rank's search); -1 if none yet.  (synchronises the stream) */
int tss_search_global_best(tss_search* s, int32_t* count);
/* Best layout (re-validated by kernel (a) before it is returned).  TSS_KERNEL_WINDOW_PLACEMENTS: the global layout, before
 * the first run the start layout (the greedy placement cover). */
int tss_search_best_layout(tss_search* s, tss_platform* out, int32_t cap, int32_t* n_out);
int tss_search_n_chains(const tss_search* s);
/* Which TSS_KERNEL_* variant advances this portfolio (what TSS_KERNEL_AUTO resolved to); 0 for the 1x1 window decomposition
 * and the placement search, which have a single kernel each; TSS_KERNEL_WINDOW_PLACEMENTS for that search. */
int tss_search_kernel(const tss_search* s);
/* Introspection for the parity tests (the CPU model in oracle/sls_model.cpp replays the same trajectories): per-chain
 * state after the last epoch.  S / best_S: support rows u32[n_chains][32]; any pointer may be NULL. */
int tss_search_read_chains(tss_search* s, uint32_t* S, uint32_t* best_S, int32_t* k, int32_t* best, uint32_t* step, uint64_t* scored);
/* Same for the placement search (platform sets beyond {1x1}): items / best_items u16[n_chains][1024], a placement is
 * key << 10 | y << 5 | x with key indexing key_dims (effective (w, h) per dims key: defs order, unflipped then flipped,
 * src/encoder.rs:121-130; room for 16 entries); best = best objective value (platform count or total weight). */
int tss_search_read_placements(tss_search* s, uint16_t* items, int32_t* k, uint16_t* best_items, int32_t* best_k, int32_t* best, uint32_t* step,
                               tss_dims* key_dims, int32_t* n_keys);
/* Warm start: replaces every chain's CURRENT layout by the given support rows (u32[n_chains][32], row r of chain c at
 * S[c*32 + r], bit x = support at (x, r); bits outside the grid are an error).  Best layouts, bounds and step counters are
 * kept; the next epoch continues from these layouts (the drivers' natural seed is the layout of the previous solve,
 * crates/repl/src/main.rs:331-346).  Only for the 1x1 search on grids up to 32x32. */
int tss_search_write_chains(tss_search* s, const uint32_t* S);

/* GUI objective (crates/gui/src/app.rs:53-62,235-245): minimise PlatformLayout::total_weight (platform_layout.rs:174-183)
 * instead of the platform count.  weights = records (def_w, def_h, weight) keyed by canonical def dims, exactly the
 * PlatformLimits.weights map; call before the first tss_search_run.  Afterwards tss_search_best_count /
 * tss_search_set_bound speak total weight.  Needs a platform set beyond {1x1} on a grid up to 32x32, or a search created
 * with TSS_KERNEL_WINDOW_PLACEMENTS. */
int tss_search_set_weights(tss_search* s, const int32_t* weights, int32_t n_weights);

/* Values of the SLS specification's hash / tie-break functions (csrc/sls_spec.hpp) at fixed probe points, so the
 * parity tests can assert that the CPU model (which re-declares them) follows the same published rule.  out[9]. */
void tss_sls_spec_probe(uint32_t* out);

/* The solve-with-bound entry point (the SAT side of crates/repl/src/main.rs:292-329 / crates/gui/src/solver_backend.rs:69-97):
 * find a layout with at most `card_limit` platforms (card_limit < 0: unbounded, any complete layout) within
 * `budget_ms` and/or `max_steps` SLS steps per chain, returning the best layout found.  With neither budget given
 * the call behaves like ONE SAT call: it returns the first layout within the bound and gives up after 2^18 steps
 * per chain (the engine cannot prove UNSAT, so "nothing found" must terminate).  A NEGATIVE `max_steps` (with no
 * `budget_ms`) is the same SAT-like call with the give-up point moved to -max_steps steps per chain: the bound-tightening
 * loop uses it to hand an instance it cannot answer quickly to the exact solver after a bounded, small effort.
 * Returns TSS_SAT with the layout, TSS_UNKNOWN if none was found (never TSS_UNSAT). */
int tss_solve_upper_bound(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                          int32_t card_limit, uint64_t seed, int32_t budget_ms, int64_t max_steps, tss_platform* out,
                          int32_t cap, int32_t* n_out);
/* The GUI's weight-minimising solve (crates/gui/src/solver_backend.rs:69-97 with PlatformLimits.weight_limit): a layout of
 * total weight <= weight_limit (< 0: unbounded), best found within the budget; *out_weight = its total weight. */
int tss_solve_min_weight(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs,
                         const int32_t* weights, int32_t n_weights, int64_t weight_limit, uint64_t seed, int32_t budget_ms,
                         int64_t max_steps, tss_platform* out, int32_t cap, int32_t* n_out, int64_t* out_weight);
/* LOWER bound on the platform count of any complete layout (not in the reference; SURVEY.md §8(f)): a packing of ceiling
 * tiles no two of which a single platform of the set can support — validate()'s rule, src/encoder/platform_layout.rs:104-141,
 * applied to every in-bounds placement of every dims key — so every layout needs one platform per packed tile.  Randomized
 * greedy restarts on the GPU (`restarts` <= 0: 16 per SM), the winning packing is re-verified on the device before it is
 * returned.  out_xy[2*i], out_xy[2*i+1] = packed tile i (capacity `cap` tiles); *n_out = the bound.  When
 * tss_solve_upper_bound reaches this count the bound-tightening loop (crates/repl/src/main.rs:280-366) is finished without
 * the exact solver.  Any platform set on grids up to 32x32; larger grids (up to 256x256) with 1x1 supports, by parallel rounds on
 * the whole bitboard (`restarts` <= 0: one per SM); TSS_E_UNSUPPORTED otherwise. */
int tss_lower_bound(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, uint64_t seed,
                    int32_t restarts, int32_t* out_xy, int32_t cap, int32_t* n_out);
/* The FRACTIONAL version of that bound (csrc/lp.cu): weights y_t >= 0 on the ceiling tiles such that no in-bounds placement's
 * reach holds more than the placement COSTS; every layout then costs at least sum(y).  Cost = 1 per platform (n_weights = 0: a
 * bound on the platform count, what the REPL minimises, main.rs:346) or, with `weights` (records (def_w, def_h, weight), the
 * PlatformLimits.weights map), what PlatformLayout::total_weight charges the platform (platform_layout.rs:174-183): a bound on
 * the GUI's objective (crates/gui/src/app.rs:235-245).  The LP is solved on the GPU (dense primal simplex, at most `max_pivots`
 * pivots, <= 0: default; `target` > 0: stop as soon as the bound reaches `target` — every simplex iterate is feasible, so stopping
 * early only weakens the bound — which is all the bound-tightening loop asks: "is there no layout within limit = target - 1?";
 * <= 0: to optimality) and the result is CERTIFIED in integer arithmetic: out_weights[w*h] (optional) = floor(y * scale) per
 * tile, *out_total = their sum, *out_max_load = the largest sum over the reach of any placement, recomputed from the reach
 * bitboards, and *out_bound = min over placements of ceil(total * cost / load) (= ceil(total / max_load) with unit costs) —
 * valid whatever the floating point solve did.  It dominates tss_lower_bound up to rounding (README terrain, 1x1 supports:
 * 12 -> 14 = the optimum).  out_info[3] (optional) = pivots, 1 if the simplex reached optimality, constraints.  Grids up to 32x32
 * take that simplex.  Grids larger than 32x32, up to 256x256, take a first-order method instead (csrc/lp_big.cu: optimistic
 * multiplicative weights on the zero-sum game of the LP, no tableau) with the same certificate over every in-bounds placement:
 * any platform set of at most 16 dims keys, each at most 6x6 (what the window placement search takes, or 1x1 alone), count or
 * weights; anything else returns TSS_E_UNSUPPORTED.  There `max_pivots` caps the ITERATIONS (<= 0: 3 000), `target` > 0 stops
 * as soon as the integer-certified bound reaches `target` (checked every 250 iterations), tiles in the reach of a platform that
 * costs nothing are fixed at 0, and out_info = iterations, 0 (the method never proves optimality), constraints (placements whose
 * reach holds ceiling and that cost something).  Two calls on the same device give the same weights. */
int tss_lower_bound_lp(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, const int32_t* weights,
                       int32_t n_weights, int32_t max_pivots, int64_t target, int32_t* out_weights, int64_t* out_total, int64_t* out_max_load,
                       int64_t* out_bound, int32_t* out_info);
/* Terrain batch (SURVEY.md C5): n independent terrains [n][w*h] (grids up to 32x32), 1x1 supports; `steps` SLS steps
 * per chain, `chains_per_terrain` independent chains per terrain sharing their bound every 1024 steps (0 = one CTA
 * = 4 chains, 8 for grids of <= 16 rows; otherwise rounded up to a multiple of that).  out_counts[n] = best count per
 * terrain; out_layouts (optional) = packed support rows [n][h*wpr]. */
int tss_solve_batch(tss_engine* e, const uint8_t* grids, int32_t w, int32_t h, int64_t n, uint64_t seed, int64_t steps,
                    int32_t chains_per_terrain, int32_t* out_counts, uint32_t* out_layouts);

/* -------------------------------------------------- instance bridge: from a bare CNF back to terrain, platform set and limits */
/* The drivers hand their solver nothing but the clauses (`run_solver(GlucoseSimp::default(), cnf)`,
 * crates/repl/src/solver_runner.rs:8-20; `SolverBackend::start`, crates/gui/src/solver_backend.rs:69-97), while the GPU
 * search works on the terrain.  The lib crate's side of this boundary owns `Encoding::encode` / `with_limits`
 * (src/encoder.rs:435,619): every tss_encoding_with_limits call that returns clauses records (encoding, limits, CNF) in a
 * small process-wide registry (the last 8 instances), and a solver finds its instance again from the clauses it was given —
 * so the drivers need no extra call and build unchanged. */
typedef struct tss_instance_info {
    int32_t w, h, n_defs;            /* terrain size and platform set of the encoding */
    int32_t card_limit_1x1;          /* n of "at most n platforms" (PlatformLimits.card_limits[1x1], main.rs:346), -1 if none */
    int32_t n_other_card_limits;     /* card limits on other platform types (per-type limits: tss_solve_instance steers the search by
                                        them on grids up to 32x32 when the handle came from tss_instance_find) */
    int32_t has_weight_limit;
    int64_t weight_limit;            /* PlatformLimits.weight_limit (crates/gui/src/app.rs:235-245) */
    int32_t n_weights;
    int32_t exact;                   /* 1: the whole CNF equals the recorded one; 0: only its base clauses match (limits of the latest record) */
} tss_instance_info;
/* Looks up the CNF a solver received in add_cnf.  TSS_SAT: found — *enc_out is a NEW handle (tss_encoding_destroy), *info the
 * limits, weights (optional, capacity weights_cap records of (def_w, def_h, weight)) the PlatformLimits.weights map.
 * TSS_UNKNOWN: not one of the recorded instances (solve on the exact solver alone). */
int tss_instance_find(const int32_t* lits, const uint32_t* offsets, int32_t n_clauses, int32_t n_vars, tss_encoding** enc_out,
                      tss_instance_info* info, int32_t* weights, int32_t weights_cap);
/* terrain (u8[w*h]) and platform defs of an encoding */
int tss_encoding_terrain(const tss_encoding* enc, uint8_t* grid, size_t cap, int32_t* w, int32_t* h);
int tss_encoding_defs(const tss_encoding* enc, tss_dims* defs, int32_t cap, int32_t* n);
int tss_cnf_num_vars(const tss_cnf* c);
/* GPU layout -> full model of an uploaded CNF, verified: platform variables from the layout, terrain-layer variables from
 * validate()'s support layers (tss_layout_to_assignment — unit propagation alone cannot decide those), the variables the
 * limits added (totalizer / PB auxiliaries) by unit propagation, then every clause checked (kernel (c)).  assignment:
 * u8[n_vars(c) + 1].  TSS_SAT: it is a model; TSS_UNKNOWN: it is not (e.g. the layout exceeds a limit). */
int tss_witness_for_cnf(tss_engine* e, const tss_cnf* c, const tss_encoding* enc, const tss_platform* plats, int32_t n, uint8_t* assignment);
/* The completion step on its own, for ONE partial assignment u8[n_vars + 1] (0 / 1 / 2 = False / True / unassigned), in place:
 * unit propagation to the fixpoint, open variables False, every clause checked.  One fused launch when the variables fit a
 * CTA's shared memory (csrc/cnf.cu cnf_complete_kernel; in-place propagation — same fixpoint and conflict verdict as the
 * synchronous rounds of tss_cnf_propagate), the batch kernels otherwise.  *out_conflict = a clause left without a true or open
 * literal by the propagation, or -1 (then the assignment is complete and *out_n_falsified counts the clauses it falsifies);
 * after a conflict the assignment holds the propagation's state and *out_n_falsified is 0. */
int tss_cnf_complete(tss_engine* e, const tss_cnf* c, uint8_t* assignment, int32_t* out_conflict, int32_t* out_n_falsified);
/* Solve::solve as the GPU answers it: ONE SAT-like search within the instance's limit (platform count, or total weight when
 * the instance carries a weight limit) that gives up after `give_up_steps` SLS steps per chain (<= 0: the engine default),
 * then tss_witness_for_cnf.  TSS_SAT with a verified model in `assignment`; TSS_UNSAT when the instance's only limit (platform
 * count, or total weight) lies below a certified lower bound (the integral packing, checked before searching; the fractional
 * LP, computed once per instance after a search came back empty — a first search on an eighth of the give-up budget while that
 * bound is still to be computed, the whole budget only if the bound does not settle the question; grids up to 32x32) — the
 * unmodified bound-tightening loops
 * (crates/repl/src/main.rs:331-334, crates/gui/src/app.rs:212-249) then end proven optimal without their exact solver;
 * TSS_UNKNOWN otherwise: the caller asks its exact solver, which stays the only prover of UNSAT by search.
 * tss_engine_certified_unsat switches the bound-based UNSAT answers off (0) or on (non-zero, the default). */
int tss_engine_certified_unsat(tss_engine* e, int enabled);
int tss_solve_instance(tss_engine* e, const tss_cnf* c, const tss_encoding* enc, const tss_instance_info* info, const int32_t* weights,
                       uint64_t seed, int64_t give_up_steps, uint8_t* assignment);

/* ------------------------------------------------------------------------------------------ measured peaks */
/* Runs the integer-issue (LOP3 / POPC / SHFL) and shared-memory micro-benchmarks SURVEY.md §8(d) asks for.
 * out[0] LOP3 Gop/s (thread-ops), out[1] POPC Gop/s, out[2] SHFL Gop/s, out[3] shared-memory GB/s, out[4] SM clock MHz
 * observed (cycles / elapsed). */
int tss_measure_peaks(tss_engine* e, double* out, int32_t n_out);

/* ------------------------------------------------------------------------------------------ per-type platform limits */
/* The REPL's `solve -l k:v[,k:v]` (PlatformLimits.card_limits beyond 1x1, crates/repl/src/main.rs:85-101), as
 * Encoding::with_limits lowers a limit on type d: one literal per anchor, set by a platform of any dims key q that contains d or
 * its transpose (d's CLASS: the keys q with dims_le(k, q) for a key k in {d, d^T}).  A platform counts at most once towards a
 * class.  A record whose d and d^T are both absent from the platform set constrains nothing, nor does a limit of 1024 or more:
 * such records are VACUOUS and ignored.  Records are (def_w, def_h, limit), the `card` argument of tss_encoding_with_limits.
 *
 * The classes themselves, host only: key_mask[k] (capacity 16) = classes of dims key k in the engine's key order (defs order,
 * unflipped then flipped, duplicates dropped; tss_search_read_placements reports it), bit j = class j; class_limit[j]
 * (capacity 16).  1x1 records (the platform count) and vacuous records make no class; records with the same class merge into
 * the smaller limit. */
int tss_card_limit_classes(const tss_dims* defs, int32_t n_defs, const int32_t* card, int32_t n_card, int32_t* key_mask, int32_t* class_limit,
                           int32_t* n_keys, int32_t* n_classes);
/* Steers a placement search by per-type limits: an addition that would take a class beyond its limit is no candidate, so every
 * current and best layout of every chain keeps every limit (a limit of 0 blocks its class from the start).  Call before the
 * first tss_search_run.  TSS_E_INVALID for a 1x1 record (the platform count is the search's bound: tss_search_set_bound), a
 * negative limit, or after the first run; vacuous records are ignored (on a {1x1}-only set every record is); TSS_E_UNSUPPORTED
 * for a record that is not vacuous on a search other than the placement search on a grid up to 32x32 (the window searches:
 * their windows pick winners independently, which could jointly exceed a limit). */
int tss_search_set_card_limits(tss_search* s, const int32_t* card, int32_t n_card);
/* The PlatformLimits-shaped one-shot solve: card = records (def_w, def_h, limit) including the platform count (1x1); with
 * weights (n_weights > 0) the objective is the total weight, bounded by weight_limit (< 0: unbounded), and a 1x1 record is
 * TSS_E_UNSUPPORTED (one objective per search).  Defs in a class with limit 0 are dropped from the set first (as --platforms
 * would), positive limits steer the placement search (tss_search_set_card_limits; grids up to 32x32).  Budgets and the return
 * contract are tss_solve_upper_bound's: TSS_SAT with the layout and *out_objective (optional) = its count or weight, TSS_UNKNOWN
 * if none was found, never TSS_UNSAT. */
int tss_solve_with_limits(tss_engine* e, const uint8_t* grid, int32_t w, int32_t h, const tss_dims* defs, int32_t n_defs, const int32_t* card,
                          int32_t n_card, const int32_t* weights, int32_t n_weights, int64_t weight_limit, uint64_t seed, int32_t budget_ms,
                          int64_t max_steps, tss_platform* out, int32_t cap, int32_t* n_out, int64_t* out_objective);

#ifdef __cplusplus
}
#endif
#endif /* TSS_H */
