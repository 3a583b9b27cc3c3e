//! Raw bindings to `include/tss.h` (ABI version 103).  Every entry point cites, in the header, the reference
//! interface it stands behind; this file only mirrors types and signatures.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const TSS_VERSION: c_int = 103;
pub const TSS_OK: c_int = 0;
pub const TSS_SAT: c_int = 10; // IPASIR / rustsat SolverResult::Sat
pub const TSS_UNSAT: c_int = 20; // only from tss_solve_instance, when the limit lies below a certified lower bound
pub const TSS_UNKNOWN: c_int = 0; // SolverResult::Interrupted
pub const TSS_KERNEL_AUTO: i32 = 0;
pub const TSS_KERNEL_WARP: i32 = 1; // one chain per warp, any grid up to 32x32
pub const TSS_KERNEL_HALF_WARP: i32 = 2; // two chains per warp, grids of at most 16 rows
pub const TSS_KERNEL_THREAD: i32 = 3; // one chain per thread, grids of at most 16 rows x 26 columns
pub const TSS_KERNEL_PAIR: i32 = 4; // one chain per thread, two grid rows per word, grids of at most 16x16
pub const TSS_KERNEL_WINDOW_PLACEMENTS: i32 = 5; // window-decomposed placement search, grids larger than 32x32

#[repr(C)]
#[derive(Copy, Clone, Default, Debug, PartialEq, Eq)]
pub struct tss_platform {
    pub x: i32,
    pub y: i32,
    pub def_w: i32, // canonical PlatformDef dims, w <= h (src/platform.rs:11-32)
    pub def_h: i32,
    pub rotated: i32, // effective dims = (def_h, def_w) when set (src/platform.rs:111-113)
}

#[repr(C)]
#[derive(Copy, Clone, Default, Debug)]
pub struct tss_dims {
    pub w: i32,
    pub h: i32,
}

#[repr(C)]
#[derive(Copy, Clone, Default, Debug)]
pub struct tss_stats {
    pub layouts_evaluated: u64,
    pub candidates_scored: u64,
    pub sls_steps: u64,
    pub clauses_checked: u64,
    pub kernel_launches: u64,
    pub n_solves: u64,
    pub device_ms: f64,
    pub best_count: i32,
    pub interrupted: i32,
    pub last_solve_steps: i64,
    pub sls_flips: u64,
}

#[repr(C)]
#[derive(Copy, Clone, Default, Debug)]
pub struct tss_instance_info {
    pub w: i32,
    pub h: i32,
    pub n_defs: i32,
    pub card_limit_1x1: i32,      // n of "at most n platforms" (main.rs:346), -1 if none
    pub n_other_card_limits: i32,
    pub has_weight_limit: i32,
    pub weight_limit: i64,
    pub n_weights: i32,
    pub exact: i32,
}

#[repr(C)]
#[derive(Copy, Clone, Default, Debug)]
pub struct tss_search_params {
    pub seed: u64,
    pub n_chains: i32,
    pub chain_offset: i32,
    pub noise_pct: i32,
    pub kernel: i32,
}

#[repr(C)]
pub struct tss_engine {
    _p: [u8; 0],
}
#[repr(C)]
pub struct tss_encoding {
    _p: [u8; 0],
}
#[repr(C)]
pub struct tss_cnf {
    _p: [u8; 0],
}
#[repr(C)]
pub struct tss_search {
    _p: [u8; 0],
}

unsafe extern "C" {
    pub fn tss_version() -> c_int;
    pub fn tss_engine_create(device: c_int, out: *mut *mut tss_engine) -> c_int;
    pub fn tss_engine_destroy(e: *mut tss_engine);
    pub fn tss_last_error(e: *const tss_engine) -> *const c_char;
    pub fn tss_interrupt(e: *mut tss_engine);
    pub fn tss_clear_interrupt(e: *mut tss_engine);
    pub fn tss_get_stats(e: *const tss_engine, out: *mut tss_stats) -> c_int;

    // the SAT side of crates/repl/src/main.rs:292-329 / crates/gui/src/solver_backend.rs:69-97
    pub fn tss_solve_upper_bound(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, card_limit: i32, seed: u64,
        budget_ms: i32, max_steps: i64, out: *mut tss_platform, cap: i32, n_out: *mut i32,
    ) -> c_int;
    // the GUI's weight objective (crates/gui/src/app.rs:235-245)
    pub fn tss_solve_min_weight(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, weights: *const i32, n_weights: i32,
        weight_limit: i64, seed: u64, budget_ms: i32, max_steps: i64, out: *mut tss_platform, cap: i32, n_out: *mut i32,
        out_weight: *mut i64,
    ) -> c_int;

    // PlatformLayout::validate (src/encoder/platform_layout.rs:85-149) on the GPU
    pub fn tss_validate(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, plats: *const tss_platform, n: i32, out_unsupported: *mut u8,
        out_flags: *mut u8,
    ) -> c_int;

    // the CNF the exact solver receives: upload once, verify GPU witnesses against it (kernel (c))
    pub fn tss_cnf_upload(
        e: *mut tss_engine, lits: *const i32, offsets: *const u32, n_clauses: i32, n_vars: i32, out: *mut *mut tss_cnf,
    ) -> c_int;
    pub fn tss_cnf_destroy(c: *mut tss_cnf);
    pub fn tss_cnf_check(
        e: *mut tss_engine, c: *const tss_cnf, assignments: *const u8, n: i64, out_n_falsified: *mut i32,
        out_first_falsified: *mut i32,
    ) -> c_int;
    pub fn tss_cnf_propagate(
        e: *mut tss_engine, c: *const tss_cnf, assignments: *mut u8, n: i64, out_conflict: *mut i32, out_rounds: *mut i32,
    ) -> c_int;

    // the lib crate's side: Encoding::encode / with_limits (src/encoder.rs:435,619); with_limits records the instance
    pub fn tss_encoding_create(grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, out: *mut *mut tss_encoding) -> c_int;
    pub fn tss_encoding_destroy(enc: *mut tss_encoding);
    pub fn tss_encoding_sizes(enc: *const tss_encoding, n_vars: *mut i32, n_clauses: *mut i32, n_lits: *mut i64, n_dims: *mut i32) -> c_int;
    pub fn tss_encoding_var_maps(enc: *const tss_encoding, plat_var: *mut i32, terr_var: *mut i32) -> c_int;
    pub fn tss_encoding_with_limits(
        enc: *const tss_encoding, card: *const i32, n_card: i32, weights: *const i32, n_weights: i32, has_weight_limit: i32, weight_limit: i64,
        n_vars: *mut i32, n_clauses: *mut i32, n_lits: *mut i64, lits: *mut i32, offsets: *mut u32,
    ) -> c_int;
    pub fn tss_layout_from_assignment(enc: *const tss_encoding, assignment: *const u8, n: i32, out: *mut tss_platform, cap: i32, n_out: *mut i32) -> c_int;
    pub fn tss_layout_to_assignment(e: *mut tss_engine, enc: *const tss_encoding, plats: *const tss_platform, n: i32, assignment: *mut u8) -> c_int;

    // the solver's side: from the clauses back to the instance, then Solve::solve on the GPU (csrc/instance.cpp)
    pub fn tss_instance_find(
        lits: *const i32, offsets: *const u32, n_clauses: i32, n_vars: i32, enc_out: *mut *mut tss_encoding, info: *mut tss_instance_info,
        weights: *mut i32, weights_cap: i32,
    ) -> c_int;
    pub fn tss_witness_for_cnf(e: *mut tss_engine, c: *const tss_cnf, enc: *const tss_encoding, plats: *const tss_platform, n: i32, assignment: *mut u8) -> c_int;
    pub fn tss_cnf_complete(e: *mut tss_engine, c: *const tss_cnf, assignment: *mut u8, out_conflict: *mut i32, out_n_falsified: *mut i32) -> c_int;
    pub fn tss_engine_certified_unsat(e: *mut tss_engine, enabled: c_int) -> c_int;
    pub fn tss_engine_limit_bounds(e: *mut tss_engine, enabled: c_int) -> c_int;
    pub fn tss_engine_window_limits(e: *mut tss_engine, enabled: c_int) -> c_int;
    pub fn tss_solve_instance(
        e: *mut tss_engine, c: *const tss_cnf, enc: *const tss_encoding, info: *const tss_instance_info, weights: *const i32, seed: u64,
        give_up_steps: i64, assignment: *mut u8,
    ) -> c_int;
    // packing lower bound: when the count meets it the loop needs no proof
    pub fn tss_lower_bound(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, seed: u64, restarts: i32, out_xy: *mut i32, cap: i32,
        n_out: *mut i32,
    ) -> c_int;

    pub fn tss_lower_bound_lp(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, weights: *const i32, n_weights: i32, max_pivots: i32,
        target: i64, out_weights: *mut i32, out_total: *mut i64, out_max_load: *mut i64, out_bound: *mut i64, out_info: *mut i32,
    ) -> c_int;
    pub fn tss_lower_bound_lp_limits(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, card: *const i32, n_card: i32, weights: *const i32,
        n_weights: i32, max_pivots: i32, target: i64, out_weights: *mut i32, out_class_weights: *mut i32, out_total: *mut i64, out_max_load: *mut i64,
        out_bound: *mut i64, out_info: *mut i32,
    ) -> c_int;
    pub fn tss_encoding_terrain(enc: *const tss_encoding, grid: *mut u8, cap: usize, w: *mut i32, h: *mut i32) -> c_int;
    pub fn tss_encoding_defs(enc: *const tss_encoding, defs: *mut tss_dims, cap: i32, n: *mut i32) -> c_int;
    pub fn tss_cnf_num_vars(c: *const tss_cnf) -> c_int;
    pub fn tss_debug_smem_violations() -> c_int;

    // a persistent portfolio instead of one-shot calls
    pub fn tss_search_create(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, params: *const tss_search_params,
        out: *mut *mut tss_search,
    ) -> c_int;
    pub fn tss_search_destroy(s: *mut tss_search);
    pub fn tss_search_run(s: *mut tss_search, steps: i64, target_count: i32) -> c_int;
    pub fn tss_search_kernel(s: *const tss_search) -> c_int;
    pub fn tss_search_best_count(s: *mut tss_search, count: *mut i32) -> c_int;
    pub fn tss_search_set_bound(s: *mut tss_search, count: i32) -> c_int;
    pub fn tss_search_write_chains(s: *mut tss_search, rows: *const u32) -> c_int;
    pub fn tss_search_best_layout(s: *mut tss_search, out: *mut tss_platform, cap: i32, n_out: *mut i32) -> c_int;

    // multi-GPU portfolio: the host only ships the 128-byte NCCL id
    pub fn tss_comm_unique_id(e: *mut tss_engine, out128: *mut u8) -> c_int;
    pub fn tss_comm_init(e: *mut tss_engine, id128: *const u8, rank: i32, world: i32) -> c_int;

    // ---- the rest of include/tss.h (not used by the `tss` shim; here so that the whole ABI is declared in one place)
    pub fn tss_engine_set_stream(e: *mut tss_engine, cuda_stream: *mut c_void) -> c_int;
    pub fn tss_device_info(e: *const tss_engine, name: *mut c_char, cap: c_int, sm_count: *mut c_int, clock_khz: *mut c_int) -> c_int;
    pub fn tss_comm_world(e: *const tss_engine) -> c_int;
    pub fn tss_world_parse_toml(text: *const c_char, grid: *mut u8, cap: usize, w: *mut i32, h: *mut i32, ragged: *mut i32, err: *mut c_char, err_cap: usize) -> c_int;
    pub fn tss_world_to_toml(grid: *const u8, w: i32, h: i32, out: *mut c_char, cap: usize) -> c_int;
    pub fn tss_world_synthetic(w: i32, h: i32, seed: u64, t: u64, density_q24: u32, grid: *mut u8) -> c_int;
    pub fn tss_encoding_dims(enc: *const tss_encoding, out_dims: *mut tss_dims) -> c_int;
    pub fn tss_encoding_cnf(enc: *const tss_encoding, lits: *mut i32, offsets: *mut u32) -> c_int;
    pub fn tss_layout_trivial_optimization(grid: *const u8, w: i32, h: i32, plats: *mut tss_platform, n: i32) -> c_int;
    pub fn tss_layout_merge_supports(grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, plats: *mut tss_platform, n: i32, cap: i32) -> c_int;
    pub fn tss_layout_total_weight(plats: *const tss_platform, n: i32, weights: *const i32, n_weights: i32) -> i64;
    pub fn tss_platform_overlaps(a: *const tss_platform, b: *const tss_platform) -> c_int;
    pub fn tss_eval_sites(e: *mut tss_engine, grid: *const u8, w: i32, h: i32, sites: *const u8, n: i64, out_uncovered: *mut i32, out_count: *mut i32) -> c_int;
    pub fn tss_eval_packed(e: *mut tss_engine, grid_rows: *const u32, w: i32, h: i32, layouts: *const u32, n: i64, out_uncovered: *mut i32, out_count: *mut i32) -> c_int;
    pub fn tss_eval_compact_dev(e: *mut tss_engine, grid_dev: *const c_void, w: i32, h: i32, layouts_dev: *const c_void, n: i64, per_layout_terrain: i32, out_dev: *mut i32) -> c_int;
    pub fn tss_compact_row_bytes(w: i32, h: i32) -> usize;
    pub fn tss_compact_layout_bytes(w: i32, h: i32) -> usize;
    pub fn tss_eval_platforms(e: *mut tss_engine, grid: *const u8, w: i32, h: i32, plats: *const tss_platform, offsets: *const u32, n: i64, out: *mut i32) -> c_int;
    pub fn tss_search_global_best(s: *mut tss_search, count: *mut i32) -> c_int;
    pub fn tss_search_n_chains(s: *const tss_search) -> c_int;
    pub fn tss_search_read_chains(s: *mut tss_search, S: *mut u32, best_S: *mut u32, k: *mut i32, best: *mut i32, step: *mut u32, scored: *mut u64) -> c_int;
    pub fn tss_search_read_placements(
        s: *mut tss_search, items: *mut u16, k: *mut i32, best_items: *mut u16, best_k: *mut i32, best: *mut i32, step: *mut u32, key_dims: *mut tss_dims,
        n_keys: *mut i32,
    ) -> c_int;
    pub fn tss_search_set_weights(s: *mut tss_search, weights: *const i32, n_weights: i32) -> c_int;
    pub fn tss_search_set_card_limits(s: *mut tss_search, card: *const i32, n_card: i32) -> c_int;
    pub fn tss_search_create_with_limits(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, card: *const i32, n_card: i32,
        params: *const tss_search_params, out: *mut *mut tss_search,
    ) -> c_int;
    pub fn tss_card_limit_classes(
        defs: *const tss_dims, n_defs: i32, card: *const i32, n_card: i32, key_mask: *mut i32, class_limit: *mut i32, n_keys: *mut i32,
        n_classes: *mut i32,
    ) -> c_int;
    pub fn tss_solve_with_limits(
        e: *mut tss_engine, grid: *const u8, w: i32, h: i32, defs: *const tss_dims, n_defs: i32, card: *const i32, n_card: i32,
        weights: *const i32, n_weights: i32, weight_limit: i64, seed: u64, budget_ms: i32, max_steps: i64, out: *mut tss_platform, cap: i32,
        n_out: *mut i32, out_objective: *mut i64,
    ) -> c_int;
    pub fn tss_sls_spec_probe(out: *mut u32);
    pub fn tss_solve_batch(
        e: *mut tss_engine, grids: *const u8, w: i32, h: i32, n: i64, seed: u64, steps: i64, chains_per_terrain: i32, out_counts: *mut i32,
        out_layouts: *mut u32,
    ) -> c_int;
    pub fn tss_measure_peaks(e: *mut tss_engine, out: *mut f64, n_out: i32) -> c_int;
}
