// The solver side of the drop-in boundary (include/tss.h "instance bridge"): what a `Solve + Interrupt` implementation needs
// to answer `solve()` from the GPU when all it was given is a CNF (crates/repl/src/solver_runner.rs:8-20,
// crates/gui/src/solver_backend.rs:69-97).  Host C++ only; every GPU step goes through the public C ABI, so this file is
// also the reference for the call sequence of the Rust shim (rust/tss/src/lib.rs) and of tools/tss_repl.cpp.
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <mutex>

#include "encoding_handle.hpp"
#include "engine.hpp"

using namespace tss;

namespace {

struct Record {
    std::shared_ptr<const tss_encoding_data> d;
    PlatformLimits limits;
    std::shared_ptr<const Cnf> cnf;   // what with_limits returned (base clauses first, then the lowered limits)
};
std::mutex g_mutex;
std::deque<Record> g_records;   // most recent first
constexpr size_t kMaxRecords = 8;

bool same_prefix(const Cnf& base, const int32_t* lits, const uint32_t* offsets, int n_clauses) {
    if (base.n_clauses() > n_clauses) return false;
    const size_t nl = base.lits.size();
    if (offsets[base.n_clauses()] != nl) return false;
    return std::memcmp(base.offsets.data(), offsets, sizeof(uint32_t) * base.offsets.size()) == 0 &&
           (nl == 0 || std::memcmp(base.lits.data(), lits, sizeof(int32_t) * nl) == 0);
}

}  // namespace

namespace tss {
void instance_record(const std::shared_ptr<const tss_encoding_data>& d, const PlatformLimits& limits, const std::shared_ptr<const Cnf>& cnf) {
    std::lock_guard<std::mutex> lock(g_mutex);
    g_records.push_front(Record{d, limits, cnf});
    if (g_records.size() > kMaxRecords) g_records.pop_back();
}
}  // namespace tss

// TSS_TRACE=1: wall microseconds of the stages of tss_solve_instance / tss_witness_for_cnf on stderr (profiles/tss_repl_timing.py)
namespace {
struct Trace {
    bool on = std::getenv("TSS_TRACE") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void lap(const char* what) {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[tss trace] %-28s %8.1f us\n", what, std::chrono::duration<double, std::micro>(now - t).count());
        t = now;
    }
};
}  // namespace

extern "C" {

int tss_cnf_num_vars(const tss_cnf* c);   // cnf.cu

int tss_instance_find(const int32_t* lits, const uint32_t* offsets, int32_t n_clauses, int32_t n_vars, tss_encoding** enc_out,
                      tss_instance_info* info, int32_t* weights, int32_t weights_cap) {
    if (!offsets || n_clauses < 0 || !enc_out || !info || (offsets[n_clauses] > 0 && !lits)) return TSS_E_INVALID;
    *enc_out = nullptr;
    std::memset(info, 0, sizeof *info);
    std::lock_guard<std::mutex> lock(g_mutex);
    const Record* hit = nullptr;
    bool exact = false;
    for (const Record& r : g_records) {   // the whole CNF as recorded (most recent first) ...
        if (r.cnf->n_vars == n_vars && r.cnf->n_clauses() == n_clauses && same_prefix(*r.cnf, lits, offsets, n_clauses)) { hit = &r; exact = true; break; }
    }
    if (!hit)
        for (const Record& r : g_records) {   // ... else the same base clauses (limits lowered by someone else's encoder): limits of the latest record
            if (r.d->enc.base.n_vars <= n_vars && same_prefix(r.d->enc.base, lits, offsets, n_clauses)) { hit = &r; break; }
        }
    if (!hit) return TSS_UNKNOWN;
    tss_encoding* enc = new (std::nothrow) tss_encoding();
    if (!enc) return TSS_E_INVALID;
    enc->d = hit->d;
    enc->has_card_limits = true;
    for (const auto& c : hit->limits.card_limits) enc->card_limits.insert(enc->card_limits.end(), {c.def.w, c.def.h, (int32_t)std::min(c.value, (long)INT32_MAX)});
    *enc_out = enc;
    info->w = hit->d->enc.w;
    info->h = hit->d->enc.h;
    info->n_defs = (int32_t)hit->d->enc.defs.size();
    info->card_limit_1x1 = -1;
    for (const auto& c : hit->limits.card_limits) {
        if (c.def.w == 1 && c.def.h == 1) info->card_limit_1x1 = (int32_t)c.value;
        else info->n_other_card_limits++;
    }
    info->has_weight_limit = hit->limits.has_weight_limit;
    info->weight_limit = hit->limits.weight_limit;
    info->n_weights = (int32_t)hit->limits.weights.size();
    info->exact = exact;
    if (weights)
        for (int i = 0; i < info->n_weights && i < weights_cap; i++) {
            weights[3 * i] = hit->limits.weights[(size_t)i].def.w;
            weights[3 * i + 1] = hit->limits.weights[(size_t)i].def.h;
            weights[3 * i + 2] = (int32_t)hit->limits.weights[(size_t)i].value;
        }
    return TSS_SAT;
}

int tss_encoding_terrain(const tss_encoding* enc, uint8_t* grid, size_t cap, int32_t* w, int32_t* h) {
    if (!enc || !w || !h) return TSS_E_INVALID;
    *w = enc->d->enc.w;
    *h = enc->d->enc.h;
    if (!grid || cap < enc->d->grid.size()) return TSS_E_CAPACITY;
    std::memcpy(grid, enc->d->grid.data(), enc->d->grid.size());
    return TSS_OK;
}

int tss_encoding_defs(const tss_encoding* enc, tss_dims* defs, int32_t cap, int32_t* n) {
    if (!enc || !n) return TSS_E_INVALID;
    *n = (int32_t)enc->d->enc.defs.size();
    if (!defs || cap < *n) return TSS_E_CAPACITY;
    for (int i = 0; i < *n; i++) defs[i] = tss_dims{enc->d->enc.defs[(size_t)i].w, enc->d->enc.defs[(size_t)i].h};
    return TSS_OK;
}

int tss_witness_for_cnf(tss_engine* e, const tss_cnf* c, const tss_encoding* enc, const tss_platform* plats, int32_t n, uint8_t* assignment) {
    if (!e) return TSS_E_INVALID;
    if (!c || !enc || !assignment || n < 0 || (n > 0 && !plats)) return e->fail(TSS_E_INVALID, "tss_witness_for_cnf: bad arguments");
    const int nv = tss_cnf_num_vars(c), nb = enc->d->enc.base.n_vars;
    if (nv < nb) return e->fail(TSS_E_INVALID, "tss_witness_for_cnf: the CNF has %d variables, the encoding %d", nv, nb);
    // platform variables from the layout (every dims key contained in a platform, encoder.rs:449-458), terrain layers from the
    // evaluator's support layers (kernel (a)); whatever the limits added (totalizer / PB auxiliaries) starts unassigned
    Trace tr;
    int rc = tss_layout_to_assignment(e, enc, plats, n, assignment);
    if (rc < 0) return rc;
    tr.lap("witness: layout_to_assignment");
    std::memset(assignment + nb + 1, 2, (size_t)(nv - nb));
    int32_t conflict = -1, n_falsified = 0;
    // ... and is implied: unit propagation assigns it, open variables become False, and the model is checked against every
    // clause the exact solver received (kernel (c)) — in ONE launch when the variables fit a CTA's shared memory
    rc = tss_cnf_complete(e, c, assignment, &conflict, &n_falsified);
    if (rc < 0) return rc;
    tr.lap("witness: cnf_complete");
    if (conflict >= 0) return TSS_UNKNOWN;   // e.g. more platforms than the bound allows
    return n_falsified == 0 ? TSS_SAT : TSS_UNKNOWN;
}

int tss_engine_certified_unsat(tss_engine* e, int enabled) {
    if (!e) return TSS_E_INVALID;
    e->certified_unsat = enabled != 0;
    return TSS_OK;
}

int tss_solve_instance(tss_engine* e, const tss_cnf* c, const tss_encoding* enc, const tss_instance_info* info, const int32_t* weights,
                       uint64_t seed, int64_t give_up_steps, uint8_t* assignment) {
    if (!e) return TSS_E_INVALID;
    if (!c || !enc || !info || !assignment) return e->fail(TSS_E_INVALID, "tss_solve_instance: bad arguments");
    const Encoding& E = enc->d->enc;
    // per-type limits: the placement search steers by the limits recorded on a handle of tss_instance_find, on grids up to 32x32,
    // with one objective (the platform count or the total weight); anything else is left to the exact solver
    const bool per_type = info->n_other_card_limits > 0;
    if (per_type && (!enc->has_card_limits || E.w > 32 || E.h > 32 || (info->has_weight_limit && info->card_limit_1x1 >= 0))) return TSS_UNKNOWN;
    std::vector<tss_dims> defs;
    for (const Dims& d : E.defs) defs.push_back(tss_dims{d.w, d.h});
    // A limit below a CERTIFIED lower bound has no model: answer UNSAT without searching.  Only when the platform count is the
    // sole limit (the REPL's loop); the integral packing first (~0.1 ms, computed once per instance), the fractional LP only after
    // the search came back empty-handed.
    Trace tr;
    const bool small = e->certified_unsat && E.w <= 32 && E.h <= 32;
    const bool count_only = small && info->card_limit_1x1 >= 0 && !info->has_weight_limit;
    const bool weight_only = small && info->card_limit_1x1 < 0 && info->has_weight_limit && info->n_weights > 0 && weights;
    if (weight_only) {
        std::lock_guard<std::mutex> lock(enc->d->bounds_mutex);
        if (enc->d->lp_weight_bound >= 0 && enc->d->lp_weights == std::vector<int32_t>(weights, weights + 3 * (size_t)info->n_weights) &&
            info->weight_limit < enc->d->lp_weight_bound)
            return TSS_UNSAT;
    }
    if (count_only) {
        std::lock_guard<std::mutex> lock(enc->d->bounds_mutex);
        if (enc->d->packing_bound == -1) {
            int32_t lb = 0;
            enc->d->packing_bound = tss_lower_bound(e, enc->d->grid.data(), E.w, E.h, defs.data(), (int32_t)defs.size(), seed, 0, nullptr, 0, &lb) == TSS_OK ? lb : -2;
        }
        tr.lap("solve: packing bound");
        if (enc->d->packing_bound >= 0 && info->card_limit_1x1 < enc->d->packing_bound) return TSS_UNSAT;
        if (enc->d->lp_count_bound >= 0 && info->card_limit_1x1 < enc->d->lp_count_bound) return TSS_UNSAT;
    }
    std::vector<tss_platform> plats((size_t)E.w * E.h + 1);
    int32_t n = 0;
    auto search = [&](int64_t give_up, uint64_t sd) -> int {   // a SAT-like call with a give-up point (tss.h)
        int r;
        if (per_type) {
            const bool weighted = info->has_weight_limit && info->n_weights > 0 && weights;
            int64_t obj = 0;
            r = tss_solve_with_limits(e, enc->d->grid.data(), E.w, E.h, defs.data(), (int32_t)defs.size(), enc->card_limits.data(),
                                      (int32_t)(enc->card_limits.size() / 3), weighted ? weights : nullptr, weighted ? info->n_weights : 0,
                                      weighted ? info->weight_limit : -1, sd, 0, give_up > 0 ? -give_up : 0, plats.data(), (int32_t)plats.size(), &n, &obj);
        } else if (info->has_weight_limit && info->n_weights > 0 && weights) {
            int64_t wt = 0;
            r = tss_solve_min_weight(e, enc->d->grid.data(), E.w, E.h, defs.data(), (int32_t)defs.size(), weights, info->n_weights, info->weight_limit, sd, 0,
                                     give_up > 0 ? give_up : 0, plats.data(), (int32_t)plats.size(), &n, &wt);
        } else {
            r = tss_solve_upper_bound(e, enc->d->grid.data(), E.w, E.h, defs.data(), (int32_t)defs.size(), info->card_limit_1x1, sd, 0, give_up > 0 ? -give_up : 0,
                                      plats.data(), (int32_t)plats.size(), &n);
        }
        tr.lap("solve: search");
        return r;
    };
    // The fractional bound, asked only for what this call needs — "does the bound reach limit + 1?" — so the simplex may stop
    // early; computed again, to the new target, only if a later call asks about a limit the cached bound does not settle and the
    // solve was not final.  true = the limit lies below the certified bound.
    const std::vector<int32_t> wv = weight_only ? std::vector<int32_t>(weights, weights + 3 * (size_t)info->n_weights) : std::vector<int32_t>();
    auto count_pending = [&] { return enc->d->lp_count_bound == -1 || (enc->d->lp_count_bound >= 0 && !enc->d->lp_count_final && info->card_limit_1x1 >= enc->d->lp_count_bound); };
    auto weight_pending = [&] {
        return enc->d->lp_weight_bound == -1 || enc->d->lp_weights != wv || (enc->d->lp_weight_bound >= 0 && !enc->d->lp_weight_final && info->weight_limit >= enc->d->lp_weight_bound);
    };
    auto lp_refutes = [&]() -> bool {
        std::lock_guard<std::mutex> lock(enc->d->bounds_mutex);
        int64_t lb = 0;
        int32_t lp_info[3] = {0, 0, 0};
        if (count_only) {
            if (count_pending()) {
                const int ok = tss_lower_bound_lp(e, enc->d->grid.data(), E.w, E.h, defs.data(), (int32_t)defs.size(), nullptr, 0, 0, (int64_t)info->card_limit_1x1 + 1,
                                                  nullptr, nullptr, nullptr, &lb, lp_info);
                enc->d->lp_count_bound = ok == TSS_OK ? lb : -2;
                enc->d->lp_count_final = lp_info[1] != 0;
                tr.lap("solve: fractional bound");
            }
            return enc->d->lp_count_bound >= 0 && info->card_limit_1x1 < enc->d->lp_count_bound;
        }
        if (weight_only) {   // the same question about the GUI's weight limit (crates/gui/src/app.rs:235-239)
            if (weight_pending()) {
                enc->d->lp_weights = wv;
                const int ok = tss_lower_bound_lp(e, enc->d->grid.data(), E.w, E.h, defs.data(), (int32_t)defs.size(), weights, info->n_weights, 0, info->weight_limit + 1,
                                                  nullptr, nullptr, nullptr, &lb, lp_info);
                enc->d->lp_weight_bound = ok == TSS_OK ? lb : -2;
                enc->d->lp_weight_final = lp_info[1] != 0;
                tr.lap("solve: fractional bound (weights)");
            }
            return enc->d->lp_weight_bound >= 0 && info->weight_limit < enc->d->lp_weight_bound;
        }
        return false;
    };
    // When the bound for this limit is still to be computed, the search first gets an eighth of its give-up budget: the limits of
    // the loop's last iterations are the ones nothing satisfies, and there the long search was the larger half of the call
    // (test/ex2.toml with 1x1 supports, limit 13: 1.6 ms of searching before 3.3 ms of simplex).  Found nothing and not refuted:
    // the search runs again with the whole budget and other seeds.
    bool pending = false;
    if (count_only || weight_only) {
        std::lock_guard<std::mutex> lock(enc->d->bounds_mutex);
        pending = count_only ? count_pending() : weight_pending();
    }
    const int64_t first_budget = give_up_steps / 8 > 128 ? give_up_steps / 8 : 128;
    const bool two_phase = pending && give_up_steps > first_budget;
    int rc = search(two_phase ? first_budget : give_up_steps, seed);
    if (rc == TSS_SAT) return tss_witness_for_cnf(e, c, enc, plats.data(), n, assignment);
    if (rc == TSS_UNKNOWN && (count_only || weight_only) && !e->interrupted()) {   // nothing found within the limit: can the fractional bound certify that nothing exists?
        if (lp_refutes()) return TSS_UNSAT;
        if (two_phase) {
            rc = search(give_up_steps, seed ^ 0x9e3779b97f4a7c15ull);
            if (rc == TSS_SAT) return tss_witness_for_cnf(e, c, enc, plats.data(), n, assignment);
        }
    }
    return rc;
}

}  // extern "C"
