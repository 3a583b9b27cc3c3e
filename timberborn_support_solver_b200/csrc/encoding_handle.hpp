// The object behind `tss_encoding*` (include/tss.h) and the process-wide instance registry that lets a solver which is handed
// a bare CNF (crates/repl/src/solver_runner.rs:8-20) find the terrain, platform set, variable map and limits it came from.
#pragma once
#include <memory>
#include <mutex>
#include <vector>

#include "host_model.hpp"

struct tss_encoding_data {
    tss::Encoding enc;
    std::vector<uint8_t> grid;
    // certified lower bounds of this terrain / platform set, computed at most once (tss_solve_instance): the bound-tightening loop
    // asks about the same instance with a smaller limit every iteration (crates/repl/src/main.rs:346)
    mutable std::mutex bounds_mutex;
    mutable int packing_bound = -1;        // tss_lower_bound; -1 = not computed, -2 = not available for this instance
    mutable long long lp_count_bound = -1; // tss_lower_bound_lp on the platform count
    mutable bool lp_count_final = false, lp_weight_final = false;   // the simplex ran to optimality (not stopped at a target): asking again cannot improve the bound
    mutable std::vector<int32_t> lp_weights;   // the weight table `lp_weight_bound` was computed for
    mutable long long lp_weight_bound = -1;    // tss_lower_bound_lp on the total weight
    // the per-type records (def_w, def_h, limit; 1x1 excluded) each LP bound above was computed with (tss_lower_bound_lp_limits);
    // empty: the plain LP of the whole set, which holds for every limit
    mutable std::vector<int32_t> lp_count_card, lp_weight_card;
    // the CNF of the last tss_encoding_with_limits call: callers ask twice, once for the sizes and once for the clauses, and the
    // registry keeps the same object (no second lowering of the limits, no copy of the clauses)
    mutable std::mutex lowered_mutex;
    mutable tss::PlatformLimits lowered_limits;
    mutable std::shared_ptr<const tss::Cnf> lowered;
};

// a handle is a shared reference: the registry keeps encodings alive after the caller destroyed its own handle
struct tss_encoding {
    std::shared_ptr<const tss_encoding_data> d;
    // a handle from tss_instance_find: the recorded PlatformLimits.card_limits as (def_w, def_h, limit) records, 1x1 included
    bool has_card_limits = false;
    std::vector<int32_t> card_limits;
};

namespace tss {
// records (encoding, limits, the CNF with_limits produced); called by tss_encoding_with_limits
void instance_record(const std::shared_ptr<const tss_encoding_data>& d, const PlatformLimits& limits, const std::shared_ptr<const Cnf>& cnf);
}  // namespace tss
