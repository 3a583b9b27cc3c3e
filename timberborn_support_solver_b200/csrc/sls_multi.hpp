// Chain state of the placement search (sls_multi.cu), shared with the window-decomposed placement search that drives it on
// grids larger than 32x32 (lns_placements.cu).
#pragma once
#include <cstdint>

#include <cuda_runtime.h>

namespace tss {
namespace slsm {

constexpr int MAX_ITEMS = 1024;
constexpr int MAX_KEYS = 16;

struct MultiState {  // persistent per-chain state in HBM
    uint16_t items[MAX_ITEMS];       // key << 10 | y << 5 | x
    uint16_t best_items[MAX_ITEMS];
    int32_t k, best;      // platforms now; best OBJECTIVE value found (platform count, or total weight in weight mode)
    uint32_t step;
    int32_t tabu_add, tabu_rem, done;
    int32_t best_k;       // number of platforms in best_items
    uint32_t pad[1];
};

// Per-window inputs of sls_multi_kernel<false, true>.  `need`: the tiles the window still has to cover (its ceiling minus
// the cover of the platforms frozen for the phase); it replaces the ceiling in the uncovered and covered-once boards.
// `occ`: the frozen footprints, the occupancy every chain of the window starts from.  `box` = (x0, y0, x1, y1): an
// addition must satisfy x0 <= x, x + w <= x1, y0 <= y, y + h <= y1, which keeps its reach inside the window.
struct WindowM {
    const uint32_t* need;         // [n_windows][32]
    const uint32_t* occ;          // [n_windows][32]
    const int4* box;              // [n_windows]
    int seeds;                    // chains per window: chain c belongs to window c / seeds
};

}  // namespace slsm
}  // namespace tss
