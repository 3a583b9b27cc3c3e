// TEST INFRASTRUCTURE ONLY: the scalar replay of the placement search with per-type platform limits
// (timberborn_support_solver_b200/csrc/sls_multi.cu sls_multi_kernel<false, false, true>), built and bound by
// tests/limits_model.py.
//
// The oracle's model of the placement search (oracle/slsm_model.cpp) is included as it stands: its Runner keeps the terrain,
// the cover counts, the removal rule and the hash functions.  Only the step loop is restated here, with the two rules the
// limits add: n_j = the current platforms whose key lies in class j (mask[key] bit j), full = { j : n_j >= limit[j] } after
// every flip; an addition whose key lies in a full class is no candidate, and the swap trigger compares against the smallest
// cost of a key in no full class.  Without classes this loop is the oracle's step for step.
#include "../oracle/slsm_model.cpp"

namespace {

struct LimitedRunner : Runner {
    const int* mask;
    const int* lim;
    int n_classes;
    int ncls[32] = {0};
    uint32_t full = 0;
    int cfree = 0;

    LimitedRunner(const Terrain& t, const int* k, const int* cs, int nk, Chain& ch, uint32_t b, const int* m, const int* l, int nc)
        : Runner(t, k, cs, nk, ch, b), mask(m), lim(l), n_classes(nc) {}

    void count(int code, int sign) {
        for (int j = 0; j < n_classes; j++)
            if ((mask[code >> 10] >> j) & 1) ncls[j] += sign;
        full = 0;
        for (int j = 0; j < n_classes; j++)
            if (ncls[j] >= lim[j]) full |= 1u << j;
        cfree = 1 << 30;
        for (int q = 0; q < n_keys; q++)
            if (!((uint32_t)mask[q] & full)) cfree = std::min(cfree, costs[q]);
    }
    uint32_t uncovered_rows() const {
        uint32_t rowmask = 0;
        for (int y = 0; y < 32; y++)
            for (int x = 0; x < 32; x++)
                if (T.ceil[y][x] && cnt[y * 32 + x] == 0) rowmask |= 1u << y;
        return rowmask;
    }

    void run(long long steps, int epoch_bound, int target, int noise_pct) {
        if (c.done) return;
        if (target >= 0 && epoch_bound <= target) return;
        std::memset(cnt, 0, sizeof cnt);
        std::memset(occ, 0, sizeof occ);
        int Wt = 0;
        for (int i = 0; i < c.k; i++) {
            apply(c.items[i], +1);
            Wt += costs[c.items[i] >> 10];
            count(c.items[i], +1);
        }
        count(0, 0);
        long long it = 0;
        for (; it < steps; it++, c.step++) {
            const int limit = std::min(epoch_bound, c.best);
            const uint32_t hs = step_hash(base, c.step);
            uint32_t hl[32];
            for (int l = 0; l < 32; l++) hl[l] = lane_hash(hs, (uint32_t)l);
            if (Wt >= limit) {
                if (c.k == 0) { c.done = 1; break; }
                scored += (uint64_t)c.k;
                c.tabu_add = remove_min_loss(hl, -1);
                Wt -= costs[c.tabu_add >> 10];
                count(c.tabu_add, -1);
                continue;
            }
            uint32_t rowmask = uncovered_rows();
            if (!rowmask) {
                c.best = Wt;
                c.best_items = c.items;
                c.best_k = c.k;
                if (Wt <= target || c.k == 0) { c.done = 1; it++; c.step++; break; }
                continue;
            }
            if (Wt + cfree >= limit && c.k > 0) {
                scored += (uint64_t)c.k;
                c.tabu_add = remove_min_loss(hl, c.tabu_rem);
                Wt -= costs[c.tabu_add >> 10];
                count(c.tabu_add, -1);
                rowmask = uncovered_rows();
            }
            const int ty = pick_rotated(rowmask, hs & 31u);
            uint32_t urow = 0;
            for (int x = 0; x < 32; x++)
                if (T.ceil[ty][x] && cnt[ty * 32 + x] == 0) urow |= 1u << x;
            const int tx = pick_rotated(urow, (hs >> 5) & 31u);
            const bool noise = ((hs >> 10) & 127u) < noise_q7(noise_pct);
            uint32_t best_key = 0;
            int best_code = -1;
            for (int pass = 0; pass < 2; pass++) {
                uint32_t mx = 0;
                int mx_code = 0, n_inb = 0;
                for (int l = 0; l < 32; l++) {
                    const uint32_t r = lane_hash(hl[l], (uint32_t)(pass + 40));
                    const uint32_t u = r & 0xffffu;
                    const int key = pass == 0 ? (int)((u * (uint32_t)n_keys) >> 16) : order[(((u * u) >> 16) * (uint32_t)n_keys) >> 16];
                    const int w = keys[2 * key], h = keys[2 * key + 1];
                    const int x = tx - 3 - (w - 1) + (int)((((r >> 16) & 0xffu) * (uint32_t)(w + 6)) >> 8);
                    const int y = ty - 3 - (h - 1) + (int)(((r >> 24) * (uint32_t)(h + 6)) >> 8);
                    const bool inb = x >= 0 && y >= 0 && x + w <= T.W && y + h <= T.H;
                    if (!inb) continue;
                    n_inb++;
                    const int code = (key << 10) | (y << 5) | x;
                    const int g = count_in_reach(x, y, w, h, 0), cost = costs[key];
                    const bool blocked = ((uint32_t)mask[key] & full) != 0;
                    const bool ok = !overlaps(x, y, w, h) && g > 0 && code != c.tabu_add && Wt + cost < limit && !blocked;
                    if (!ok) continue;
                    const uint32_t rank = ((uint32_t)g * 64u) / (uint32_t)cost;
                    const uint32_t kk = ((noise ? 0x10000u : (rank << 16)) | ((r >> 16) ^ (r & 0xffffu))) | 1u;
                    if (kk > mx) { mx = kk; mx_code = code; }
                }
                scored += (uint64_t)n_inb;
                if (mx > best_key) { best_key = mx; best_code = mx_code; }
            }
            if (best_code < 0) continue;
            apply(best_code, +1);
            c.items.push_back((uint16_t)best_code);
            c.k++;
            Wt += costs[best_code >> 10];
            count(best_code, +1);
            c.tabu_rem = best_code;
            flips++;
        }
        steps_done += (uint64_t)it;
    }
};

}  // namespace

extern "C" {

// tsso_slsm_model's interface plus mask[n_keys] (classes of each key) and lim[n_classes].
int limits_model(const uint8_t* grid, int w, int h, const int* keys, const int* costs, int n_keys, const int* mask, const int* lim, int n_classes,
                 int n_chains, uint32_t chain_offset, uint64_t seed, int noise_pct, const long long* epochs, int n_epochs, int share_bound,
                 uint16_t* out_items, int* out_k, uint16_t* out_best_items, int* out_best_k, int* out_best, uint32_t* out_step, uint64_t* totals) {
    if (w > 32 || h > 32 || n_keys < 1 || n_keys > 16 || n_classes < 0 || n_classes > 16) return -1;
    Terrain T;
    T.W = w; T.H = h;
    std::memset(T.ceil, 0, sizeof T.ceil);
    for (int y = 0; y < h; y++)
        for (int x = 0; x < w; x++) T.ceil[y][x] = grid[y * w + x] != 0;
    std::vector<Chain> chains(n_chains);
    int shared = NO_BOUND;
    totals[0] = totals[1] = totals[2] = 0;
    for (int e = 0; e < n_epochs; e++) {
        long long steps = epochs[3 * e];
        int bound = (int)epochs[3 * e + 1], target = (int)epochs[3 * e + 2];
        if (share_bound) bound = std::min(bound, shared);
        for (int i = 0; i < n_chains; i++) {
            LimitedRunner r(T, keys, costs, n_keys, chains[i], chain_base(seed, chain_offset + (uint32_t)i), mask, lim, n_classes);
            r.run(steps, bound, target, noise_pct);
            totals[0] += r.scored;
            totals[1] += r.steps_done;
            totals[2] += r.flips;
        }
        for (auto& c : chains) shared = std::min(shared, c.best);
    }
    for (int i = 0; i < n_chains; i++) {
        std::memset(out_items + (size_t)i * MAX_ITEMS, 0, sizeof(uint16_t) * MAX_ITEMS);
        std::memset(out_best_items + (size_t)i * MAX_ITEMS, 0, sizeof(uint16_t) * MAX_ITEMS);
        std::copy(chains[i].items.begin(), chains[i].items.end(), out_items + (size_t)i * MAX_ITEMS);
        std::copy(chains[i].best_items.begin(), chains[i].best_items.end(), out_best_items + (size_t)i * MAX_ITEMS);
        out_k[i] = chains[i].k; out_best[i] = chains[i].best; out_best_k[i] = chains[i].best_k; out_step[i] = chains[i].step;
    }
    return 0;
}

}  // extern "C"
