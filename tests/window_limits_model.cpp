// TEST INFRASTRUCTURE ONLY: the scalar replay of the window-decomposed placement search's chains under per-window class budgets
// (timberborn_support_solver_b200/csrc/sls_multi.cu sls_multi_kernel<false, true, true>, driven by csrc/lns_placements.cu), built
// and bound by tests/window_limits_model.py.
//
// The replay of the WINDOW step rule (tests/window_model.cpp) is included as it stands: its Runner keeps the window's terrain,
// need and occupancy boards, the box, the cover counts, the removal rule and the hash functions.  Only the step loop is restated
// here, with the class counters of the LIMITS rule (as tests/limits_model.cpp restates them for the epoch kernel): n_j = the
// current platforms whose key lies in class j, full = { j : n_j >= budget[j] } after every flip; an addition whose key lies in a
// full class is no candidate, and the swap trigger compares against the smallest cost of a key in no full class.  Without
// classes this loop is window_model.cpp's step for step.
#include "window_model.cpp"

namespace {

struct WindowLimitedRunner : Runner {
    const int* mask;
    const int* lim;   // the window's budgets
    int n_classes;
    int ncls[32] = {0};
    uint32_t full = 0;
    int cfree = 0;
    int binding = 0;   // some class was full at some point: only then can the run differ from window_model.cpp's

    WindowLimitedRunner(const Terrain& t, const int* k, const int* cs, int nk, Chain& ch, uint32_t b, const int* m, const int* l, int nc)
        : Runner(t, k, cs, nk, ch, b), mask(m), lim(l), n_classes(nc) {}

    void count(int code, int sign) {
        for (int j = 0; j < n_classes; j++)
            if ((mask[code >> 10] >> j) & 1) ncls[j] += sign;
        full = 0;
        for (int j = 0; j < n_classes; j++)
            if (ncls[j] >= lim[j]) full |= 1u << j;
        binding |= full != 0;
        cfree = 1 << 30;
        for (int q = 0; q < n_keys; q++)
            if (!((uint32_t)mask[q] & full)) cfree = std::min(cfree, costs[q]);
    }
    uint32_t uncovered_rows() const {
        uint32_t rowmask = 0;
        for (int y = 0; y < 32; y++)
            for (int x = 0; x < 32; x++)
                if (needs(y, x) && cnt[y * 32 + x] == 0) rowmask |= 1u << y;
        return rowmask;
    }

    void run(long long steps, int noise_pct) {   // one epoch without a bound or target, as lns_placements.cu launches it
        if (c.done) return;
        std::memset(cnt, 0, sizeof cnt);
        std::memcpy(occ, occ0, sizeof occ);
        int Wt = 0;
        for (int i = 0; i < c.k; i++) {
            apply(c.items[i], +1);
            Wt += costs[c.items[i] >> 10];
            count(c.items[i], +1);
        }
        count(0, 0);
        long long it = 0;
        for (; it < steps; it++, c.step++) {
            const int limit = std::min(NO_BOUND, c.best);
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
                if (c.k == 0) { c.done = 1; it++; c.step++; break; }
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
                if (needs(ty, x) && cnt[ty * 32 + x] == 0) urow |= 1u << x;
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
                    const bool inb = x >= box[0] && y >= box[1] && x + w <= box[2] && y + h <= box[3];
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

// tsso_slsm_window_model's interface plus mask[n_keys] (classes of each key), budget[n_classes] (the window's class budgets) and
// out_ncls[n_chains][16] = each chain's class counts of its best layout, out_binding[n_chains] = 1 if a class of the chain was
// ever full (else its run is tsso_slsm_window_model's).
int tsso_slsm_window_limits_model(const uint8_t* terrain, const uint8_t* need, const uint8_t* occ, const int* box, const int* keys, const int* costs,
                                  int n_keys, int n_chains, uint32_t chain_offset, uint64_t seed, int noise_pct, long long steps, const uint16_t* items,
                                  int n_items, int best, uint32_t step, const int* mask, const int* budget, int n_classes, uint16_t* out_best_items,
                                  int* out_best_k, int* out_best, int* out_ncls, int* out_binding, uint64_t* totals) {
    if (n_keys < 1 || n_keys > 16 || n_items < 0 || n_items > MAX_ITEMS || n_classes < 1 || n_classes > 16) return -1;
    Terrain T;
    T.W = 32; T.H = 32;
    for (int y = 0; y < 32; y++)
        for (int x = 0; x < 32; x++) T.ceil[y][x] = terrain[y * 32 + x] != 0;
    for (int i = 0; i < n_chains; i++) {
        Chain c;
        c.items.assign(items, items + n_items);
        c.best_items = c.items;
        c.k = c.best_k = n_items;
        c.best = best;
        c.step = step;
        WindowLimitedRunner r(T, keys, costs, n_keys, c, chain_base(seed, chain_offset + (uint32_t)i), mask, budget, n_classes);
        r.need = need;
        r.occ0 = occ;
        for (int j = 0; j < 4; j++) r.box[j] = box[j];
        r.run(steps, noise_pct);
        totals[0] += r.scored;
        totals[1] += r.steps_done;
        totals[2] += r.flips;
        std::memset(out_best_items + (size_t)i * MAX_ITEMS, 0, sizeof(uint16_t) * MAX_ITEMS);
        std::copy(c.best_items.begin(), c.best_items.end(), out_best_items + (size_t)i * MAX_ITEMS);
        out_best_k[i] = c.best_k;
        out_best[i] = c.best;
        out_binding[i] = r.binding;
        for (int j = 0; j < 16; j++) out_ncls[i * 16 + j] = 0;
        for (int q = 0; q < c.best_k; q++)
            for (int j = 0; j < n_classes; j++) out_ncls[i * 16 + j] += (mask[c.best_items[q] >> 10] >> j) & 1;
    }
    return 0;
}

}  // extern "C"
