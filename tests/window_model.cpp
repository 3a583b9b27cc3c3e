// TEST INFRASTRUCTURE ONLY: the scalar replay of the window-decomposed placement search's chains
// (timberborn_support_solver_b200/csrc/sls_multi.cu sls_multi_kernel<false, true>, driven by csrc/lns_placements.cu), built
// and bound by tests/window_model.py.
//
// The step rule is the placement search's, restated tile by tile exactly as oracle/slsm_model.cpp does (constants and hash
// functions re-declared, the kernel's 32 candidate lanes emulated sequentially) with the three differences of WINDOW mode:
// the tiles that still need cover replace the ceiling in the uncovered / covered-once tests, the occupancy starts at the
// frozen footprints, and additions must lie inside the window's box.  Feasibility and objective are those of the reference
// (oracle/slsm_model.cpp's header cites them): footprints in bounds and disjoint, a tile is supported iff it is within three
// ceiling-masked 4-neighbour steps of a ceiling tile under some footprint, objective = total cost of the platforms.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

constexpr uint32_t K1 = 0x9E3779B9u, K2 = 0x85EBCA6Bu;
constexpr int NO_BOUND = 1 << 20;
constexpr int MAX_ITEMS = 1024;

uint32_t fmix32(uint32_t h) { h ^= h >> 16; h *= 0x85EBCA6Bu; h ^= h >> 13; h *= 0xC2B2AE35u; h ^= h >> 16; return h; }
uint32_t chain_base(uint64_t seed, uint32_t chain) { return fmix32((uint32_t)seed ^ fmix32((uint32_t)(seed >> 32) + chain * K1 + 0x5bd1e995u)); }
uint32_t step_hash(uint32_t base, uint32_t step) { return fmix32(base ^ (step * K1)); }
uint32_t lane_hash(uint32_t hs, uint32_t lane) { return fmix32(hs ^ ((lane + 1u) * K2)); }
uint32_t noise_q7(int noise_pct) { return (uint32_t)((noise_pct * 128 + 50) / 100); }
uint32_t tie_remove_hl(uint32_t hl, uint32_t chunk) { return (hl * (2u * chunk + 1u)) >> 16; }

int pick_rotated(uint32_t bits, uint32_t o) {
    uint32_t rot = o ? ((bits >> o) | (bits << (32 - o))) : bits;
    return (int)((__builtin_ctz(rot) + o) & 31u);
}

struct Terrain {
    int W, H;
    uint8_t ceil[32][32];  // [y][x]
};

// tiles supported by a platform with footprint (x, y, w, h): three ceiling-masked dilations from the ceiling under it
std::vector<int> reach_of(const Terrain& T, int x, int y, int w, int h) {
    uint8_t sup[32][32];
    std::memset(sup, 0, sizeof sup);
    for (int yy = y; yy < y + h; yy++)
        for (int xx = x; xx < x + w; xx++)
            if (yy >= 0 && yy < 32 && xx >= 0 && xx < 32 && T.ceil[yy][xx]) sup[yy][xx] = 1;
    // (paths of length <= 3 from the footprint stay inside the box footprint + 3 on every side)
    const int x0 = std::max(x - 3, 0), x1 = std::min(x + w + 3, 32), y0 = std::max(y - 3, 0), y1 = std::min(y + h + 3, 32);
    for (int round = 0; round < 3; round++) {
        uint8_t nxt[32][32];
        std::memcpy(nxt, sup, sizeof sup);
        for (int yy = y0; yy < y1; yy++)
            for (int xx = x0; xx < x1; xx++) {
                if (!sup[yy][xx]) continue;
                const int nx[4] = {xx + 1, xx, xx - 1, xx}, ny[4] = {yy, yy + 1, yy, yy - 1};
                for (int d = 0; d < 4; d++)
                    if (nx[d] >= 0 && nx[d] < 32 && ny[d] >= 0 && ny[d] < 32 && T.ceil[ny[d]][nx[d]]) nxt[ny[d]][nx[d]] = 1;
            }
        std::memcpy(sup, nxt, sizeof sup);
    }
    std::vector<int> out;
    for (int yy = y0; yy < y1; yy++)
        for (int xx = x0; xx < x1; xx++)
            if (sup[yy][xx]) out.push_back(yy * 32 + xx);
    return out;
}

struct Chain {
    std::vector<uint16_t> items, best_items;
    int k = 0, best = NO_BOUND, best_k = 0, tabu_add = -1, tabu_rem = -1, done = 0;
    uint32_t step = 0;
};

struct Runner {
    const Terrain& T;
    const int* keys;   // (w, h) per key
    const int* costs;
    std::vector<int> order;  // keys by area, largest first (stable)
    int n_keys;
    Chain& c;
    uint32_t base;
    uint8_t cnt[1024], occ[1024];
    uint64_t scored = 0, steps_done = 0;
    // WINDOW mode (the window-decomposed placement search, csrc/lns_placements.cu): `need` = the tiles still to be covered
    // (replaces the ceiling in the uncovered / covered-once tests), `occ0` = the frozen footprints every run starts from, and
    // additions must lie inside `box` = (x0, y0, x1, y1).  Outside WINDOW mode: the ceiling, no occupancy, the grid.
    const uint8_t* need = nullptr;
    const uint8_t* occ0 = nullptr;
    int box[4];

    Runner(const Terrain& t, const int* k, const int* cs, int nk, Chain& ch, uint32_t b) : T(t), keys(k), costs(cs), n_keys(nk), c(ch), base(b) {
        box[0] = 0; box[1] = 0; box[2] = t.W; box[3] = t.H;
        order.resize(nk);
        for (int i = 0; i < nk; i++) order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](int a, int bb) { return keys[2 * a] * keys[2 * a + 1] > keys[2 * bb] * keys[2 * bb + 1]; });
    }

    bool needs(int y, int x) const { return need ? need[y * 32 + x] != 0 : T.ceil[y][x] != 0; }
    void dims(int code, int& x, int& y, int& w, int& h) const { x = code & 31; y = (code >> 5) & 31; w = keys[2 * (code >> 10)]; h = keys[2 * (code >> 10) + 1]; }
    void apply(int code, int sign) {
        int x, y, w, h;
        dims(code, x, y, w, h);
        for (int t : reach_of(T, x, y, w, h)) cnt[t] = (uint8_t)(cnt[t] + sign);
        for (int yy = y; yy < y + h; yy++)
            for (int xx = x; xx < x + w; xx++) occ[yy * 32 + xx] = sign > 0;
    }
    int count_in_reach(int x, int y, int w, int h, int want) const {  // tiles of the reach whose cover count equals `want`
        int n = 0;
        for (int t : reach_of(T, x, y, w, h)) n += (needs(t >> 5, t & 31) && cnt[t] == want);
        return n;
    }
    bool overlaps(int x, int y, int w, int h) const {
        for (int yy = y; yy < y + h; yy++)
            for (int xx = x; xx < x + w; xx++)
                if (yy >= 0 && yy < 32 && xx >= 0 && xx < 32 && occ[yy * 32 + xx]) return true;
        return false;
    }

    int remove_min_loss(const uint32_t* hl, int exclude) {
        uint32_t best_key = 0xffffffffu;
        int best_i = 0;
        for (int i = 0; i < c.k; i++) {
            int code = c.items[i], x, y, w, h;
            dims(code, x, y, w, h);
            if (code == exclude && c.k > 1) continue;  // the placement added in the previous step is not removed again
            uint32_t key = ((uint32_t)count_in_reach(x, y, w, h, 1) << 16) | tie_remove_hl(hl[i & 31], (uint32_t)(i >> 5));
            if (key < best_key) { best_key = key; best_i = i; }
        }
        int code = c.items[best_i];
        c.items[best_i] = c.items[c.k - 1];
        c.items.pop_back();
        c.k--;
        apply(code, -1);
        return code;
    }

    void run(long long steps, int epoch_bound, int target, int noise_pct) {
        if (c.done) return;
        if (target >= 0 && epoch_bound <= target) return;  // a layout within the target is already known: the epoch does nothing
        std::memset(cnt, 0, sizeof cnt);
        if (occ0) std::memcpy(occ, occ0, sizeof occ);
        else std::memset(occ, 0, sizeof occ);
        int Wt = 0, cmin = costs[0];
        for (int i = 1; i < n_keys; i++) cmin = std::min(cmin, costs[i]);
        for (int i = 0; i < c.k; i++) { apply(c.items[i], +1); Wt += costs[c.items[i] >> 10]; }
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
                continue;
            }
            uint32_t rowmask = 0;
            for (int y = 0; y < 32; y++)
                for (int x = 0; x < 32; x++)
                    if (needs(y, x) && cnt[y * 32 + x] == 0) rowmask |= 1u << y;
            if (!rowmask) {
                c.best = Wt;
                c.best_items = c.items;
                c.best_k = c.k;
                if (Wt <= target || c.k == 0) { c.done = 1; it++; c.step++; break; }
                continue;
            }
            if (Wt + cmin >= limit && c.k > 0) {
                scored += (uint64_t)c.k;
                c.tabu_add = remove_min_loss(hl, c.tabu_rem);
                Wt -= costs[c.tabu_add >> 10];
                rowmask = 0;
                for (int y = 0; y < 32; y++)
                    for (int x = 0; x < 32; x++)
                        if (needs(y, x) && cnt[y * 32 + x] == 0) rowmask |= 1u << y;
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
                for (int l = 0; l < 32; l++) {  // the kernel's 32 lanes, lowest lane wins ties
                    const uint32_t r = lane_hash(hl[l], (uint32_t)(pass + 40));
                    const uint32_t u = r & 0xffffu;  // pass 0: uniform key; pass 1: squared draw over the keys sorted by area (largest first)
                    const int key = pass == 0 ? (int)((u * (uint32_t)n_keys) >> 16) : order[(((u * u) >> 16) * (uint32_t)n_keys) >> 16];
                    const int w = keys[2 * key], h = keys[2 * key + 1];
                    const int x = tx - 3 - (w - 1) + (int)((((r >> 16) & 0xffu) * (uint32_t)(w + 6)) >> 8);
                    const int y = ty - 3 - (h - 1) + (int)(((r >> 24) * (uint32_t)(h + 6)) >> 8);
                    const bool inb = x >= box[0] && y >= box[1] && x + w <= box[2] && y + h <= box[3];
                    if (!inb) continue;
                    n_inb++;
                    const int code = (key << 10) | (y << 5) | x;
                    const int g = count_in_reach(x, y, w, h, 0), cost = costs[key];
                    const bool ok = !overlaps(x, y, w, h) && g > 0 && code != c.tabu_add && Wt + cost < limit;
                    if (!ok) continue;
                    const uint32_t rank = cost == 1 ? (uint32_t)g : ((uint32_t)g * 64u) / (uint32_t)cost;
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
            c.tabu_rem = best_code;
        }
        steps_done += (uint64_t)it;
    }
};

}  // namespace

extern "C" {

// WINDOW mode of the same step rule (csrc/sls_multi.cu sls_multi_kernel<false, true>, driven by csrc/lns_placements.cu):
// `terrain` = the window's ceiling u8[32*32] (reach is derived from it), `need` the tiles still to be covered, `occ` the frozen
// footprints, `box` = (x0, y0, x1, y1) the additions must lie in.  Every chain starts from the same placements `items`
// (window-local codes) with best = `best` and step = `step`, and runs ONE epoch of `steps` steps without a bound or target.
// Outputs per chain: best_items u16[1024], best_k, best; totals[2] += candidates scored, steps executed.
int tsso_slsm_window_model(const uint8_t* terrain, const uint8_t* need, const uint8_t* occ, const int* box, const int* keys, const int* costs, int n_keys,
                           int n_chains, uint32_t chain_offset, uint64_t seed, int noise_pct, long long steps, const uint16_t* items, int n_items,
                           int best, uint32_t step, uint16_t* out_best_items, int* out_best_k, int* out_best, uint64_t* totals) {
    if (n_keys < 1 || n_keys > 16 || n_items < 0 || n_items > MAX_ITEMS) return -1;
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
        Runner r(T, keys, costs, n_keys, c, chain_base(seed, chain_offset + (uint32_t)i));
        r.need = need;
        r.occ0 = occ;
        for (int j = 0; j < 4; j++) r.box[j] = box[j];
        r.run(steps, NO_BOUND, -1, noise_pct);
        totals[0] += r.scored;
        totals[1] += r.steps_done;
        std::memset(out_best_items + (size_t)i * MAX_ITEMS, 0, sizeof(uint16_t) * MAX_ITEMS);
        std::copy(c.best_items.begin(), c.best_items.end(), out_best_items + (size_t)i * MAX_ITEMS);
        out_best_k[i] = c.best_k;
        out_best[i] = c.best;
    }
    return 0;
}

}  // extern "C"
