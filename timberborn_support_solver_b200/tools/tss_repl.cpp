// tss_repl — `load <project.toml>; solve [-l k:v,...]` of the reference's REPL (crates/repl/src/main.rs:248-261,280-366) as a
// plain C++ program over the C ABI of libtss (include/tss.h): the bound-tightening loop with the GPU engine behind the
// solver interface and an optional external exact solver for what the GPU cannot answer.
//
// Every iteration performs EXACTLY the call sequence of the Rust shim's `add_cnf` + `solve` (rust/tss/src/lib.rs):
//     tss_encoding_with_limits            Encoding::with_limits + into_cnf            (main.rs:292-293)
//     tss_cnf_upload, tss_instance_find   Solve::add_cnf: the solver sees only the clauses and finds its instance again
//     tss_solve_instance                  Solve::solve: SAT-like GPU search, witness verified against those clauses
//     [exact solver on the same clauses]  only when the GPU has no answer and the lower bound has not closed the gap
//     tss_layout_from_assignment          PlatformLayout::from_assignment             (main.rs:328-329)
//     tss_validate                        layout.validate (warn only)                 (main.rs:353-361)
// and prints what the REPL prints (main.rs:331-352).  UNSAT comes from the exact solver (`--exact CMD`, any DIMACS solver that
// prints `s SATISFIABLE|UNSATISFIABLE` and `v ...` lines, e.g. `z3 -dimacs`, glucose, kissat) or from tss_solve_instance when the
// limit lies below a certified lower bound of the instance (packing / fractional LP); a search that finds nothing proves nothing.
//
// `--limit-bounds` lets tss_solve_instance certify the UNSAT of a `-l` loop with the class-aware LP, which keeps the per-type
// limits (tss_engine_limit_bounds); `--no-lower-bound` switches every bound off, this one included.
//
// `--window-limits` lets tss_solve_instance answer `-l` instances on grids larger than 32x32 with the window placement search
// (tss_engine_window_limits); it finds layouts, it proves nothing, so without `--exact` such a loop ends "unknown".
//
// `--gui` runs the GUI's loop instead (crates/gui/src/app.rs:212-249): the default-8 set with the GUI's default weights
// (app.rs:53-62), no card limits; after every solution limits.weight_limit = total_weight - 1 (while that is positive), until
// the solver says Unsat — the weight limit's pseudo-boolean constraint is part of the clauses the witness is checked against.
//
//   tss_repl PROJECT.toml [--platforms default|1x1] [-l k:v[,k:v]] [--gui] [--exact "CMD"] [--seed N] [--no-lower-bound] [--limit-bounds] [--window-limits] [--quiet] [--repeat N] [--phases]
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/tss.h"

namespace {

double now_ms() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// `-l` arguments: k is N (-> NxN) or AxB, resolved to a canonical def (w <= h) (main.rs:120-142, 85-101)
bool parse_limits(const std::string& arg, std::vector<int32_t>& card) {
    std::stringstream ss(arg);
    std::string item;
    while (std::getline(ss, item, ',')) {
        const size_t colon = item.find(':');
        if (colon == std::string::npos) return false;
        const std::string k = item.substr(0, colon);
        int a = 0, b = 0;
        const size_t x = k.find('x');
        if (x == std::string::npos) a = b = std::atoi(k.c_str());
        else { a = std::atoi(k.substr(0, x).c_str()); b = std::atoi(k.substr(x + 1).c_str()); }
        if (a <= 0 || b <= 0) return false;
        card.push_back(a < b ? a : b);
        card.push_back(a < b ? b : a);
        card.push_back(std::atoi(item.substr(colon + 1).c_str()));
    }
    return true;
}

// runs an external DIMACS solver on the clauses; returns 10 / 20 / 0 and fills the assignment (u8[n_vars + 1])
int run_exact(const std::string& cmd, const std::vector<int32_t>& lits, const std::vector<uint32_t>& offsets, int n_vars, std::vector<uint8_t>& assignment) {
    char path[] = "/tmp/tss_repl_XXXXXX";
    const int fd = mkstemp(path);
    if (fd < 0) return 0;
    FILE* f = fdopen(fd, "w");
    std::fprintf(f, "p cnf %d %zu\n", n_vars, offsets.size() - 1);
    for (size_t c = 0; c + 1 < offsets.size(); c++) {
        for (uint32_t k = offsets[c]; k < offsets[c + 1]; k++) std::fprintf(f, "%d ", lits[k]);
        std::fprintf(f, "0\n");
    }
    std::fclose(f);
    FILE* p = popen((cmd + " " + path + " 2>/dev/null").c_str(), "r");
    int result = 0;
    if (p) {
        assignment.assign((size_t)n_vars + 1, 0);
        assignment[0] = 2;
        char* line = nullptr;
        size_t cap = 0;
        while (getline(&line, &cap, p) > 0) {
            if (!std::strncmp(line, "s SATISFIABLE", 13) || !std::strncmp(line, "sat", 3)) result = 10;
            else if (!std::strncmp(line, "s UNSATISFIABLE", 15) || !std::strncmp(line, "unsat", 5)) result = 20;
            else if (line[0] == 'v') {
                std::stringstream ss(line + 1);
                long v;
                while (ss >> v)
                    if (v != 0 && std::labs(v) <= n_vars) assignment[(size_t)std::labs(v)] = v > 0;
            }
        }
        std::free(line);
        pclose(p);
    }
    std::remove(path);
    return result;
}

}  // namespace

int main(int argc, char** argv) {
    std::string project, exact_cmd, platforms = "default";
    std::vector<int32_t> card;
    uint64_t seed = 0;
    bool use_lb = true, limit_lb = false, window_limits = false, quiet = false, phases = false, gui = false;
    int repeat = 1;
    double ph[8] = {};   // --phases: wall ms per call site, summed over the warm repeats
    static const char* const PH[8] = {"encoding_create", "with_limits", "cnf_upload", "instance_find", "solve_instance", "from_assignment", "validate", "destroy"};
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        if (a == "--platforms" && i + 1 < argc) platforms = argv[++i];
        else if (a == "--exact" && i + 1 < argc) exact_cmd = argv[++i];
        else if (a == "--seed" && i + 1 < argc) seed = std::strtoull(argv[++i], nullptr, 10);
        else if (a == "-l" && i + 1 < argc) { if (!parse_limits(argv[++i], card)) { std::fprintf(stderr, "bad -l argument\n"); return 2; } }
        else if (a.rfind("-l", 0) == 0 && a.size() > 2) { if (!parse_limits(a.substr(2), card)) { std::fprintf(stderr, "bad -l argument\n"); return 2; } }
        else if (a == "--no-lower-bound") use_lb = false;
        else if (a == "--limit-bounds") limit_lb = true;
        else if (a == "--window-limits") window_limits = true;
        else if (a == "--quiet") quiet = true;
        else if (a == "--phases") phases = true;
        else if (a == "--gui") gui = true;
        else if (a == "--repeat" && i + 1 < argc) repeat = std::atoi(argv[++i]) > 0 ? std::atoi(argv[i]) : 1;
        else if (project.empty()) project = a;
        else { std::fprintf(stderr, "usage: tss_repl PROJECT.toml [--platforms default|1x1] [-l k:v[,k:v]] [--exact CMD] [--seed N] [--no-lower-bound] [--limit-bounds] [--window-limits] [--quiet]\n"); return 2; }
    }
    if (project.empty()) { std::fprintf(stderr, "no project file\n"); return 2; }
    std::ifstream in(project);
    if (!in) { std::fprintf(stderr, "Error reading file %s\n", project.c_str()); return 1; }
    std::stringstream buf;
    buf << in.rdbuf();
    std::vector<uint8_t> grid(1 << 20);
    int32_t w = 0, h = 0, ragged = 0;
    char err[256] = "";
    if (tss_world_parse_toml(buf.str().c_str(), grid.data(), grid.size(), &w, &h, &ragged, err, sizeof err) != TSS_OK) {
        std::fprintf(stderr, "Error parsing file: %s\n", err);
        return 1;
    }
    grid.resize((size_t)w * h);
    // PLATFORMS_DEFAULT (src/platform.rs:23-32), what the REPL solves with (main.rs:254)
    const tss_dims all_defs[8] = {{1, 1}, {1, 2}, {1, 3}, {1, 4}, {1, 5}, {1, 6}, {3, 3}, {5, 5}};
    const int n_defs = platforms == "1x1" && !gui ? 1 : 8;
    // DEFAULT_PLATFORMS of the GUI (crates/gui/src/app.rs:53-62): records (def_w, def_h, weight)
    const int32_t gui_weights[24] = {1, 1, 5, 1, 2, 1, 1, 3, 1, 1, 4, 1, 1, 5, 1, 1, 6, 1, 3, 3, 2, 5, 5, 4};
    const int32_t* wts = gui ? gui_weights : nullptr;
    const int32_t n_wts = gui ? 8 : 0;
    long long best_weight = -1;
    const double t_start = now_ms();

    tss_engine* e = nullptr;
    if (tss_engine_create(-1, &e) != TSS_OK) { std::fprintf(stderr, "no usable CUDA device (the GPU path has no CPU fallback)\n"); return 1; }
    const double t_setup = now_ms();
    // --repeat N: the whole `solve` N times in this process (fresh encoding, limits and bounds each time; the engine and its
    // cached workspaces stay), printing only the first: the loop's warm timing without process start-up
    const std::vector<int32_t> card0 = card;
    std::vector<double> loop_ms;
    int32_t lower = -1;
    int gpu_solves = 0, exact_solves = 0, best = -1;
    std::string verdict = "open";
    double t_loop = now_ms();
    for (int rep = 0; rep < repeat; rep++) {
        const bool say = rep == 0;
#define SAY(...) do { if (say) std::printf(__VA_ARGS__); } while (0)
        card = card0;
        lower = -1; gpu_solves = exact_solves = 0; best = -1; verdict = "open";
        int32_t has_wl = 0;
        int64_t wl = 0;
        best_weight = -1;
        t_loop = now_ms();   // one `solve`: encode, bounds, loop (engine creation = CUDA context start-up, ~1-4 s of a fresh process, is reported apart)
        tss_encoding* enc = nullptr;
        double tp = now_ms();
#define PHASE(i) do { const double t_ = now_ms(); if (rep > 0) ph[i] += t_ - tp; tp = t_; } while (0)
        if (tss_encoding_create(grid.data(), w, h, all_defs, n_defs, &enc) != TSS_OK) { std::fprintf(stderr, "encode failed\n"); return 1; }
        PHASE(0);
        int32_t K = 0;
        tss_encoding_sizes(enc, nullptr, nullptr, nullptr, &K);

        // the certified lower bounds live behind tss_solve_instance (it answers TSS_UNSAT below them), exactly where the Rust shim's
        // solve() sees them: this driver, like the REPL's, knows nothing about bounds
        tss_engine_certified_unsat(e, use_lb ? 1 : 0);
        tss_engine_limit_bounds(e, use_lb && limit_lb ? 1 : 0);
        tss_engine_window_limits(e, window_limits ? 1 : 0);

        int64_t give_up = 1024;
        for (;;) {
            int32_t n_vars = 0, n_clauses = 0;
            int64_t n_lits = 0;
            tss_encoding_with_limits(enc, card.data(), (int32_t)card.size() / 3, wts, n_wts, has_wl, wl, &n_vars, &n_clauses, &n_lits, nullptr, nullptr);
            std::vector<int32_t> lits((size_t)n_lits + 1);
            std::vector<uint32_t> offsets((size_t)n_clauses + 1);
            tss_encoding_with_limits(enc, card.data(), (int32_t)card.size() / 3, wts, n_wts, has_wl, wl, &n_vars, &n_clauses, &n_lits, lits.data(), offsets.data());
            lits.resize((size_t)n_lits);
            PHASE(1);

            // ---- Solve::add_cnf: all the solver is given are the clauses
            tss_cnf* cnf = nullptr;
            if (tss_cnf_upload(e, lits.data(), offsets.data(), n_clauses, n_vars, &cnf) != TSS_OK) { std::fprintf(stderr, "%s\n", tss_last_error(e)); return 1; }
            PHASE(2);
            tss_encoding* inst = nullptr;
            tss_instance_info info;
            int32_t found_weights[3 * 16];   // the PlatformLimits.weights map, handed back by the registry like the rest of the instance
            const int found = tss_instance_find(lits.data(), offsets.data(), n_clauses, n_vars, &inst, &info, found_weights, 16);

            PHASE(3);
            // ---- Solve::solve
            std::vector<uint8_t> assignment((size_t)n_vars + 1, 2);
            int result = 0;
            std::string source = "gpu";
            if (found == TSS_SAT) {
                tss_clear_interrupt(e);
                const int rc = tss_solve_instance(e, cnf, inst, &info, info.n_weights > 0 ? found_weights : nullptr, seed++, give_up, assignment.data());
                if (rc < 0) std::fprintf(stderr, "tss_solve_instance: %s\n", tss_last_error(e));   // logged, never fatal (crates/gui/src/app.rs:160-173)
                result = rc == TSS_SAT ? 10 : rc == TSS_UNSAT ? 20 : 0;   // UNSAT: the limit lies below a certified lower bound
                gpu_solves++;
                if (result == 10) {
                    tss_stats st;
                    tss_get_stats(e, &st);
                    give_up = 32 * st.last_solve_steps > 1024 ? 32 * st.last_solve_steps : 1024;
                }
            }
            PHASE(4);
            if (result == 0 && !exact_cmd.empty()) {   // the exact solver: every UNSAT answer comes from here
                result = run_exact(exact_cmd, lits, offsets, n_vars, assignment);
                source = "exact";
                exact_solves++;
            }
            tp = now_ms();
            if (inst) tss_encoding_destroy(inst);
            tss_cnf_destroy(cnf);
            PHASE(7);
            if (result == 20) {
                SAY("No solution found for the current constraints\n");
                verdict = best < 0 ? "unsatisfiable" : source == "exact" ? "optimal (exact solver)" : "optimal (lower bound)";
                if (best >= 0 && source != "exact") lower = gui ? (int)best_weight : best;   // the certified bound that closed the loop is at least the limit it refused + 1
                break;
            }
            if (result != 10) { SAY("Solver interrupted\n"); verdict = "unknown (no exact solver answer)"; break; }

            std::vector<tss_platform> plats((size_t)w * h + 1);
            int32_t n = 0;
            tss_layout_from_assignment(enc, assignment.data(), n_vars + 1, plats.data(), (int32_t)plats.size(), &n);
            PHASE(5);
            if (n == 0) { SAY("Found a solution with no platforms - aborting\n"); verdict = "optimal (no platforms)"; best = 0; break; }
            best = n;
            bool last = false;
            if (gui) {   // app.rs:235-245: weight_limit = total_weight - 1 while that is positive
                best_weight = (long long)tss_layout_total_weight(plats.data(), n, gui_weights, 8);
                SAY("Got a solution with weight %lld\n", best_weight);
                has_wl = 1;
                wl = best_weight - 1;
                last = wl <= 0;
            } else {
                bool has = false;
                for (size_t i = 0; i < card.size(); i += 3)
                    if (card[i] == 1 && card[i + 1] == 1) { card[i + 2] = n - 1; has = true; }
                if (!has) { card.push_back(1); card.push_back(1); card.push_back(n - 1); }
            }
            SAY("Solution found (%d platforms total)\n", n);
            std::map<std::pair<int, int>, int> stats;
            for (int i = 0; i < n; i++) stats[{plats[i].def_w, plats[i].def_h}]++;
            for (auto& [d, c] : stats) SAY("%dx%d: %d\n", d.first, d.second, c);
            std::vector<uint8_t> unsupported((size_t)w * h), flags((size_t)n);
            const int uns = tss_validate(e, grid.data(), w, h, plats.data(), n, unsupported.data(), flags.data());
            PHASE(6);
            int bad = uns;
            for (int i = 0; i < n; i++) bad += flags[i] != 0;
            if (!quiet) SAY(bad == 0 ? "Solution validation OK (%s)\n" : "Solution validation FAILED (%s)\n", source.c_str());
            if (bad != 0) { verdict = "invalid layout"; break; }
            if (last) { verdict = "optimal (weight 1)"; break; }
        }
        tss_encoding_destroy(enc);
        loop_ms.push_back(now_ms() - t_loop);
    }
    std::printf("Done\n");
    std::sort(loop_ms.begin() + (loop_ms.size() > 1 ? 1 : 0), loop_ms.end());   // the first run is cold (allocations): median of the rest
    const double warm = loop_ms.size() > 1 ? loop_ms[1 + (loop_ms.size() - 1) / 2] : loop_ms[0];
    std::printf("# best=%d lower_bound=%d verdict=\"%s\" gpu_solves=%d exact_solves=%d ms=%.3f setup_ms=%.1f repeats=%zu warm_ms=%.3f weight=%lld\n", best, lower,
                verdict.c_str(), gpu_solves, exact_solves, loop_ms[0], t_setup - t_start, loop_ms.size(), warm, best_weight);
    if (phases && repeat > 1) {
        std::printf("# phases (ms per solve, mean of %d warm repeats):", repeat - 1);
        for (int i = 0; i < 8; i++) std::printf(" %s=%.3f", PH[i], ph[i] / (repeat - 1));
        std::printf("\n");
    }
    tss_engine_destroy(e);
    return 0;
}
