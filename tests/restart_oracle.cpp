// TEST INFRASTRUCTURE ONLY -- the restart-set model the tests of restart sets check against; compiled by
// tests/restart_oracle.py into a temporary directory.  The product path never loads it.
//
// A Model whose public `restart` (Model.cs:9) the caller overwrote with a sparse, not normalised vector q = w at m distinct
// nodes, run on the built `graph` (the CSR oracle/liboracle.so returns: row_ptr, col, val, null rows empty) in strict IEEE
// double, every loop in the reference's order (Model.cs:52-115).  The initial rank:
//   init 0  `new Model(graph, c)`            rank = 1           (Model.cs:24)
//   init 1  `new Model(graph, c, init_node)` rank = N at init_node (Model.cs:44)
//   init 2  rank = fl(N * q_i)
// Two forms of deliverRanks:
//   literal   -- the O(N^2) restart loops exactly as written (Model.cs:92-93, :96-97);
//   collapsed -- `next[r] += rank_restart * q_r` for the m listed r only, at the same point of the i-loop.  Every other
//                addend of the literal loop is `x * 0.0 == +-0.0` and `y + 0.0 == y`, so both forms are bit-identical while
//                x is finite; a NaN or Inf x makes `x * 0.0` NaN for EVERY node, and the collapsed form then runs the
//                literal loop for that source (as oracle/rwr_oracle.cpp does for one seed).  O(E + N m) per iteration.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -fno-fast-math -fPIC -shared
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

extern "C" {

// mode 0 = run(int n_iter), 1 = run(double thr), 2 = run() [thr = (1/double.MaxValue) * N].  max_iter > 0 bounds a
// threshold run (the reference has no bound): returns 1 when it was hit, 0 otherwise, -1 on a bad argument.
int ro_run(int32_t n, const int64_t* row_ptr, const int32_t* col, const double* val, double damping, int32_t init,
           int32_t init_node, const int32_t* nodes, const double* w, int32_t m, int32_t mode, int32_t n_iter, double thr,
           int32_t literal, int64_t max_iter, double* rank_out, int64_t* iters_out) {
    if (n < 0 || m < 1 || init < 0 || init > 2 || (init == 1 && (init_node < 0 || init_node >= n))) return -1;
    for (int32_t k = 0; k < m; k++)
        if (nodes[k] < 0 || nodes[k] >= n) return -1;
    std::vector<double> rank((size_t)n, 0.0), next((size_t)n, 0.0), restart((size_t)n, 0.0);
    for (int32_t k = 0; k < m; k++) restart[nodes[k]] = w[k];
    for (int i = 0; i < n; i++)
        rank[i] = init == 0 ? 1.0 : (init == 1 ? (i == init_node ? (double)n : 0.0) : (double)n * restart[i]);
    int64_t delivered = 0;
    auto deliver = [&]() {                                      // Model.cs:76-100
        delivered++;
        for (int i = 0; i < n; i++) {
            const int64_t b = row_ptr[i], e = row_ptr[i + 1];
            double rank_restart;
            if (e > b) {
                const double rank_randomWalk = (1 - damping) * rank[i];         // :84
                for (int64_t l = b; l < e; l++) next[col[l]] += rank_randomWalk * val[l];   // :87
                rank_restart = rank[i] - rank_randomWalk;                       // :91
            } else {
                rank_restart = rank[i];                                         // :96-97
            }
            if (!literal && std::isfinite(rank_restart)) {
                for (int32_t k = 0; k < m; k++) next[nodes[k]] += rank_restart * w[k];
            } else {
                for (int r = 0; r < n; r++) next[r] += rank_restart * restart[r];   // :93 / :97
            }
        }
    };
    auto update = [&]() {                                       // Model.cs:103-108
        for (int i = 0; i < n; i++) { rank[i] = next[i]; next[i] = 0; }
    };
    auto converged = [&](double threshold) {                    // Model.cs:110-115
        double diff = 0;
        for (int i = 0; i < n; i++) diff += (rank[i] > next[i]) ? (rank[i] - next[i]) : (next[i] - rank[i]);
        return diff < threshold;
    };
    int rc = 0;
    if (mode == 0) {                                            // Model.cs:68-73
        for (int it = 0; it < n_iter; it++) { deliver(); update(); }
    } else {                                                    // Model.cs:52-66
        const double threshold = mode == 2 ? (1 / std::numeric_limits<double>::max()) * n : thr;
        while (true) {
            deliver();
            if (converged(threshold)) { update(); break; }
            update();
            if (max_iter > 0 && delivered >= max_iter) { rc = 1; break; }
        }
    }
    if (rank_out && n) std::memcpy(rank_out, rank.data(), sizeof(double) * (size_t)n);
    if (iters_out) *iters_out = delivered;
    return rc;
}

}  // extern "C"
