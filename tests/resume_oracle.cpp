// TEST INFRASTRUCTURE ONLY -- the model the tests of continued runs and caller-written ranks check against; compiled by
// tests/resume_oracle.py into a temporary directory.  The product path never loads it.
//
// A stateful Model (Model.cs:5-116) on the built `graph` (the CSR oracle/liboracle.so returns: row_ptr, col, val, null rows
// empty) in strict IEEE double, every loop in the reference's order: `rank` starts from any vector rank0 (the constructor's,
// or one the caller wrote into the public field, Model.cs:7), `restart` is one-hot, uniform or a weighted node set, and a
// sequence of run(int) / run(double) / run() calls follows, each from whatever `rank` holds when it starts.
// Two forms of deliverRanks, as in tests/restart_oracle.cpp:
//   literal   -- the O(N^2) restart loops exactly as written (Model.cs:92-93, :96-97);
//   collapsed -- `next[r] += rank_restart * q_r` for the listed r only; a NaN or Inf rank_restart runs the literal loop for
//                that source (x * 0.0 is NaN for every node then).  Bit-identical to the literal form.
//
// Build: g++ -O2 -std=c++17 -ffp-contract=off -fno-fast-math -fPIC -shared
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <vector>

extern "C" {

// restart: m >= 1 weights w at the distinct nodes `nodes`; m == 0 the uniform restart 1/N of `new Model(graph, c)`.
// op k: kind 0 = run(int count[k]), 1 = run(double thr[k]), 2 = run() [thr = (1/double.MaxValue) * N]; count[k] > 0 bounds
// a threshold run (the reference has no bound).  iters_out[k]: deliverRanks() calls of op k.  Returns -1 on a bad argument.
int rs_run(int32_t n, const int64_t* row_ptr, const int32_t* col, const double* val, double damping, const double* rank0,
           const int32_t* nodes, const double* w, int32_t m, int32_t n_ops, const int32_t* kind, const int64_t* count,
           const double* thr, int32_t literal, double* rank_out, int64_t* iters_out) {
    if (n < 0 || m < 0 || n_ops < 0) return -1;
    for (int32_t k = 0; k < m; k++)
        if (nodes[k] < 0 || nodes[k] >= n) return -1;
    std::vector<double> rank(rank0, rank0 + n), next((size_t)n, 0.0), restart((size_t)n, 0.0);
    std::vector<int32_t> listed;
    std::vector<double> q;
    if (m == 0) {
        for (int i = 0; i < n; i++) { restart[i] = 1.0 / n; listed.push_back(i); q.push_back(1.0 / n); }
    } else {
        for (int32_t k = 0; k < m; k++) { restart[nodes[k]] = w[k]; listed.push_back(nodes[k]); q.push_back(w[k]); }
    }
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
                for (size_t k = 0; k < listed.size(); k++) next[listed[k]] += rank_restart * q[k];
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
    for (int32_t k = 0; k < n_ops; k++) {
        const int64_t d0 = delivered;
        if (kind[k] == 0) {                                     // Model.cs:68-73
            for (int64_t it = 0; it < count[k]; it++) { deliver(); update(); }
        } else {                                                // Model.cs:52-66
            const double threshold = kind[k] == 2 ? (1 / std::numeric_limits<double>::max()) * n : thr[k];
            while (true) {
                deliver();
                if (converged(threshold)) { update(); break; }
                update();
                if (count[k] > 0 && delivered - d0 >= count[k]) break;
            }
        }
        if (iters_out) iters_out[k] = delivered - d0;
    }
    if (rank_out && n) std::memcpy(rank_out, rank.data(), sizeof(double) * (size_t)n);
    return 0;
}

}  // extern "C"
