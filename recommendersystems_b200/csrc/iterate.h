// iterate.h -- run state shared by iterate.cu (power iteration) and select.cu (top-k / ranking).
#pragma once

#include "graph.h"

struct IterCtl {
    double S;          // restart mass of the iteration being computed: sum_{non-dangling}(r - fl((1-c) r)) + sum_{dangling} r
    double resid;      // last L1 residual sum |r - y|  (Model.cs:110-115)
    int done;          // threshold mode: converged, later launches are no-ops
    int iters;         // deliverRanks() calls performed
    unsigned ticket;
    int seed;           // internal label of the seed, -1: uniform restart.  Read by k_finish_ws from here, not from its
                        // launch parameters, so that a captured iteration graph can be replayed for any seed
    unsigned tile_ctr;  // k_spmv_ws: next tile to hand out (reset by k_finish_ws)
    double red[2];     // row-partitioned graphs: this rank's {restart mass, residual} partials, summed over the ranks in place
    int fault;         // k_spmv_ws gave up waiting for a peer's slice (exchange timeout): the run is void
    unsigned long long wait_clk;   // probe (RWR_XCHG_TRACE): cycles the warps of k_spmv_ws spent waiting for slices, summed
    int sparse;         // the run may still push from its frontier (frontier.cu); cleared for good once it goes dense
    int sparse_iters;   // iterations done by the frontier kernels: the dense kernels of iteration `it` return when it < this
};

struct rwr_result {
    rwr_graph* g = nullptr;            // the caller keeps the graph alive while results exist
    int device = 0;
    int32_t n_seeds = 0;
    int32_t precision = RWR_FP64;
    std::vector<int32_t> seeds;        // original labels (-1: uniform restart)
    std::vector<int32_t> restart_nodes; // restart-set run (rwr_run_*_restart): the listed nodes, original labels; else empty
    std::vector<double> restart_weights; // their weights (a continuation rebuilds the restart set from both)
    double c = 0.0;                    // damping of the run
    std::vector<int32_t> iters;        // per slot: deliverRanks() calls since the constructor state or the last written rank
    std::vector<char> written;         // per slot: the rank was written by the caller (rwr_set_rank) since the last run from
                                       // the constructor state
    // per slot, the state a continuation starts from besides the rank: the restart mass S the next iteration adds
    // (IterCtl.S) and the iterations the frontier kernels did (IterCtl.sparse_iters), copied on the device after each run
    DevBuf<double> s_keep;
    DevBuf<int32_t> sparse_keep;
    double residual = 0.0;
    float iterate_ms = 0.f, total_ms = 0.f;
    int64_t launches = 0;
    // ranks, internal labels: column s occupies [s*ld, s*ld + n)
    size_t ld = 0;
    DevBuf<double> y64;
    DevBuf<float> y32;
};
