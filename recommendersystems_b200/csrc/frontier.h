// frontier.h -- the sparse prefix of a single-seed run (frontier.cu): the first iterations pushed from the seed's frontier.
#pragma once

#include "graph.h"

template <typename T> struct IterParams;

// iterations that may run sparsely (their frontier kernels are launched before the dense ones).  On C2 the third is
// always dense, and its attempt -- the frontier of up to 175 k rows, the scan of their degrees, 13 no-op launches --
// cost 0.05 ms per run (profiles/r03_frontier_probe_k3.txt).
constexpr int FR_ITERS = 2;
// Graphs with fewer links stay dense unless RWR_FRONTIER_BUDGET is set.  20-iteration run on smaller graphs of the C2
// generator (profiles/r03_frontier_probe.txt): the sparse prefix is slower at 0.9 / 3.9 / 9.7 M links, even at 19.8 M,
// 2.5 % faster at 32 M and 5.6 % at 61 M -- two sparse iterations cost ~0.1 ms, mostly launches.
constexpr int64_t FR_MIN_LINKS = 32 << 20;

// Device workspace of the sparse prefix, carved out of one scratch block (RunWorkspace::alloc).
struct FrontierWs {
    u64 budget = 0;        // push links per sparse iteration; 0: the run stays dense
    size_t cap = 0;        // expanded entries: budget + 1 (the seed's zero entry)
    u32 words = 0;         // frontier bitmap words over the original labels
    int g_words = 0, g_scan_f = 0, g_exp = 0, t_max = 0, g_scan_t = 0, g_sum = 0, passes = 0;
    u32* sc = nullptr;     // [4] frontier size, expanded entries, radix table length
    u32* bits = nullptr;   // [words] next frontier (original labels); all zero between iterations
    u32* fid = nullptr;    // [budget + 2] frontier, original labels ascending
    u32* fdeg = nullptr;   // [budget + 2] their out-degrees
    u32* foff = nullptr;   // [budget + 2] exclusive prefix of fdeg (foff[nf] = push links)
    u32* bsum = nullptr;   // block sums of the scans
    u32* table = nullptr;  // [256 * t_max] radix digit table
    u32* key[2] = {nullptr, nullptr};       // [cap] target labels (sort ping-pong)
    void* val[2] = {nullptr, nullptr};      // [cap] products
};

// links per sparse iteration for this graph and run (0: no sparse path).  Reads RWR_NO_FRONTIER and
// RWR_FRONTIER_BUDGET on every call.
u64 frontier_budget(const rwr_graph* g);
// the layout of the workspace for `budget` inside `base` (null: sizes only); returns its bytes
size_t frontier_carve(const rwr_graph* g, u64 budget, size_t elt, void* base, FrontierWs& fw);
// graph build: records whether every weight and inv entry is finite (NaN / Inf graphs never run sparsely)
void frontier_prepare(rwr_graph* g);
// one sparse iteration (a no-op on the device once the run has gone dense); emit: build the next frontier.  Returns the
// number of kernels launched (also added to g->pool.launches).
template <typename T>
int frontier_launch(rwr_graph* g, const FrontierWs& fw, const IterParams<T>& p, bool emit);
