// stream.h -- the flagged edge stream of the warp-streamed SpMV (stream.cu): geometry and host entry points.
#pragma once

#include "graph.h"

constexpr int WS_WARPS = 16;                     // independent warps per CTA, one CTA per SM
constexpr int WS_THREADS = WS_WARPS * 32;        // 512
constexpr int WS_STEP = 128;                     // links per warp step: one int4 of indices per lane
constexpr int WS_R = 2;                          // rounds per pipeline stage
constexpr int WS_STAGE = WS_R * WS_STEP;         // 256 links per stage
constexpr int WS_TILE = 4096;                    // links per tile (unit of work distribution and of the fix-up)
constexpr int WS_TILE_SMALL = 512;               // tile size of graphs with fewer than WS_SMALL_GRAPH_LINKS links
constexpr int WS_TILE_MEDIUM = 1024;             // ... with fewer than WS_MEDIUM_GRAPH_LINKS links
constexpr int WS_SMALL_GRAPH_LINKS = 8 << 20;
constexpr int WS_MEDIUM_GRAPH_LINKS = 48 << 20;
constexpr int WS_SPT = WS_TILE / WS_STAGE;
static_assert(WS_TILE_SMALL % (2 * WS_STAGE) == 0 && WS_TILE_MEDIUM % (2 * WS_STAGE) == 0 && WS_TILE % (2 * WS_STAGE) == 0,
              "a tile is an even number of stages");       // 32 stages per tile
constexpr int WS_HDR = 128;                      // mbarrier, ahead of the hub table
constexpr int FIN_THREADS = 256;
constexpr size_t WS_HUB_AUTO_BYTES = 99 * 1024;         // automatic hub size, FP64: fits the 100 KB carve-out step with the 1 KB the system reserves
constexpr size_t WS_HUB_AUTO_BYTES_FP32 = 163 * 1024;   // same, FP32: the 164 KB step
static_assert(WS_R == 2, "ws_consume is written for two rounds (8 links per lane) per stage");

template <typename T> struct IterParams;
struct RestartSet;

void stream_prepare(rwr_graph* g);               // builds ws_src / ws_val64 / ws_tile from the pull CSR
int ws_hub_entries(const rwr_graph* g, int precision);
int ws_main_grid(const rwr_graph* g);
int ws_fix_grid(const rwr_graph* g);
int ws_fin_grid(const rwr_graph* g);
// one iteration = k_spmv_ws (row sums) + k_cutrows_ws (rows cut by a tile boundary) + k_finish_ws (fused epilogue); a
// restart-set run (rs) gets the epilogue k_finish_set_ws
template <typename T>
void ws_launch_iteration(rwr_graph* g, const IterParams<T>& p, bool resid, double thr, int use_thr, const RestartSet* rs = nullptr);
template <typename T> void ws_launch_spmv_only(rwr_graph* g, const IterParams<T>& p);
template <typename T>
void ws_launch_finish_only(rwr_graph* g, const IterParams<T>& p, bool resid, double thr, int use_thr, const RestartSet* rs = nullptr);
