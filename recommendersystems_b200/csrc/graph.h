// graph.h -- the device-resident graph handle shared by the translation units of librwr_b200.
#pragma once

#include "common.cuh"

// Merge-path work item geometry of the batched SpMM (spmm.cu; the table is built by k_partition in iterate.cu).  One
// chunk = CHUNK_ITEMS path items (rows + nnz), so a chunk holds at most CHUNK_ITEMS non-zeros; with the <= 3 alignment
// slack of the int4 index loads its span fits the CHUNK_SPAN-entry index buffer.
constexpr int GROUP_THREADS = 128;
constexpr int CHUNK_ROUNDS = 2;                                   // int4 index loads per thread per chunk
constexpr int CHUNK_SPAN = GROUP_THREADS * 4 * CHUNK_ROUNDS;      // 1024
constexpr int CHUNK_ITEMS = CHUNK_SPAN - 4;                       // 1020
constexpr int IDX_PAD = 8;                                        // ints of slack after the index array

struct rwr_comm;

#include "ownmap.h"

struct rwr_graph {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    rwr_opts opts{};
    DevPool pool;
    ScratchPool scratch;    // reusable request-path workspaces

    int32_t n = 0;          // nodes
    int64_t e0 = 0;         // raw links
    bool built = false;

    // ---- Graph.nodes / Graph.edges (original labels, canonical (source, insertion) order)
    DevBuf<int64_t> node_id;
    DevBuf<u8> node_type;
    DevBuf<int32_t> raw_src, raw_dst;
    DevBuf<u8> raw_type;
    DevBuf<double> raw_w;
    DevBuf<u32> raw_ptr;    // [n+1]

    // ---- Graph.graph: push CSR of W in original labels (parity probe A1-A3)
    int64_t nnz = 0;
    bool compacted = false;             // false: col/src_of alias raw_dst/raw_src, row_ptr aliases raw_ptr
    DevBuf<u32> row_ptr_own;
    DevBuf<int32_t> col_own, src_of_own;
    DevBuf<double> val;                 // normalised weights [nnz]
    u32* row_ptr = nullptr;             // [n+1]
    int32_t* col = nullptr;             // [nnz]
    int32_t* src_of = nullptr;          // [nnz] source of every explicit link
    DevBuf<double> inv_orig;            // [n] original labels: common normalised weight of a uniform row, 1.0 for a
                                        //     non-uniform row, 0.0 for a dangling row
    int32_t n_dangling = 0;
    bool all_uniform = false;
    bool fr_finite = false;             // every inv and weight entry is finite: single-seed runs may push from the frontier
    u32 max_out_degree = 0, max_in_degree = 0;

    // ---- internal labelling (descending out-degree) and the pull CSR of W^T in internal labels
    bool relabelled = false;
    int32_t n_hot = 0;                  // labels [0, n_hot): degree-sorted hot nodes; beyond: clustered cold nodes
    DevBuf<int32_t> new_of_old, old_of_new;   // [n]
    int layout = RWR_LAYOUT_VALUED;
    DevBuf<u32> in_ptr;                 // [n+1]
    DevBuf<int32_t> in_src;             // [nnz + IDX_PAD] internal source ids, original-source ascending inside a row
    DevBuf<double> in_val64;            // [nnz] (valued layout)
    DevBuf<float> in_val32;             // lazily built for FP32 runs
    DevBuf<double> inv64;               // [n] internal labels
    DevBuf<float> inv32;
    DevBuf<int2> part;                  // [n_chunks + 1] merge-path start coordinates (row, nnz)
    int32_t n_chunks = 0;
    // ---- edge stream of the warp-streamed SpMV (stream.cu)
    DevBuf<int32_t> ws_src;             // [ws_tiles * WS_TILE] source label | bit 31 on the last link of a row
    DevBuf<double> ws_val64;            // valued layout
    DevBuf<float> ws_val32;             // lazily built for FP32 runs
    DevBuf<u32> ws_tile;                // [ws_tiles + 1]
    int32_t ws_tiles = 0;
    int32_t ws_tile_links = 0;          // links per tile of this graph's stream (WS_TILE, or WS_TILE_SMALL for small graphs)
    int64_t ws_nnz = 0;                 // nnz + one padding link per row without in-links
    // column blocking of x (experimental, RWR_X_BLOCKS): the stream holds x_blocks streams back to back, block b with the
    // links whose source label lies in [b * x_block_size, (b + 1) * x_block_size), over v_rows virtual rows each
    int32_t x_blocks = 1;
    int32_t x_block_size = 0;
    int32_t v_rows = 0;                 // rows of this rank (= row_end - row_begin)
    // slice-aligned compact column blocks of a partitioned graph (stream.cu: overlapped exchange): block k of the stream
    // holds the links whose source belongs to rank (rank - k) mod P, only the non-empty (row, block) pairs are stored
    bool ws_compact = false;
    int32_t v_compact = 0;              // non-empty (row, block) pairs == virtual rows of the stream
    DevBuf<u32> vrow_ptr, vpair;        // CSR over the rank's rows: the virtual rows (compact numbers) of a row, block order
    int32_t blk_first_tile[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // tile that holds the first link of stream block k
    DevBuf<int64_t> node_id_int;        // [n] internal labels (top-k)
    DevBuf<u8> node_type_int;
    DevBuf<int32_t> items_by_id_desc;   // lazily: internal indices of ITEM nodes, id descending (full ranking)
    int32_t n_items = 0;

    // ---- hold-out state (N2, experiment.cu): test users (original labels) and their held-out tweet ids
    std::vector<int32_t> held_users;
    std::vector<int64_t> held_ptr;      // [held_users + 1]
    std::vector<int64_t> held_ids;      // node ids, ascending per user
    // ---- node id -> internal label lookup for the evaluation (N1, select.cu): ids in unsigned order, lazily built
    DevBuf<u64> ids_sorted;
    DevBuf<u32> label_of_sorted;

    // ---- row-partitioned mode
    // part_build: every rank holds the raw links and the push CSR of the sources it owns (OwnMap) only; degrees, labels and
    // per-node arrays are made global with allReduces, the transpose is an all-to-all keyed by the owner of the target row.
    // false on a partitioned handle only for the RWR_FAKE_COMM probe (one slice cut out of a whole graph on one GPU).
    bool part_build = false;
    OwnMap own;
    int64_t nnz_global = 0, e0_global = 0;  // whole-graph counts of a part_build handle (nnz / e0 are this rank's)
    int64_t nnz_in = 0;                     // links in the pull arrays (in_src): nnz, or the links received by the transpose
    DevBuf<u32> deg_all;                    // [n] explicit out-degree of every node (global), part_build only
    rwr_comm* comm = nullptr;
    int32_t row_begin = 0, row_end = 0;   // internal rows of W^T owned by this rank
    std::vector<int> part_rows;           // [n_ranks + 1] first row of every rank's slice
    std::vector<int> part_hot;            // [n_ranks] hot (degree-sorted, dealt one by one) nodes at the head of every slice
    std::vector<int> deal_rows;           // [n_ranks + 1] first label the deal gave to every slice; part_rows is deal_rows rounded
                                          // down to a multiple of 32 (a 128-byte line of x never spans two owners)
    // hub table of a partitioned graph: the part_hub_seg hottest labels of every slice, slice after slice; the edge stream
    // stores hub sources as their table slot and every other source as label + part_hub (stream.cu: HubMap)
    int32_t part_hub = 0, part_hub_seg = 0;
    // gather vectors of a partitioned graph live in two persistent buffers that every peer maps through CUDA IPC: the
    // epilogue kernel stores a rank's slice of the next x straight into the peers' copies over NVLink (dist.cu)
    bool p2p = false;
    void* px[2] = {nullptr, nullptr};     // (n + 8) * 8 bytes each, cudaMalloc
    std::vector<void*> peer_px[2];        // [n_ranks] the same buffers of every rank (own entry = px[b])
    // overlapped exchange (dist.cu, stream.cu): the next k_spmv_ws pushes this rank's slice to the peers while it gathers;
    // psync is the peer-mapped page of arrival tags
    bool overlap = false;
    void* psync = nullptr;                // DistSync, cudaMalloc, mapped by every peer
    std::vector<void*> peer_psync;        // [n_ranks]
    unsigned* push_done = nullptr;        // [8] per-peer CTA counters of the push warps
    uint64_t xtag = 0;                    // tag of the last slice produced (monotone over the life of the handle)

    // fixed-count runs replay a captured CUDA graph of their n_iter x (k_spmv_ws, k_cutrows_ws, k_finish_ws) launches: small
    // graphs (the reference's ego networks are a few thousand nodes) are launch-bound otherwise.  One per precision.
    struct IterGraph {
        cudaGraphExec_t exec = nullptr;
        bool seen = false;              // the key below was used by a direct run; the next identical run captures
        int n_iter = 0, hub = 0;
        double c = 0.0;
        u64 fr_budget = 0;              // links per sparse iteration (0: no frontier kernels in the graph)
        int64_t launches = 0;           // kernels one replay stands for
        const void* ptr[9] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    } iter_graph[2];
    float build_ms = 0.f, synth_ms = 0.f;
    int sm_count = 148;
    int max_smem_optin = 0;
};

// graph.cu
void graph_init_device(rwr_graph* g, const rwr_opts* opts);
void graph_finish_create(rwr_graph* g);          // canonicalise raw links on the device (sort by source if needed)
// iterate.cu
void iterate_prepare(rwr_graph* g);              // partition table, hub sizing
