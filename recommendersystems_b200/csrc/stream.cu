// stream.cu -- K7: the power iteration  r <- (1-c) W^T r + S q  as a warp-streamed SpMV over a flagged edge stream.
//
// Restates the push loop of Recommenders/RWRBased/Model.cs:76-100 as a pull over W^T, with a layout and a schedule
// built around what bounds this kernel on a B200: not HBM bytes but the ~1 scattered gather per cycle per SM that the
// L1TEX path sustains (profiles/microbench/gather_bench.cu: 289 G reads/s from L2, 1500 G reads/s from shared memory),
// and the L1 capacity that holds the sectors of the gathers in flight.  Everything else is arranged so that the gather
// queue never runs dry.  One iteration = three launches:
//   k_spmv_ws     raw row sums y_t = sum_i x_i over the links of row t (x is pre-scaled: x_i = fl(fl((1-c) r_i) w_i))
//   k_cutrows_ws  the few rows cut by a tile boundary, assembled from per-tile partial sums in tile order
//   k_finish_ws   the fused per-row epilogue (restart AXPY, next x, restart-mass and L1-residual partials, their
//                 fixed-order reduction, the convergence test of Model.cs:110-115) -- streamed and coalesced
//
// Layout ("edge stream", built once per graph by stream_prepare):
//   ws_src[q]   source label of the q-th stored link of W^T, rows back to back; bit 31 set on the LAST link of a row.
//               A row without in-links gets one padding link to the always-zero entry x[n], so every row owns >= 1
//               link, row ids are implicit (count the end flags) and y / x_next of such rows are written like any other.
//               A row of more than 256 links holds its links by ascending source label (ties by pull-CSR position);
//               shorter rows keep the pull CSR's order.  A 256-link stage that holds a row end is stored lane-major
//               (a lane owns 8 consecutive links, what the segmented scan needs); a stage inside one row, without a
//               row end, is stored link-major (gather instruction (j, k) reads the 32 consecutive links j*128 + k*32 ..),
//               so that the label-sorted sources of a long row share 128-byte lines (ws_stage_link).
//   ws_val[q]   normalised weight of the link (valued layout only; the index-only layout folds the row's common
//               weight into x, see graph.cu)
//   ws_tile[t]  row of the first link of tile t | bit 31 when that row started in an earlier tile.  A tile is 4096 links
//               (1024 / 512 for graphs under 48 M / 8 M links).
//
// Schedule of k_spmv_ws: 16 independent warps per SM (20 in FP32 index-only), no block-level barrier inside the loop.
// Tiles are handed out dynamically, one atomic per tile drawn a tile ahead.  A warp walks its tile in stages of 256
// links (two coalesced int4 of indices per lane, evict-first): indices are loaded two stages ahead and the gathers of x
// one stage ahead -- one generic-address load per link, into the shared-memory hub table (the hottest sources) or L2.
// Row sums use registers and shuffles only: a stage without a row end adds into a per-lane accumulator; a stage with
// row ends runs a warp-level segmented scan with early exit, and the lanes holding a row end store the sums.  The open
// row at a tile boundary goes to tail[t] / head[t].  No floating-point atomics anywhere: a run is bit-reproducible; the
// association of a row sum differs from the reference's sequential one by O(log deg) ulp (all addends >= 0).
//
// Row-partitioned graphs (K10, dist.cu) reuse the same kernels on a rank's rows:
//   * the hub table holds the hottest labels of EVERY slice (HubMap: the stream stores table slots / shifted labels);
//   * the stream can be cut into column blocks: padded virtual rows (rwr_opts.x_blocks), or -- for the overlapped exchange --
//     compact slice-aligned blocks, block k = the links whose source belongs to rank (r - k) mod P (k_pair_*,
//     k_ws_fill_compact), added up per row by k_finish_ws<.., 2> through a CSR of (row, block) pairs;
//   * the XWAIT instantiation of k_spmv_ws has 15 gathering warps that wait, block by block, for the arrival tags of the
//     peers' slices, and one push warp (ws_push_slices) that sends this rank's slice to the peers with TMA bulk copies.
#include <algorithm>
#include <climits>
#include <cmath>

#include "iterate_dev.cuh"
#include "primitives.cuh"
#include "stream.h"
#include "dist.h"

constexpr u32 END_BIT = 0x80000000u;

#ifdef RWR_PROFILE_CLOCKS
__device__ unsigned long long g_clk_ws[16];
#define WCLK_DECL long long wclk0 = clock64(), wclk1; unsigned long long wclk[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define WCLK(slot) do { wclk1 = clock64(); wclk[slot] += (unsigned long long)(wclk1 - wclk0); wclk0 = wclk1; } while (0)
#define WCLK_FLUSH do { if (lane == 0) for (int i = 0; i < 8; i++) atomicAdd(&g_clk_ws[i], wclk[i]); } while (0)
#else
#define WCLK_DECL
#define WCLK(slot)
#define WCLK_FLUSH
#endif

// ------------------------------------------------------------------------------------------------ layout build
__global__ void k_ws_len(const u32* __restrict__ in_ptr, int n, u32* __restrict__ len) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) {
        const u32 d = in_ptr[r + 1] - in_ptr[r];
        len[r] = d ? d : 1u;
    }
}

// largest r in [0, n) with ptr2[r] <= q   (ptr2 strictly increasing: every row owns >= 1 link)
__device__ __forceinline__ int ws_row_of(const u32* __restrict__ ptr2, int n, u32 q) {
    int lo = 0, hi = n;                       // invariant: ptr2[lo] <= q < ptr2[hi]  (ptr2[n] = total > q)
    while (hi - lo > 1) {
        const int mid = (int)(((unsigned)lo + (unsigned)hi) >> 1);
        if (ptr2[mid] <= q) lo = mid; else hi = mid;
    }
    return lo;
}

// Hub table of a partitioned graph.  The label order is dealt over the slices (graph.cu: k_deal_labels), so the hottest
// sources are the first labels of EVERY slice, not one label prefix.  The stream therefore stores a source as
//   slot = s * seg_len + (label - start[s])   when it is one of the seg_len hottest labels of slice s   (slot < H)
//   label + H                                 otherwise (k_spmv_ws gets the gather vector shifted down by H entries)
// and k_spmv_ws keeps its one-compare, one-load gather.  H == 0: labels are stored as they are.
struct HubMap {
    int parts, seg_len, H;
    int start[8];
};
__device__ __forceinline__ u32 hub_translate(const HubMap& m, u32 label) {
    if (m.H == 0) return label;
    for (int s = 0; s < m.parts; s++) {
        const u32 j = label - (u32)m.start[s];
        if (j < (u32)m.seg_len) return (u32)(s * m.seg_len) + j;
    }
    return label + (u32)m.H;
}

// Link of a stage (0 .. WS_STAGE-1) that physical offset o of the stage holds.  Lane L loads the int4 at o = j*128 + L*4
// in round j, and gathers its element k with instruction (j, k).
//   lane-major: o holds link L*8 + j*4 + k -- a lane owns 8 consecutive links, which the segmented scan of a stage with
//               row ends needs;
//   link-major: o holds link j*128 + k*32 + L -- instruction (j, k) gathers 32 consecutive links, so a row sorted by
//               source label touches fewer 128-byte lines.
// The build stores a stage link-major exactly when it holds no end-of-row flag (it lies inside one row whose last link
// comes after it).  ws_consume sums such a stage on its H == 0 path, where every lane adds its own 8 values into its own
// partial and which links a lane holds does not matter; any other stage must stay lane-major.
__device__ __forceinline__ u32 ws_stage_link(u32 o, bool link_major) {
    const u32 rnd = o / WS_STEP, ln = (o % WS_STEP) / 4, k = o % 4;
    return link_major ? rnd * WS_STEP + k * 32 + ln : ln * (WS_R * 4) + rnd * 4 + k;
}

// The stream covers the links [q0, q0 + nnz2) of the whole-graph numbering (q0 > 0 for a row slice of a partitioned graph).
// A row of more than WS_STAGE links (the only rows that can hold a flag-free stage) is stored in the order of lperm:
// row i of the slice owns lperm[loff[i] ..], pull-CSR positions sorted by source label (ws_long_row_order).  Every other
// row keeps the pull CSR's order.
__global__ void k_ws_fill(const u32* __restrict__ ptr2, const u32* __restrict__ in_ptr, const int32_t* __restrict__ in_src,
                          const double* __restrict__ in_val, const u32* __restrict__ loff, const u32* __restrict__ lperm, int n,
                          int row_begin, u32 q0, u32 nnz2, size_t padded, const HubMap hm, int32_t* __restrict__ ws_src,
                          double* __restrict__ ws_val /* may be null */) {
    const size_t phys = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (phys >= padded) return;
    const u32 o = (u32)(phys % WS_STAGE);
    const size_t qs = phys - o;                   // first link of the stage
    const u32 zero_entry = (u32)n + (u32)hm.H;   // x[n] == 0
    bool link_major = false;
    int r = 0;
    if (qs < nnz2) {
        r = ws_row_of(ptr2, n, q0 + (u32)qs);
        link_major = ptr2[r + 1] > q0 + (u32)qs + WS_STAGE;      // the row's last link lies after the stage: no end flag
    }
    const size_t q = qs + ws_stage_link(o, link_major);
    if (q >= nnz2) {                          // tail padding of the last tile: zero entry, no flag
        ws_src[phys] = (int32_t)zero_entry;
        if (ws_val) ws_val[phys] = 0.0;
        return;
    }
    if (!link_major) r = ws_row_of(ptr2, n, q0 + (u32)q);
    const u32 j = q0 + (u32)q - ptr2[r];
    const u32 b = in_ptr[r], deg = in_ptr[r + 1] - b;
    if (deg == 0) {
        ws_src[phys] = (int32_t)(zero_entry | END_BIT);
        if (ws_val) ws_val[phys] = 0.0;
    } else {
        const u32 pos = deg > (u32)WS_STAGE ? lperm[loff[r - row_begin] + j] : b + j;
        ws_src[phys] = (int32_t)(hub_translate(hm, (u32)in_src[pos]) | (j == deg - 1 ? END_BIT : 0u));
        if (ws_val) ws_val[phys] = in_val[pos];
    }
}

// ---- source-label order of the long rows ------------------------------------------------------------------------------
// Rows of the slice [row_begin, row_begin + R) with more than WS_STAGE links: cnt[i] = their link count, 0 for the others.
__global__ void k_ws_long_len(const u32* __restrict__ in_ptr, int row_begin, int R, u32* __restrict__ cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < R) {
        const u32 d = in_ptr[row_begin + i + 1] - in_ptr[row_begin + i];
        cnt[i] = d > (u32)WS_STAGE ? d : 0u;
    }
}
// one warp per row: key (row, source label), value the pull-CSR position
__global__ void k_ws_long_keys(const u32* __restrict__ in_ptr, const int32_t* __restrict__ in_src, const u32* __restrict__ loff,
                               int row_begin, int R, int label_bits, u64* __restrict__ keys, u32* __restrict__ vals) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (i >= (size_t)R) return;
    const u32 b = in_ptr[row_begin + i], deg = in_ptr[row_begin + i + 1] - b;
    if (deg <= (u32)WS_STAGE) return;
    const u32 base = loff[i];
    for (u32 j = lane; j < deg; j += 32) {
        keys[base + j] = ((u64)i << label_bits) | (u64)(u32)in_src[b + j];
        vals[base + j] = b + j;
    }
}

// The pull-CSR positions of the slice's rows of more than WS_STAGE links, row after row, each row by ascending source label
// (ties by position: the sort is stable and starts from position order); loff (R + 1 entries) = where each row starts.
// Returns an empty buffer when no row is that long.
static DevBuf<u32> ws_long_row_order(rwr_graph* g, int row_begin, int R, DevBuf<u32>& loff) {
    cudaStream_t st = g->stream;
    loff.alloc((size_t)R + 1);
    k_ws_long_len<<<div_up((size_t)R, 256), 256, 0, st>>>(g->in_ptr.p, row_begin, R, loff.p);
    KERNEL_CHECK();
    const u32 m = prim::scan_total<u32>(loff.p, loff.p, (size_t)R, true, st, &g->pool);
    if (m == 0) return DevBuf<u32>();
    prim::SortBuffers<u64> sb;
    sb.alloc(m, true);
    const int label_bits = ceil_log2_u64((u64)g->n);
    k_ws_long_keys<<<div_up((size_t)R * 32, 256), 256, 0, st>>>(g->in_ptr.p, g->in_src.p, loff.p, row_begin, R, label_bits,
                                                               sb.keys(), sb.vals());
    KERNEL_CHECK();
    sb.sort(m, label_bits + ceil_log2_u64((u64)R), st, &g->pool);
    return sb.take_vals();
}

__global__ void k_ws_tiles(const u32* __restrict__ ptr2, int n, u32 q0, int row_end, int n_tiles, u32 tile_links,
                           u32* __restrict__ ws_tile) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    if (t == n_tiles) { ws_tile[t] = (u32)row_end; return; }
    const u32 q = q0 + (u32)t * tile_links;
    const int r = ws_row_of(ptr2, n, q);
    ws_tile[t] = (u32)r | (q > ptr2[r] ? END_BIT : 0u);
}

// ---- column blocking of x with virtual rows (experimental; DESIGN.md section 9) ----------------------------------
// The links [lb, le) of the pull CSR are the rows [row_begin, row_end) of this rank.  Link p of row r whose source lies
// in block b belongs to the virtual row b * R + (r - row_begin); keys / vals feed the stable sort by block that puts the
// links into (block, row, accumulation order) order.
__global__ void k_vrow_count(const u32* __restrict__ in_ptr, const int32_t* __restrict__ in_src, int row_begin, int row_end,
                             u32 lb, u32 le, u32 block_size, int R, u32* __restrict__ cnt, u32* __restrict__ keys,
                             u32* __restrict__ vals) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)(le - lb)) return;
    const u32 p = lb + (u32)i;
    int lo = row_begin, hi = row_end;            // in_ptr[lo] <= p < in_ptr[hi]
    while (hi - lo > 1) {
        const int mid = (int)(((unsigned)lo + (unsigned)hi) >> 1);
        if (in_ptr[mid] <= p) lo = mid; else hi = mid;
    }
    const u32 b = (u32)in_src[p] / block_size;
    atomicAdd(&cnt[(size_t)b * R + (size_t)(lo - row_begin)], 1u);
    keys[i] = b;
    vals[i] = (u32)i;
}

__global__ void k_vrow_len(const u32* __restrict__ cnt, size_t v, u32* __restrict__ len) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < v) { const u32 c = cnt[i]; len[i] = c ? c : 1u; }
}

// like k_ws_fill, over the virtual rows: ptr2[v] = first stream position of virtual row v, cnt_ptr[v] = first entry of
// `perm` (links in (block, row, accumulation) order, relative to lb) that belongs to it
__global__ void k_ws_fill_blocked(const u32* __restrict__ ptr2, const u32* __restrict__ cnt_ptr, const u32* __restrict__ perm,
                                  const int32_t* __restrict__ in_src, const double* __restrict__ in_val, int V, int n, u32 nnz2,
                                  size_t padded, const HubMap hm, int32_t* __restrict__ ws_src,
                                  double* __restrict__ ws_val /* may be null */) {
    const size_t phys = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (phys >= padded) return;
    const u32 o = (u32)(phys % WS_STAGE);
    const u32 rnd = o / WS_STEP, ln = (o % WS_STEP) / 4, k = o % 4;
    const size_t q = phys - o + (size_t)(ln * (WS_R * 4) + rnd * 4 + k);
    const u32 zero_entry = (u32)n + (u32)hm.H;
    if (q >= nnz2) {
        ws_src[phys] = (int32_t)zero_entry;
        if (ws_val) ws_val[phys] = 0.0;
        return;
    }
    const int v = ws_row_of(ptr2, V, (u32)q);
    const u32 j = (u32)q - ptr2[v];
    const u32 b = cnt_ptr[v], cnt = cnt_ptr[v + 1] - b;
    if (cnt == 0) {
        ws_src[phys] = (int32_t)(zero_entry | END_BIT);
        if (ws_val) ws_val[phys] = 0.0;
    } else {
        const u32 link = perm[b + j];
        ws_src[phys] = (int32_t)(hub_translate(hm, (u32)in_src[link]) | (j == cnt - 1 ? END_BIT : 0u));
        if (ws_val) ws_val[phys] = in_val[link];
    }
}

// ---- slice-aligned compact blocks (partitioned graph, overlapped exchange) -------------------------------------------
// Stream block k of rank r holds the links whose source belongs to rank (r - k) mod P: block 0 gathers from the rank's own
// slice of x, block k from the slice that arrives k-th (dist.cu: every rank pushes its slice to r+1 first, then r+2, ...).
// Only the non-empty (row, block) pairs become virtual rows -- no padding links -- and k_finish_ws finds the pair of a
// row in block k through a presence bitmap and a per-word prefix count.
struct SliceMap {
    int parts, rank;
    int start[9];
};
__device__ __forceinline__ int slice_of(const SliceMap& m, u32 label) {
    int s = 0;
    for (int r = 1; r < m.parts; r++) s += (label >= (u32)m.start[r]);
    return s;
}
__global__ void k_pair_count(const u32* __restrict__ in_ptr, const int32_t* __restrict__ in_src, int row_begin, int row_end,
                             u32 lb, u32 le, const SliceMap sm, int R, u32* __restrict__ cnt, u32* __restrict__ keys,
                             u32* __restrict__ vals) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)(le - lb)) return;
    const u32 p = lb + (u32)i;
    int lo = row_begin, hi = row_end;            // in_ptr[lo] <= p < in_ptr[hi]
    while (hi - lo > 1) {
        const int mid = (int)(((unsigned)lo + (unsigned)hi) >> 1);
        if (in_ptr[mid] <= p) lo = mid; else hi = mid;
    }
    const int k = (sm.rank - slice_of(sm, (u32)in_src[p]) + sm.parts) % sm.parts;
    atomicAdd(&cnt[(size_t)k * R + (size_t)(lo - row_begin)], 1u);
    keys[i] = (u32)k;
    vals[i] = (u32)i;
}
__global__ void k_pair_flags(const u32* __restrict__ cnt, size_t v, u32* __restrict__ flags) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < v) flags[i] = cnt[i] ? 1u : 0u;
}
// The pairs of a row, in block order, as a CSR over the rows: vrow_ptr[i] .. vrow_ptr[i + 1] index vpair[], which holds the
// compact (block-major) number of each pair -- what k_finish_ws adds up for row i.
__global__ void k_pair_row_counts(const u32* __restrict__ cnt, int R, int blocks, u32* __restrict__ per_row) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    u32 c = 0;
    for (int k = 0; k < blocks; k++) c += cnt[(size_t)k * R + i] != 0;
    per_row[i] = c;
}
__global__ void k_pair_row_fill(const u32* __restrict__ cnt, const u32* __restrict__ cidx, const u32* __restrict__ vrow_ptr, int R,
                                int blocks, u32* __restrict__ vpair) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= R) return;
    u32 p = vrow_ptr[i];
    for (int k = 0; k < blocks; k++)
        if (cnt[(size_t)k * R + i] != 0) vpair[p++] = cidx[(size_t)k * R + i];
}
// stream position q -> the pair that owns it (ptr2v has one entry per (block, row) pair, empty pairs repeat their start)
__global__ void k_ws_fill_compact(const u32* __restrict__ ptr2v, const u32* __restrict__ perm, const int32_t* __restrict__ in_src,
                                  const double* __restrict__ in_val, int V, int n, u32 nnz2, size_t padded, const HubMap hm,
                                  int32_t* __restrict__ ws_src, double* __restrict__ ws_val /* may be null */) {
    const size_t phys = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (phys >= padded) return;
    const u32 o = (u32)(phys % WS_STAGE);
    const u32 rnd = o / WS_STEP, ln = (o % WS_STEP) / 4, k = o % 4;
    const size_t q = phys - o + (size_t)(ln * (WS_R * 4) + rnd * 4 + k);
    if (q >= nnz2) {
        ws_src[phys] = (int32_t)((u32)n + (u32)hm.H);
        if (ws_val) ws_val[phys] = 0.0;
        return;
    }
    const int v = ws_row_of(ptr2v, V, (u32)q);
    const u32 link = perm[q];                        // perm is in (block, row, accumulation) order == stream order
    ws_src[phys] = (int32_t)(hub_translate(hm, (u32)in_src[link]) | ((u32)q + 1 == ptr2v[v + 1] ? END_BIT : 0u));
    if (ws_val) ws_val[phys] = in_val[link];
}
__global__ void k_ws_tiles_compact(const u32* __restrict__ ptr2v, const u32* __restrict__ cidx, int V, u32 v_compact, int n_tiles,
                                   u32 tile_links, u32* __restrict__ ws_tile) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > n_tiles) return;
    if (t == n_tiles) { ws_tile[t] = v_compact; return; }
    const u32 q = (u32)t * tile_links;
    const int v = ws_row_of(ptr2v, V, q);
    ws_tile[t] = cidx[v] | (q > ptr2v[v] ? END_BIT : 0u);
}

// rwr_opts.x_blocks (0 = auto, 1 = off, 2..64 = forced); the probe knob RWR_X_BLOCKS=<B> overrides it.  Auto is off: a
// slice of C4 (x = 400 MB) runs at the same L1TEX bound with and without blocking (profiles/r02_c4slice_*), the padding
// links of the empty virtual rows cost more than the L2 misses they remove.
static int x_blocks_wanted(const rwr_graph* g) {
    int v = g->opts.x_blocks;
    if (const char* e = getenv("RWR_X_BLOCKS")) v = atoi(e);
    return (v >= 2 && v <= 64) ? v : 1;
}

void stream_prepare(rwr_graph* g) {
    cudaStream_t st = g->stream;
    const int n = g->n;
    g->ws_tiles = 0;
    g->ws_nnz = 0;
    if (n == 0) {
        g->ws_tile.alloc(1, &g->pool);
        CUDA_CHECK(cudaMemsetAsync(g->ws_tile.p, 0, sizeof(u32), st));
        return;
    }
    const u64 nnz2_max = (u64)g->nnz_in + (u64)n;
    if (nnz2_max + WS_TILE >= (1ull << 32)) RWR_FAIL(RWR_E_UNSUPPORTED, "edge stream of %llu links exceeds 32-bit offsets", (unsigned long long)nnz2_max);
    DevBuf<u32> ptr2;
    ptr2.alloc((size_t)n + 1);
    k_ws_len<<<div_up(n, 256), 256, 0, st>>>(g->in_ptr.p, n, ptr2.p);
    KERNEL_CHECK();
    u32 nnz2 = prim::scan_total<u32>(ptr2.p, ptr2.p, n, true, st, &g->pool);
    // row-partitioned graph: this rank keeps the rows [row_begin, row_end) of W^T
    u32 q0 = 0;
    g->row_begin = 0;
    g->row_end = n;
    const int parts = dist_n_ranks(g->comm);
    if (parts > 1) {                            // slices of equal row counts: graph.cu interleaved the labels for this
        const int rank = dist_rank(g->comm);
        g->row_begin = g->part_rows[rank];
        g->row_end = g->part_rows[rank + 1];
        u32 lim[2] = {0, 0};
        CUDA_CHECK(cudaMemcpyAsync(&lim[0], ptr2.p + g->row_begin, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(&lim[1], ptr2.p + g->row_end, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        q0 = lim[0];
        nnz2 = lim[1] - lim[0];
    }
    // column blocking (experimental): the stream is rebuilt over x_blocks * (row_end - row_begin) virtual rows
    DevBuf<u32> ptr2v, cnt_ptr, perm;
    u32 link_base = 0;
    g->x_blocks = 1;
    g->v_rows = g->row_end - g->row_begin;
    g->x_block_size = n;
    {
        const int want = x_blocks_wanted(g);
        const int R = g->v_rows;
        if (want > 1 && R > 0) {
            const u32 block_size = (u32)((((size_t)n + want - 1) / want + 15) & ~(size_t)15);
            const int xb = (int)(((size_t)n + block_size - 1) / block_size);
            if (xb > 1) {
                const u64 V64 = (u64)xb * (u64)R;
                if (V64 >= (1ull << 31)) RWR_FAIL(RWR_E_UNSUPPORTED, "%d blocks of %d rows exceed 2^31 virtual rows", xb, R);
                const size_t V = (size_t)V64;
                u32 lim[2] = {0, 0};
                CUDA_CHECK(cudaMemcpyAsync(&lim[0], g->in_ptr.p + g->row_begin, sizeof(u32), cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaMemcpyAsync(&lim[1], g->in_ptr.p + g->row_end, sizeof(u32), cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaStreamSynchronize(st));
                const u32 lb = lim[0], le = lim[1];
                const size_t er = (size_t)(le - lb);
                if ((u64)er + V64 + WS_TILE >= (1ull << 32)) RWR_FAIL(RWR_E_UNSUPPORTED, "blocked edge stream exceeds 32-bit offsets");
                prim::SortBuffers<u32> sb;
                cnt_ptr.alloc(V + 1); ptr2v.alloc(V + 1);
                sb.alloc(er, true);
                CUDA_CHECK(cudaMemsetAsync(cnt_ptr.p, 0, (V + 1) * sizeof(u32), st));
                if (er) {
                    k_vrow_count<<<div_up(er, 256), 256, 0, st>>>(g->in_ptr.p, g->in_src.p, g->row_begin, g->row_end, lb, le, block_size,
                                                                 R, cnt_ptr.p, sb.keys(), sb.vals());
                    KERNEL_CHECK();
                }
                k_vrow_len<<<div_up(V, 256), 256, 0, st>>>(cnt_ptr.p, V, ptr2v.p);
                KERNEL_CHECK();
                nnz2 = prim::scan_total<u32>(ptr2v.p, ptr2v.p, V, true, st, &g->pool);
                prim::exclusive_scan<u32>(cnt_ptr.p, cnt_ptr.p, V, cnt_ptr.p + V, st, &g->pool);
                sb.sort(er, ceil_log2_u64((u64)xb), st, &g->pool);
                perm = sb.take_vals();
                link_base = lb;
                q0 = 0;
                g->x_blocks = xb;
                g->x_block_size = (int32_t)block_size;
            }
        }
    }
    // slice-aligned compact blocks: a partitioned graph whose exchange is overlapped with the next SpMV (dist.cu)
    DevBuf<u32> cidx;
    g->ws_compact = false;
    g->v_compact = 0;
    if (parts > 1 && parts <= 8 && g->x_blocks == 1 && g->v_rows > 0 && dist_overlap_wanted(g)) {
        const int R = g->v_rows;
        const size_t V = (size_t)parts * (size_t)R;
        u32 lim[2] = {0, 0};
        CUDA_CHECK(cudaMemcpyAsync(&lim[0], g->in_ptr.p + g->row_begin, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(&lim[1], g->in_ptr.p + g->row_end, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        const u32 lb = lim[0], le = lim[1];
        const size_t er = (size_t)(le - lb);
        if (er > 0) {
            SliceMap smap{};
            smap.parts = parts;
            smap.rank = dist_rank(g->comm);
            for (int r = 0; r <= parts; r++) smap.start[r] = g->part_rows[r];
            DevBuf<u32> cnt;
            prim::SortBuffers<u32> sb;
            cnt.alloc(V + 1); ptr2v.alloc(V + 1); cidx.alloc(V + 1);
            sb.alloc(er, true);
            CUDA_CHECK(cudaMemsetAsync(cnt.p, 0, (V + 1) * sizeof(u32), st));
            k_pair_count<<<div_up(er, 256), 256, 0, st>>>(g->in_ptr.p, g->in_src.p, g->row_begin, g->row_end, lb, le, smap, R, cnt.p,
                                                         sb.keys(), sb.vals());
            KERNEL_CHECK();
            nnz2 = prim::scan_total<u32>(cnt.p, ptr2v.p, V, true, st, &g->pool);
            k_pair_flags<<<div_up(V, 256), 256, 0, st>>>(cnt.p, V, cidx.p);
            KERNEL_CHECK();
            const u32 vc = prim::scan_total<u32>(cidx.p, cidx.p, V, true, st, &g->pool);
            sb.sort(er, ceil_log2_u64((u64)parts), st, &g->pool);
            perm = sb.take_vals();
            link_base = lb;
            q0 = 0;
            g->x_blocks = parts;
            g->ws_compact = true;
            g->v_compact = (int32_t)vc;
            g->vrow_ptr.alloc((size_t)R + 1, &g->pool);
            g->vpair.alloc((size_t)vc + 1, &g->pool);
            k_pair_row_counts<<<div_up((size_t)R, 256), 256, 0, st>>>(cnt.p, R, parts, g->vrow_ptr.p);
            KERNEL_CHECK();
            prim::exclusive_scan<u32>(g->vrow_ptr.p, g->vrow_ptr.p, R, g->vrow_ptr.p + R, st, &g->pool);
            k_pair_row_fill<<<div_up((size_t)R, 256), 256, 0, st>>>(cnt.p, cidx.p, g->vrow_ptr.p, R, parts, g->vpair.p);
            KERNEL_CHECK();
            // first stream position of every block -> the tile that holds it (k_spmv_ws waits for a block's slice there)
            std::vector<u32> bstart(parts);
            for (int k = 0; k < parts; k++)
                CUDA_CHECK(cudaMemcpyAsync(&bstart[k], ptr2v.p + (size_t)k * R, sizeof(u32), cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaStreamSynchronize(st));
            for (int k = 0; k < 8; k++) g->blk_first_tile[k] = k < parts ? (int32_t)bstart[k] : INT32_MAX;   // links -> tiles below
        }
    }
    const bool blocked = g->x_blocks > 1;
    // hub table of a partitioned graph (see HubMap): the same entry count for both precisions, the FP64 carve-out step
    HubMap hm{};
    g->part_hub = 0;
    g->part_hub_seg = 0;
    if (parts > 1 && parts <= 8 && g->opts.hub_entries != 0 && (int)g->part_hot.size() == parts && !getenv("RWR_PART_NO_HUB")) {
        long cap = g->opts.hub_entries > 0 ? (long)g->opts.hub_entries : (long)((WS_HUB_AUTO_BYTES - WS_HDR) / 8);
        // overlapped exchange: k_push_slices lives beside k_spmv_ws on every SM; its buffers come out of the same 100 KB step
        if (g->ws_compact) cap = std::min<long>(cap, (long)((WS_HUB_AUTO_BYTES - WS_HDR - DIST_PUSH_SMEM_BYTES) / 8));
        if ((size_t)g->max_smem_optin > (size_t)WS_HDR) cap = std::min<long>(cap, (long)(((size_t)g->max_smem_optin - WS_HDR) / 8));
        long seg = cap / parts;
        for (int r = 0; r < parts; r++)                // a segment holds hot labels of ONE owner (ownership is deal_rows rounded to 32)
            seg = std::min<long>(seg, std::min<long>((long)g->part_hot[r], (long)g->part_rows[r + 1] - (long)g->deal_rows[r]));
        seg &= ~3L;
        if (seg > 0) {
            hm.parts = parts; hm.seg_len = (int)seg; hm.H = (int)seg * parts;
            for (int r = 0; r < parts; r++) hm.start[r] = g->deal_rows[r];
            g->part_hub = hm.H;
            g->part_hub_seg = hm.seg_len;
        }
    }
    // tile size: WS_TILE links, but smaller graphs (the reference's ego networks) get smaller tiles so that their links
    // still spread over every warp of every SM (big_x_probe.py with RWR_TILE_LINKS: 3.9 M links 39 / 42 / 59 us per
    // iteration with 512 / 1024 / 4096-link tiles, 19.8 M links 92 / 84 / 96 us, 61 M links 244 / 214 / 208 us)
    int tile_links = nnz2 < (u32)WS_SMALL_GRAPH_LINKS ? WS_TILE_SMALL : (nnz2 < (u32)WS_MEDIUM_GRAPH_LINKS ? WS_TILE_MEDIUM : WS_TILE);
    if (const char* et = getenv("RWR_TILE_LINKS")) {            // probe knob: any multiple of 512
        const int v = atoi(et);
        if (v >= 512 && v % 512 == 0) tile_links = v;
    }
    g->ws_tile_links = tile_links;
    const int n_tiles = (int)(((u64)nnz2 + tile_links - 1) / tile_links);
    const size_t padded = (size_t)n_tiles * tile_links;
    g->ws_nnz = nnz2;
    g->ws_tiles = n_tiles;
    g->ws_src.alloc(padded, &g->pool);
    const bool valued = g->layout == RWR_LAYOUT_VALUED;
    if (valued) g->ws_val64.alloc(padded, &g->pool);
    g->ws_tile.alloc((size_t)n_tiles + 1, &g->pool);
    if (g->ws_compact) {
        const int V = g->x_blocks * g->v_rows;
        for (int k = 0; k < 8; k++)
            if (g->blk_first_tile[k] != INT32_MAX) g->blk_first_tile[k] /= tile_links;
        if (padded)
            k_ws_fill_compact<<<div_up(padded, 256), 256, 0, st>>>(ptr2v.p, perm.p, g->in_src.p + link_base,
                                                                  valued ? g->in_val64.p + link_base : nullptr, V, n, nnz2, padded, hm,
                                                                  g->ws_src.p, valued ? g->ws_val64.p : nullptr);
        k_ws_tiles_compact<<<div_up((size_t)n_tiles + 1, 256), 256, 0, st>>>(ptr2v.p, cidx.p, V, (u32)g->v_compact, n_tiles,
                                                                            (u32)tile_links, g->ws_tile.p);
    } else if (blocked) {
        const int V = g->x_blocks * g->v_rows;
        if (padded)
            k_ws_fill_blocked<<<div_up(padded, 256), 256, 0, st>>>(ptr2v.p, cnt_ptr.p, perm.p, g->in_src.p + link_base,
                                                                  valued ? g->in_val64.p + link_base : nullptr, V, n, nnz2, padded, hm,
                                                                  g->ws_src.p, valued ? g->ws_val64.p : nullptr);
        k_ws_tiles<<<div_up((size_t)n_tiles + 1, 256), 256, 0, st>>>(ptr2v.p, V, 0u, V, n_tiles, (u32)tile_links, g->ws_tile.p);
    } else {
        DevBuf<u32> loff;                                  // freed with the order after the fill
        const DevBuf<u32> lperm = ws_long_row_order(g, g->row_begin, g->row_end - g->row_begin, loff);
        if (padded)
            k_ws_fill<<<div_up(padded, 256), 256, 0, st>>>(ptr2.p, g->in_ptr.p, g->in_src.p, valued ? g->in_val64.p : nullptr, loff.p,
                                                          lperm.p, n, g->row_begin, q0, nnz2, padded, hm, g->ws_src.p,
                                                          valued ? g->ws_val64.p : nullptr);
        CUDA_CHECK(cudaStreamSynchronize(st));
        k_ws_tiles<<<div_up((size_t)n_tiles + 1, 256), 256, 0, st>>>(ptr2.p, n, q0, g->row_end, n_tiles, (u32)tile_links, g->ws_tile.p);
    }
    KERNEL_CHECK();
    CUDA_CHECK(cudaStreamSynchronize(st));
    if (parts > 1) {          // the whole-graph pull arrays are only needed by the batched path, which a slice does not run
        g->in_src.release();
        g->in_val64.release();
    }
}

// Shared memory and L1 share the SM's 256 KB, and the L1 side is what holds the sectors of the gathers in flight: with
// the maximum carve-out (228 KB shared) the kernel ran 2x slower than with none (profiles/microbench/hub_sweep.py).
// Auto therefore stops at the 100 KB carve-out step in FP64 (~156 KB of L1 left) and at the 164 KB step in FP32,
// the best points of the sweep on the C2 graph.
int ws_hub_entries(const rwr_graph* g, int precision) {
    if (dist_n_ranks(g->comm) > 1) return g->part_hub;     // fixed at build time: the stream encodes the table slots
    const size_t elt = precision == RWR_FP32 ? 4 : 8;
    if ((size_t)g->max_smem_optin <= (size_t)WS_HDR) return 0;
    long cap = (long)(((size_t)g->max_smem_optin - WS_HDR) / elt) & ~3L;
    const long auto_cap = (long)(((precision == RWR_FP32 ? WS_HUB_AUTO_BYTES_FP32 : WS_HUB_AUTO_BYTES) - WS_HDR) / elt) & ~3L;
    long want = g->opts.hub_entries < 0 ? std::min(cap, auto_cap) : std::min<long>(cap, (long)g->opts.hub_entries & ~3L);
    // when x is far beyond L2 (or the labels are dealt over the slices of a partitioned graph, where the hottest sources
    // are no longer a label prefix) the table is not worth the L1 it takes: big_x_probe.py, +12 % in FP32 without it
    if (g->opts.hub_entries < 0 && (size_t)g->n * elt > ((size_t)160 << 20)) want = 0;
    long n4 = ((long)g->n + 3) & ~3L;
    return (int)std::max<long>(0, std::min(want, n4));
}

// ------------------------------------------------------------------------------------------------ the kernel
// Gathers of one stage (WS_R int4 of sources per lane).  One generic-address load per link: the address points either
// into the CTA's shared-memory hub table (hot sources) or at x in global memory (L2).  One instruction and one
// destination register per link, no branch, nothing for a later load to wait on.
#ifndef WS_GATHER_GENERIC
#define WS_GATHER_GENERIC 1
#endif
__device__ __forceinline__ void ws_ld_generic(double& v, u64 a) { asm volatile("ld.f64 %0, [%1];" : "=d"(v) : "l"(a)); }
__device__ __forceinline__ void ws_ld_generic(float& v, u64 a) { asm volatile("ld.f32 %0, [%1];" : "=f"(v) : "l"(a)); }
__device__ __forceinline__ void ws_lds_if(double& v, int s, int hub, u32 addr) {
    asm volatile("{\n\t.reg .pred ph;\n\tsetp.lt.s32 ph, %1, %2;\n\t@ph ld.shared.f64 %0, [%3];\n\t}" : "=d"(v) : "r"(s), "r"(hub), "r"(addr));
}
__device__ __forceinline__ void ws_lds_if(float& v, int s, int hub, u32 addr) {
    asm volatile("{\n\t.reg .pred ph;\n\tsetp.lt.s32 ph, %1, %2;\n\t@ph ld.shared.f32 %0, [%3];\n\t}" : "=f"(v) : "r"(s), "r"(hub), "r"(addr));
}
__device__ __forceinline__ void ws_ldg_if(double& v, int s, int hub, const double* addr, u64 pol) {
    asm volatile("{\n\t.reg .pred pg;\n\tsetp.ge.s32 pg, %1, %2;\n\t@pg ld.global.nc.L2::cache_hint.f64 %0, [%3], %4;\n\t}"
                 : "+d"(v) : "r"(s), "r"(hub), "l"(addr), "l"(pol));
}
__device__ __forceinline__ void ws_ldg_if(float& v, int s, int hub, const float* addr, u64 pol) {
    asm volatile("{\n\t.reg .pred pg;\n\tsetp.ge.s32 pg, %1, %2;\n\t@pg ld.global.nc.L2::cache_hint.f32 %0, [%3], %4;\n\t}"
                 : "+f"(v) : "r"(s), "r"(hub), "l"(addr), "l"(pol));
}

template <typename T, bool DBG>
__device__ __forceinline__ void ws_gather_stage(const IterParams<T>& p, const int4 (&iv)[WS_R], u64 hub_gen, u32 hub_addr,
                                                u64 pol_keep, u64 pol_stream, T (&v)[WS_R][4]) {
    int s[WS_R][4];
#pragma unroll
    for (int j = 0; j < WS_R; j++) {
        s[j][0] = iv[j].x & 0x7fffffff; s[j][1] = iv[j].y & 0x7fffffff; s[j][2] = iv[j].z & 0x7fffffff; s[j][3] = iv[j].w & 0x7fffffff;
    }
    if (DBG && p.debug >= 3) {          // probe instantiation only: 3 = no gathers, 4 = every gather from the hub, 5 = every gather from L2
#pragma unroll
        for (int j = 0; j < WS_R; j++)
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (p.debug == 3) { v[j][k] = (T)1; continue; }
                if (p.debug == 4) s[j][k] = p.hub ? s[j][k] % p.hub : 0;
                if (p.debug == 5) s[j][k] = p.hub + s[j][k] % (p.n - p.hub);
            }
        if (p.debug == 3) return;
    }
#if WS_GATHER_GENERIC
    const u64 xg = (u64)(uintptr_t)p.x;
#pragma unroll
    for (int j = 0; j < WS_R; j++)
#pragma unroll
        for (int k = 0; k < 4; k++)
        {
            if (!RWR_CHK(s[j][k] >= 0 && s[j][k] < p.chk_src_end, p.ctl, 2)) { v[j][k] = (T)0; continue; }
            ws_ld_generic(v[j][k], (s[j][k] < p.hub ? hub_gen : xg) + (u64)(u32)s[j][k] * sizeof(T));
        }
#else
#pragma unroll
    for (int j = 0; j < WS_R; j++)
#pragma unroll
        for (int k = 0; k < 4; k++) ws_lds_if(v[j][k], s[j][k], p.hub, hub_addr + (u32)s[j][k] * (u32)sizeof(T));
#pragma unroll
    for (int j = 0; j < WS_R; j++)
#pragma unroll
        for (int k = 0; k < 4; k++) ws_ldg_if(v[j][k], s[j][k], p.hub, p.x + s[j][k], s[j][k] < p.n_hot ? pol_keep : pol_stream);
#endif
}

// what a warp carries from one stage to the next
struct WsState {
    double lane_acc;       // partial sum of the open row: spread over the lanes, or in lane 31 only
    bool spread;
    bool cont;             // the tile's first row started in an earlier tile (its sum goes to head[tile])
    int row_base;          // row of the next row end
    int first_row;
    int tile;
};

// One stage of WS_STAGE links: this lane owns 8 consecutive links of the stream when the stage holds a row end (the build
// stores such a stage lane-major so that the two int4 loads stay coalesced), 8 links 32 apart when it does not (link-major,
// ws_stage_link); e = their end-of-row flags (bit k), v = their products in storage order.
// Registers and shuffles only: a load here would sit behind every gather already queued in the SM's L1TEX FIFO.
template <typename T, bool DBG>
__device__ __forceinline__ void ws_consume(const IterParams<T>& p, WsState& s, const u32 e, const double (&v)[8], const int lane,
                                           const u32 lt, const u32 le, const u64 pol_first) {
    const u32 FULL = 0xffffffffu;
    const u32 H = __ballot_sync(FULL, e != 0);
    if (H == 0 || (DBG && p.debug == 1)) {
        // inside one long row: per-lane partial, no cross-lane traffic (the only path on which the build may store a stage
        // link-major: which links a lane holds does not matter here, see ws_stage_link)
        const double a = __dadd_rn(__dadd_rn(v[0], v[1]), __dadd_rn(v[2], v[3]));
        const double b = __dadd_rn(__dadd_rn(v[4], v[5]), __dadd_rn(v[6], v[7]));
        s.lane_acc = __dadd_rn(s.lane_acc, __dadd_rn(a, b));
        s.spread = true;
        return;
    }
    // sum of the open row so far -> lane 0
    double c;
    if (s.spread) c = warp_sum(s.lane_acc);
    else c = __shfl_sync(FULL, s.lane_acc, 31);
    if (lane != 0) c = 0.0;
    // row ends before this lane / in the whole stage (counts are 0..8: four ballots over the bits of the count)
    const u32 cnt = __popc(e);
    const u32 b0 = __ballot_sync(FULL, cnt & 1u), b1 = __ballot_sync(FULL, cnt & 2u), b2 = __ballot_sync(FULL, cnt & 4u),
              b3 = __ballot_sync(FULL, cnt & 8u);
    const int before = __popc(b0 & lt) + 2 * __popc(b1 & lt) + 4 * __popc(b2 & lt) + 8 * __popc(b3 & lt);
    const int total = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2) + 8 * __popc(b3);
    // tail of this lane: the links after its last row end (all of them, plus the carry in lane 0, when it has none)
    const int last = e ? 31 - __clz(e) : -1;
    double tail = e ? 0.0 : c;
#pragma unroll
    for (int k = 0; k < 8; k++) tail = __dadd_rn(tail, k > last ? v[k] : 0.0);
    // segmented inclusive scan of the lane tails; a segment starts at every lane that holds a row end
    const u32 hm = H & le;
    const int start = hm ? 31 - __clz(hm) : 0;
    double x = tail;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const bool take = lane - d >= start;
        if (__ballot_sync(FULL, take) == 0) break;       // no segment reaches that far back: done
        const double t = __shfl_up_sync(FULL, x, d);
        if (take) x = __dadd_rn(x, t);
    }
    const double pre = __shfl_up_sync(FULL, x, 1);      // sum of the lanes before this one back to the last row end
    s.lane_acc = (lane == 31) ? x : 0.0;
    s.spread = false;
    // this lane's rows, in storage order; the first one also owns what came before the lane
    double acc = (lane == 0) ? c : pre;
    int row = s.row_base + before;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        acc = __dadd_rn(acc, v[k]);
        if (e & (1u << k)) {
            if (s.cont && row == s.first_row) p.head_partial[s.tile] = acc;
            else if ((!DBG || p.debug != 2) && RWR_CHK(row >= p.chk_y_begin && row < p.chk_y_end, p.ctl, 3)) st_policy(p.y + row, (T)acc, pol_first);
            row++;
            acc = 0.0;
        }
    }
    s.row_base += total;
}

// Warps per CTA: 16 (128 registers each) everywhere but FP32 index-only, whose smaller register footprint lets 20 warps
// fit without spills (+4.5 % there; 20 warps cost FP64 7 %: more sectors in flight than the L1 side holds).
template <typename T, bool VALUED, bool XWAIT = false> struct WsCfg {
    // XWAIT: 15 gathering warps + the push warp = 16 (registers are allotted to a CTA in groups of four warps: a 17th warp
    // would cost the other sixteen a fifth of their registers)
    static constexpr int WARPS = XWAIT ? WS_WARPS - 1 : ((sizeof(T) == 4 && !VALUED) ? 20 : WS_WARPS);
    static constexpr int THREADS = (WARPS + (XWAIT ? 1 : 0)) * 32;
};

// ---- the push warp of the overlapped exchange -----------------------------------------------------------------------
// One warp of every k_spmv_ws CTA (XWAIT instantiation) sends this rank's slice of the gather vector to the peers while the
// other sixteen gather: lane 0 drives the TMA -- bulk copies global -> shared (mbarrier) and shared -> peer memory (bulk
// groups), three 4-KB buffers in flight per SM -- peer rank+1 first.  When the last CTA has finished a peer, it releases
// the arrival tag there.  SM stores over NVLink reach ~750 GB/s where the copy engines managed ~350 GB/s for these
// peer-mapped buffers, and a warp inside the kernel needs no second stream, no events and no shared-memory re-split.
constexpr int PUSH_CHUNK = 4096;
constexpr int PUSH_BUFS = 3;
constexpr int PUSH_SMEM = PUSH_CHUNK * PUSH_BUFS + 128;          // buffers + mbarriers
template <typename T>
__device__ __noinline__ void ws_push_slices(const IterParams<T>& p, unsigned char* area /* 128-byte aligned */) {
    const int lane = threadIdx.x & 31;
    unsigned char* buf = area;
    u64* bar = reinterpret_cast<u64*>(area + PUSH_CHUNK * PUSH_BUFS);
    if (lane == 0) {
        for (int s = 0; s < PUSH_BUFS; s++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(&bar[s])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (p.push_delay > 0) { const long long t0 = clock64(); while (clock64() - t0 < p.push_delay) __nanosleep(1000); }
    }
    __syncwarp();
    const size_t n_chunks = (p.push_bytes16 + PUSH_CHUNK - 1) / PUSH_CHUNK;
    u32 phase = 0;                                           // bit s: parity of buffer s's barrier
    for (int j = 0; j < p.push_peers; j++) {
        if (lane == 0) {
            unsigned char* d = p.push_dst[j];
            auto chunk_len = [&](size_t c) { return (u32)((c + 1) * PUSH_CHUNK <= p.push_bytes16 ? PUSH_CHUNK : p.push_bytes16 - c * PUSH_CHUNK); };
            auto issue_load = [&](size_t c, int s) {
                // the bulk store that read buffer s (PUSH_BUFS chunks ago) must be done reading it
                asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(PUSH_BUFS - 2) : "memory");
                const u32 len = chunk_len(c);
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bar[s])), "r"(len) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(buf + s * PUSH_CHUNK)),
                             "l"(p.push_src + c * PUSH_CHUNK), "r"(len), "r"(smem_u32(&bar[s]))
                             : "memory");
            };
            size_t c = blockIdx.x;
            int s = 0;
            if (c < n_chunks) issue_load(c, s);
            while (c < n_chunks) {
                const size_t cn = c + gridDim.x;
                const int sn = (s + 1) % PUSH_BUFS;
                if (cn < n_chunks) issue_load(cn, sn);
                mbar_wait_a(smem_u32(&bar[s]), (phase >> s) & 1u);
                phase ^= 1u << s;
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(d + c * PUSH_CHUNK), "r"(smem_u32(buf + s * PUSH_CHUNK)),
                             "r"(chunk_len(c))
                             : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                c = cn;
                s = sn;
            }
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // every store to this peer has completed
            asm volatile("fence.proxy.async;" ::: "memory");
        }
        if (blockIdx.x == 0 && lane < p.push_tail)
            reinterpret_cast<unsigned*>(p.push_dst[j] + p.push_bytes16)[lane] = reinterpret_cast<const unsigned*>(p.push_src + p.push_bytes16)[lane];
        __threadfence_system();
        __syncwarp();
        if (lane == 0) {
            const unsigned cdone = atomicAdd(&p.push_done[j], 1u);
            if (cdone == gridDim.x - 1) {                  // every CTA's stores to this peer are out: hand over the tag
                p.push_done[j] = 0;
                __threadfence_system();
                asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p.push_flag[j]), "l"(p.wait_tag) : "memory");
            }
        }
        __syncwarp();
    }
}

// DBG: the probe instantiation (rwr_profile_iteration with RWR_DEBUG_MODE) carries the ablation branches; the production
// instantiation compiles none of them.
// XWAIT: the instantiation for the overlapped exchange of a partitioned graph (waits for the peers' slices block by block).
template <typename T, bool VALUED, bool DBG, bool XWAIT>
__global__ void __launch_bounds__(WsCfg<T, VALUED, XWAIT>::THREADS, 1) k_spmv_ws(const IterParams<T> p) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (p.ctl->done || p.iter < p.ctl->sparse_iters) return;
    u32 smem0;
    asm volatile("{ .reg .u64 t; cvta.to.shared.u64 t, %1; cvt.u32.u64 %0, t; }" : "=r"(smem0) : "l"(smem_raw));
    const u32 hub_addr = smem0 + WS_HDR;
    u64 hub_gen;                                   // generic address of the hub table, opaque to ptxas (a plain cvta result
                                                   // is rematerialised at every use)
    asm volatile("mov.u64 %0, %1;" : "=l"(hub_gen) : "l"(smem_raw + WS_HDR));
    const int lane = threadIdx.x & 31;

    if (threadIdx.x == 0) mbar_init(reinterpret_cast<u64*>(smem_raw), 1);
    __syncthreads();
    // partitioned graph: the hub table holds the hottest labels of every slice, segment after segment.  seg_ready[s] (in the
    // header, after the mbarrier): segment s of the table is loaded.
    volatile int* seg_ready = reinterpret_cast<volatile int*>(smem_raw + 16);
    if (p.hub_segs > 0 && XWAIT) {
        // overlapped exchange: only this rank's own slice of x is complete when the kernel starts.  Its segment is loaded
        // now; the segment of rank s is loaded by the first warp that finds the slice of s arrived (wait_for_tile below).
        T* hub = reinterpret_cast<T*>(smem_raw + WS_HDR);
        const int own = p.blk_src[0];
        if (threadIdx.x < 8) seg_ready[threadIdx.x] = 0;
        for (int i = threadIdx.x; i < p.hub_seg_len; i += blockDim.x) hub[own * p.hub_seg_len + i] = p.xhub[p.hub_start[own] + i];
        __syncthreads();
        if (threadIdx.x == 0) seg_ready[own] = 1;
        __syncthreads();
    } else if (p.hub_segs > 0) {
        T* hub = reinterpret_cast<T*>(smem_raw + WS_HDR);
        for (int i = threadIdx.x; i < p.hub; i += blockDim.x) {
            const int sg = i / p.hub_seg_len;
            hub[i] = p.xhub[p.hub_start[sg] + (i - sg * p.hub_seg_len)];
        }
        __syncthreads();
    } else if (p.hub > 0 && threadIdx.x == 0) {      // hub table: the first `hub` entries of x, TMA bulk copies (UBLKCP)
        const u32 bytes = (u32)p.hub * (u32)sizeof(T);
        mbar_expect_tx(reinterpret_cast<u64*>(smem_raw), bytes);
        for (u32 off = 0; off < bytes; off += 32768) {
            const u32 len = bytes - off < 32768 ? bytes - off : 32768;
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(hub_addr + off),
                         "l"(reinterpret_cast<const unsigned char*>(p.xhub) + off), "r"(len), "r"(smem0)
                         : "memory");
        }
    }
    if constexpr (XWAIT) {
        if ((int)(threadIdx.x >> 5) == WsCfg<T, VALUED, true>::WARPS) {            // the push warp
            if (p.push_src) {
                const size_t hub_bytes = ((size_t)p.hub * sizeof(T) + 127) & ~(size_t)127;
                ws_push_slices<T>(p, smem_raw + WS_HDR + hub_bytes);
            }
            return;
        }
    }
    const u64 pol_stream = policy_evict_first(), pol_keep = policy_evict_last();

    // Tiles are handed out dynamically (one atomic per tile, fetched a whole tile before it is needed): warps that
    // draw cheap tiles (long rows, hub hits) simply take more of them, and the hand-out order keeps the stream walk ascending.
    const int n_tiles = p.ws_tiles;
    // Overlapped exchange of a partitioned graph: the slices of x this launch gathers from are still arriving (the peers'
    // copy engines write them, then an arrival tag).  Stream block k may only be touched once the slice of rank blk_src[k]
    // is complete: a warp checks that when it DRAWS a tile (two tiles before it gathers from it), block after block.
    int ready = 1;                                 // stream blocks [0, ready) are known to be complete (block 0: own rows)
    auto wait_for_tile = [&](u32 t) {
        if constexpr (XWAIT) {
        if ((int)t >= n_tiles) return;
        while (ready < p.x_blocks && p.blk_first_tile[ready] <= (int)t) {
            if (lane == 0) {
                const unsigned long long* f = p.arrive + p.blk_src[ready];
                const long long t0 = clock64();
                unsigned long long v;
                do {
                    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
                    if (v >= p.wait_tag) break;
                    if (clock64() - t0 > (4LL << 30)) { p.ctl->fault = 1; break; }      // ~2 s: give up, the run is void
                    __nanosleep(200);
                } while (true);
                const long long dt = clock64() - t0;
                if (dt > 2000) atomicAdd(&p.ctl->wait_clk, (unsigned long long)dt);
            }
            __syncwarp();
            if (p.hub_segs > 0) {                           // the slice is here: its hub segment can be loaded (once per CTA,
                const int sg = p.blk_src[ready];            // a second warp racing here writes the same values)
                // lane 0 decides for the warp: the flag may flip between the reads of two lanes, and a __syncwarp inside a
                // branch only some lanes take never completes
                int need = (lane == 0) ? (seg_ready[sg] == 0) : 0;
                need = __shfl_sync(0xffffffffu, need, 0);
                if (need) {
                    T* hub = reinterpret_cast<T*>(smem_raw + WS_HDR);
                    for (int i = lane; i < p.hub_seg_len; i += 32) hub[sg * p.hub_seg_len + i] = p.xhub[p.hub_start[sg] + i];
                    __threadfence_block();
                    __syncwarp();
                    if (lane == 0) seg_ready[sg] = 1;
                }
                __threadfence_block();
            }
            ready++;
        }
        }
    };
    u32 grab = 0;                                  // lane 0: the tile drawn most recently (its value is only read a tile later)
    if (lane == 0) grab = atomicAdd(&p.ctl->tile_ctr, 1u);
    int cur = (int)__shfl_sync(0xffffffffu, grab, 0);
    if (lane == 0) grab = atomicAdd(&p.ctl->tile_ctr, 1u);
    int nxt = (int)__shfl_sync(0xffffffffu, grab, 0);
    if (lane == 0) grab = atomicAdd(&p.ctl->tile_ctr, 1u);
    wait_for_tile((u32)cur);
    wait_for_tile((u32)nxt);
    // link offset of this lane's first int4 in stage st of tile t (tiles past the end re-read the last one)
    auto pos_of = [&](int t, int st) -> size_t {
        t = t < n_tiles ? t : n_tiles - 1;
        return (size_t)t * p.tile_links + (size_t)(st * WS_STAGE + lane * 4);
    };

    const int spt = p.tile_links / WS_STAGE;       // stages per tile (even)
    if (cur < n_tiles) {
        const u32 lt = (1u << lane) - 1u, le = lt | (1u << lane);
        // two register stages, A and B, used alternately (the loop is unrolled by two so that no register that is the
        // target of a load in flight is ever copied): while stage X is being summed, the gathers of stage Y are in
        // flight and the indices of the stage after that are on their way into X's index registers.
        int4 ivA[WS_R], ivB[WS_R];
        T gA[WS_R][4], gB[WS_R][4], wA[WS_R][4], wB[WS_R][4];
        size_t posA = pos_of(cur, 0), posB = pos_of(cur, 1);
#pragma unroll
        for (int j = 0; j < WS_R; j++) {
            ivA[j] = ld_stream_int4(reinterpret_cast<const int4*>(p.ws_src + posA + j * WS_STEP), pol_stream);
            ivB[j] = ld_stream_int4(reinterpret_cast<const int4*>(p.ws_src + posB + j * WS_STEP), pol_stream);
        }
        u32 meta_cur = p.ws_tile[cur];
        u32 meta_nxt = p.ws_tile[nxt < n_tiles ? nxt : n_tiles];
        if (p.hub > 0 && p.hub_segs == 0) mbar_wait_a(smem0, 0);
        ws_gather_stage<T, DBG>(p, ivA, hub_gen, hub_addr, pol_keep, pol_stream, gA);
        if (VALUED) {
#pragma unroll
            for (int j = 0; j < WS_R; j++) load4_stream(p.ws_val + posA + j * WS_STEP, pol_stream, wA[j]);
        }
        WsState s;
        s.lane_acc = 0.0; s.spread = false; s.cont = false; s.row_base = 0; s.first_row = 0; s.tile = 0;

#ifdef RWR_PROFILE_CLOCKS
        double clk_sink = 0.0;
#define WCLK_LAND_IDX(FL, IVY) if (FL == 77u && IVY[0].x == -7 && IVY[1].w == -7) clk_sink += 1.0;
#define WCLK_LAND_G(GX) if (GX[0][0] + GX[0][1] + GX[0][2] + GX[0][3] + GX[1][0] + GX[1][1] + GX[1][2] + GX[1][3] == (T)-7) clk_sink += 1.0;
#else
#define WCLK_LAND_IDX(FL, IVY)
#define WCLK_LAND_G(GX)
#endif
        WCLK_DECL;
        // ST: stage of tile `cur` in X; stage ST + 1 sits in Y; the indices of stage ST + 2 (of `cur`, or of `nxt`) go to X
#define WS_HALF(ST, IVX, GX, WX, POSX, IVY, GY, WY, POSY)                                                              \
    {                                                                                                                  \
        const u32 fl = ((u32)IVX[0].x >> 31) | (((u32)IVX[0].y >> 31) << 1) | (((u32)IVX[0].z >> 31) << 2) |           \
                       (((u32)IVX[0].w >> 31) << 3) | (((u32)IVX[1].x >> 31) << 4) | (((u32)IVX[1].y >> 31) << 5) |    \
                       (((u32)IVX[1].z >> 31) << 6) | (((u32)IVX[1].w >> 31) << 7);                                    \
        WCLK_LAND_IDX(fl, IVY)                                                                                         \
        WCLK(0);                                                                                                       \
        /* gathers of the next stage, then the indices of the one after it into the registers just freed */            \
        ws_gather_stage<T, DBG>(p, IVY, hub_gen, hub_addr, pol_keep, pol_stream, GY);                                  \
        if (VALUED) {                                                                                                  \
            _Pragma("unroll") for (int j = 0; j < WS_R; j++) load4_stream(p.ws_val + POSY + j * WS_STEP, pol_stream, WY[j]); \
        }                                                                                                              \
        WCLK(1);                                                                                                       \
        POSX = ((ST) + 2 < spt) ? pos_of(cur, (ST) + 2) : pos_of(nxt, (ST) + 2 - spt);                                 \
        _Pragma("unroll") for (int j = 0; j < WS_R; j++)                                                               \
            IVX[j] = ld_stream_int4(reinterpret_cast<const int4*>(p.ws_src + POSX + j * WS_STEP), pol_stream);         \
        WCLK(2);                                                                                                       \
        WCLK_LAND_G(GX)                                                                                                \
        WCLK(3);                                                                                                       \
        if ((ST) == 0) {                                                                                               \
            s.tile = cur;                                                                                              \
            s.first_row = (int)(meta_cur & 0x7fffffffu);                                                               \
            s.cont = (meta_cur >> 31) != 0;                                                                            \
            s.row_base = s.first_row;                                                                                  \
            s.lane_acc = 0.0;                                                                                          \
            s.spread = false;                                                                                          \
        }                                                                                                              \
        {                                                                                                              \
            double v[8];                                                                                               \
            _Pragma("unroll") for (int j = 0; j < WS_R; j++)                                                           \
                _Pragma("unroll") for (int i = 0; i < 4; i++)                                                          \
                    v[j * 4 + i] = VALUED ? (double)mul_rn(GX[j][i], WX[j][i]) : (double)GX[j][i];                     \
            ws_consume<T, DBG>(p, s, fl, v, lane, lt, le, pol_stream);                                                 \
        }                                                                                                              \
        WCLK(4);                                                                                                       \
        if ((ST) == spt - 1) {                                                                                         \
            const double c = s.spread ? warp_sum(s.lane_acc) : __shfl_sync(0xffffffffu, s.lane_acc, 31);               \
            if (lane == 0) p.carry[s.tile] = c;                                                                        \
        }                                                                                                              \
        WCLK(5);                                                                                                       \
    }

        while (cur < n_tiles) {
            for (int st = 0; st < spt; st += 2) {
                WS_HALF(st, ivA, gA, wA, posA, ivB, gB, wB, posB)
                WS_HALF(st + 1, ivB, gB, wB, posB, ivA, gA, wA, posA)
            }
            // next tile: the one drawn a tile ago becomes `nxt`, and a new one is drawn for later
            cur = nxt;
            meta_cur = meta_nxt;
            nxt = (int)__shfl_sync(0xffffffffu, grab, 0);
            if (lane == 0 && nxt < n_tiles) grab = atomicAdd(&p.ctl->tile_ctr, 1u);
            wait_for_tile((u32)nxt);                      // a whole tile before the first gather from it
            meta_nxt = p.ws_tile[nxt < n_tiles ? nxt : n_tiles];
        }
#undef WS_HALF
        WCLK_FLUSH;
#ifdef RWR_PROFILE_CLOCKS
        if (clk_sink == -1.0) p.carry[0] = clk_sink;
#endif
    } else if (p.hub > 0 && p.hub_segs == 0 && threadIdx.x == 0) {
        // the thread that issued the bulk copies drew no tile (every tile was taken before this CTA started): a CTA must
        // not exit with a copy into its shared memory still in flight
        mbar_wait_a(smem0, 0);
    }
}

// rows cut by a tile boundary: their pieces (tails of the earlier tiles, head of the tile they end in) are added in
// tile order and stored like any other row sum
template <typename T>
__global__ void __launch_bounds__(FIX_THREADS) k_cutrows_ws(const IterParams<T> p) {
    if (p.ctl->done || p.iter < p.ctl->sparse_iters) return;
    const int t = blockIdx.x * FIX_THREADS + threadIdx.x;
    if (t >= p.ws_tiles) return;
    const u32 meta = p.ws_tile[t];
    const int row = (int)(meta & 0x7fffffffu);
    const int next_row = (int)(p.ws_tile[t + 1] & 0x7fffffffu);
    if ((meta >> 31) && next_row > row) {                 // a row from an earlier tile ends inside this tile
        int m = t - 1;
        while (m > 0 && p.ws_tile[m] == meta) m--;         // tiles lying wholly inside the row: same row, continued
        double total = 0.0;
        for (int i = m; i < t; i++) total = __dadd_rn(total, p.carry[i]);
        total = __dadd_rn(total, p.head_partial[t]);
        if (RWR_CHK(row >= p.chk_y_begin && row < p.chk_y_end, p.ctl, 3)) p.y[row] = (T)total;
    }
}

// The per-row epilogue of Model.cs:84-97 on the finished pull sums, streamed and coalesced:
//   y_t (+ S for the seed row, + S/N everywhere for the uniform restart), next x_t = fl(fl((1-c) y_t) * inv_t),
//   restart mass and L1 residual partials; the last block adds the partials in a fixed order -> next S, residual,
//   iteration count, convergence flag (Model.cs:57-66, :110-115).
// BLOCKED (column blocking of x, experimental): the raw sum of a row is the sum of its x_blocks virtual rows, block order.
// BMODE 2 (compact slice-aligned blocks): the virtual rows of row i are vpair[vrow_ptr[i] .. vrow_ptr[i + 1]), block order.
template <typename T, bool RESID, int BMODE>
__global__ void __launch_bounds__(FIN_THREADS) k_finish_ws(const IterParams<T> p, double thr, int use_thr) {
    __shared__ double scratch[2 * FIN_THREADS / 32];
    __shared__ int is_last;
    IterCtl* ctl = p.ctl;
    if (ctl->done || p.iter < ctl->sparse_iters) return;       // (done sparsely: frontier.cu)
    const double S = ctl->S;
    const int seed = ctl->seed;
    const T uni_add = (T)((seed < 0) ? S * p.inv_n : 0.0);
    // Model.cs:92-93 / :96-97 add `x * restart[r]` to EVERY node r: for a one-hot restart vector that is `x * 0`, nothing -- unless
    // some rank x is NaN or Inf (a row whose weights sum to 0, Graph.cs:81): then every entry of the next vector is NaN.  S is the
    // sum of those x, so `S * 0` is NaN exactly then.
    const bool poisoned = seed >= 0 && !((S * 0.0) == 0.0);
    const u64 pol_first = policy_evict_first(), pol_last = policy_evict_last();
    double accS = 0.0, accR = 0.0;
    for (int row = p.row_begin + blockIdx.x * FIN_THREADS + threadIdx.x; row < p.row_end; row += gridDim.x * FIN_THREADS) {
        T y;
        if (BMODE == 1) {
            const T* part = p.yv + (row - p.row_begin);
            y = ld_stream(part, pol_first);
            for (int b = 1; b < p.x_blocks; b++) y = add_rn(y, ld_stream(part + (size_t)b * (size_t)p.v_rows, pol_first));
        } else if (BMODE == 2) {
            const int i = row - p.row_begin;
            const u32 pb = p.vrow_ptr[i], pe = p.vrow_ptr[i + 1];
            y = (T)0;
            for (u32 q = pb; q < pe; q++)
                if (RWR_CHK(q < (u32)p.chk_pairs && p.vpair[q] < (u32)p.chk_pairs, ctl, 4)) y = add_rn(y, ld_stream(p.yv + p.vpair[q], pol_first));
        } else {
            y = ld_stream(p.y + row, pol_first);
        }
        const T invr = ld_stream(p.inv + row, pol_first);
        if (row == seed) { y = (T)__dadd_rn((double)y, S); p.y[row] = y; }
        if (seed < 0) { y = add_rn(y, uni_add); p.y[row] = y; }
        if (poisoned && row != seed) { y = (T)(S * 0.0); p.y[row] = y; }
        if (BMODE != 0) p.y[row] = y;
        const T rw = mul_rn(p.omc, y);
        // the next iteration gathers x_next: hot rows should still be in L2 then, cold rows are streamed
        const T xn = mul_rn(rw, invr);
        st_policy(p.x_next + row, xn, row < p.n_hot ? pol_last : pol_first);
        // row-partitioned: this rank's slice of the next x goes straight into every peer's copy (coalesced NVLink
        // stores, overlapped with the rest of this kernel) -- the allGather is fused into the epilogue
#pragma unroll 1
        for (int j = 0; j < p.n_peers; j++) reinterpret_cast<T*>(p.peer_next[j])[row] = xn;
        accS += (invr == (T)0) ? (double)y : (double)sub_rn(y, rw);
        if (RESID) {
            const T rp = ld_stream(p.r_prev + row, pol_first);
            accR += (double)((rp > y) ? sub_rn(rp, y) : sub_rn(y, rp));
        }
    }
    if (p.n_peers) __threadfence_system();                 // peer stores are visible before this kernel is seen complete
    if (grid_sum2<FIN_THREADS, true>(accS, accR, p.slot_S, p.slot_R, ctl, scratch, &is_last) && threadIdx.x == 0) {
        ctl->iters += 1;
        ctl->ticket = 0;
        ctl->tile_ctr = 0;                                // the next k_spmv_ws hands its tiles out from the start
        if (p.parted) {                                   // partial sums of this rank's rows: k_after_reduce finishes the job
            ctl->red[0] = accS;
            ctl->red[1] = accR;
        } else {
            ctl->S = accS;
            ctl->resid = accR;
            if (use_thr && accR < thr) ctl->done = 1;     // strict `<` (Model.cs:114)
        }
    }
}

// The epilogue of a restart-set run (rwr_run_*_restart): k_finish_ws with the sparse restart vector q of a RestartSet in
// place of e_seed or 1/N, Model.cs:92-93 / :96-97 with `restart` = q.  A member row adds S * q_r in double and rounds once,
// as the seed row adds S; its membership bit comes from one coalesced word per 32 rows, and q_r is read for member rows
// only.  A separate kernel, so that the seeded and uniform instantiations stay exactly what they were.  BMODE 0 and 1 only:
// a restart set never runs on a row-partitioned graph (no peers, no compact blocks, no allReduce of the sums).
template <typename T, bool RESID, int BMODE>
__global__ void __launch_bounds__(FIN_THREADS) k_finish_set_ws(const IterParams<T> p, double thr, int use_thr, const RestartSet rs) {
    __shared__ double scratch[2 * FIN_THREADS / 32];
    __shared__ int is_last;
    IterCtl* ctl = p.ctl;
    if (ctl->done || p.iter < ctl->sparse_iters) return;       // (done sparsely: frontier.cu)
    const double S = ctl->S;
    // the rows outside the set add `S * 0`: nothing, unless S is NaN or Inf (see k_finish_ws)
    const bool poisoned = !((S * 0.0) == 0.0);
    const u64 pol_first = policy_evict_first(), pol_last = policy_evict_last();
    double accS = 0.0, accR = 0.0;
    for (int row = p.row_begin + blockIdx.x * FIN_THREADS + threadIdx.x; row < p.row_end; row += gridDim.x * FIN_THREADS) {
        T y;
        if (BMODE == 1) {
            const T* part = p.yv + (row - p.row_begin);
            y = ld_stream(part, pol_first);
            for (int b = 1; b < p.x_blocks; b++) y = add_rn(y, ld_stream(part + (size_t)b * (size_t)p.v_rows, pol_first));
        } else {
            y = ld_stream(p.y + row, pol_first);
        }
        const T invr = ld_stream(p.inv + row, pol_first);
        const int w = row >> 5;
        const u32 word = RWR_CHK(w < rs.words, ctl, 5) ? __ldg(rs.bits + w) : 0u;
        if ((word >> (row & 31)) & 1u) {
            const u32 k = __ldg(rs.word_base + w) + (u32)__popc(word & ((1u << (row & 31)) - 1u));
            const double qr = RWR_CHK(k < (u32)rs.m, ctl, 6) ? __ldg(rs.q + k) : 0.0;
            y = (T)__dadd_rn((double)y, __dmul_rn(S, qr));
            p.y[row] = y;
        } else if (poisoned) {
            y = (T)(S * 0.0);
            p.y[row] = y;
        }
        if (BMODE != 0) p.y[row] = y;
        const T rw = mul_rn(p.omc, y);
        // the next iteration gathers x_next: hot rows should still be in L2 then, cold rows are streamed
        const T xn = mul_rn(rw, invr);
        st_policy(p.x_next + row, xn, row < p.n_hot ? pol_last : pol_first);
        accS += (invr == (T)0) ? (double)y : (double)sub_rn(y, rw);
        if (RESID) {
            const T rp = ld_stream(p.r_prev + row, pol_first);
            accR += (double)((rp > y) ? sub_rn(rp, y) : sub_rn(y, rp));
        }
    }
    if (grid_sum2<FIN_THREADS, true>(accS, accR, p.slot_S, p.slot_R, ctl, scratch, &is_last) && threadIdx.x == 0) {
        ctl->iters += 1;
        ctl->ticket = 0;
        ctl->tile_ctr = 0;                                // the next k_spmv_ws hands its tiles out from the start
        ctl->S = accS;
        ctl->resid = accR;
        if (use_thr && accR < thr) ctl->done = 1;         // strict `<` (Model.cs:114)
    }
}

// ------------------------------------------------------------------------------------------------ launch
int ws_main_grid(const rwr_graph* g) {
    return std::max(1, std::min(g->sm_count, (g->ws_tiles + WS_WARPS - 1) / WS_WARPS));
}
int ws_fix_grid(const rwr_graph* g) { return (int)div_up((size_t)std::max(g->ws_tiles, 1), FIX_THREADS); }
int ws_fin_grid(const rwr_graph* g) {
    return std::max(1, std::min(g->sm_count * 8, (int)div_up((size_t)std::max(g->row_end - g->row_begin, 1), FIN_THREADS)));
}

template <typename T>
void ws_launch_spmv_only(rwr_graph* g, const IterParams<T>& p) {
    const bool valued = g->layout == RWR_LAYOUT_VALUED;
    const size_t smem = (size_t)WS_HDR + (size_t)p.hub * sizeof(T);
    auto kern = p.debug ? (valued ? k_spmv_ws<T, true, true, false> : k_spmv_ws<T, false, true, false>)
                        : p.arrive ? (valued ? k_spmv_ws<T, true, false, true> : k_spmv_ws<T, false, false, true>)
                                   : (valued ? k_spmv_ws<T, true, false, false> : k_spmv_ws<T, false, false, false>);
    const int threads = p.arrive ? WS_WARPS * 32 : (valued ? WsCfg<T, true>::WARPS : WsCfg<T, false>::WARPS) * 32;
    // the opt-in ceiling is a per-function, per-device setting shared by every handle and thread: always the device
    // maximum (a per-launch value would race between threads whose graphs have different hub sizes); the carve-out a
    // launch gets still follows the dynamic size it asks for
    CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, g->max_smem_optin));
    IterParams<T> pv = p;
    pv.chk_src_end = g->n + p.hub + 8;
    pv.chk_y_begin = p.x_blocks > 1 ? 0 : g->row_begin;
    pv.chk_y_end = g->ws_compact ? g->v_compact : (p.x_blocks > 1 ? p.x_blocks * g->v_rows : g->row_end);
    pv.xhub = p.x;
    pv.hub_segs = 0;
    pv.hub_seg_len = 1;
    if (g->part_hub > 0 && p.hub == g->part_hub) {          // partitioned graph: segmented hub table, shifted gather vector
        pv.hub_segs = (int)g->part_hot.size();
        pv.hub_seg_len = g->part_hub_seg;
        for (int r = 0; r < pv.hub_segs; r++) pv.hub_start[r] = g->deal_rows[r];
        pv.x = p.x - g->part_hub;
    }
    if (p.x_blocks > 1) pv.y = p.yv;              // the row sums of the virtual rows go to yv
    // XWAIT: the buffers of the push warp sit behind the hub table
    const size_t smem_launch = p.arrive ? (size_t)WS_HDR + (((size_t)p.hub * sizeof(T) + 127) & ~(size_t)127) + PUSH_SMEM : smem;
    kern<<<ws_main_grid(g), threads, smem_launch, g->stream>>>(pv);
    KERNEL_CHECK();
}
// the epilogue of a restart-set run (never on a partitioned graph: no compact blocks)
template <typename T>
static void launch_finish_set(rwr_graph* g, const IterParams<T>& p, bool resid, double thr, int use_thr, const RestartSet& rs) {
    const int grid = ws_fin_grid(g);
    if (p.x_blocks > 1) {
        if (resid) k_finish_set_ws<T, true, 1><<<grid, FIN_THREADS, 0, g->stream>>>(p, thr, use_thr, rs);
        else k_finish_set_ws<T, false, 1><<<grid, FIN_THREADS, 0, g->stream>>>(p, thr, use_thr, rs);
    } else {
        if (resid) k_finish_set_ws<T, true, 0><<<grid, FIN_THREADS, 0, g->stream>>>(p, thr, use_thr, rs);
        else k_finish_set_ws<T, false, 0><<<grid, FIN_THREADS, 0, g->stream>>>(p, thr, use_thr, rs);
    }
}

template <typename T>
void ws_launch_finish_only(rwr_graph* g, const IterParams<T>& p, bool resid, double thr, int use_thr, const RestartSet* rs) {
    if (p.x_blocks > 1) {
        IterParams<T> pv = p;
        pv.y = p.yv;
        pv.chk_y_begin = 0;
        pv.chk_y_end = g->ws_compact ? g->v_compact : p.x_blocks * g->v_rows;
        pv.chk_pairs = g->v_compact;
        IterParams<T> pf = p;
        pf.chk_pairs = g->v_compact;
        k_cutrows_ws<T><<<ws_fix_grid(g), FIX_THREADS, 0, g->stream>>>(pv);
        if (rs) {
            launch_finish_set<T>(g, p, resid, thr, use_thr, *rs);
        } else if (p.compact) {
            if (resid) k_finish_ws<T, true, 2><<<ws_fin_grid(g), FIN_THREADS, 0, g->stream>>>(pf, thr, use_thr);
            else k_finish_ws<T, false, 2><<<ws_fin_grid(g), FIN_THREADS, 0, g->stream>>>(pf, thr, use_thr);
        } else {
            if (resid) k_finish_ws<T, true, 1><<<ws_fin_grid(g), FIN_THREADS, 0, g->stream>>>(p, thr, use_thr);
            else k_finish_ws<T, false, 1><<<ws_fin_grid(g), FIN_THREADS, 0, g->stream>>>(p, thr, use_thr);
        }
        KERNEL_CHECK();
        return;
    }
    IterParams<T> pc = p;
    pc.chk_y_begin = g->row_begin;
    pc.chk_y_end = g->row_end;
    k_cutrows_ws<T><<<ws_fix_grid(g), FIX_THREADS, 0, g->stream>>>(pc);
    if (rs) launch_finish_set<T>(g, p, resid, thr, use_thr, *rs);
    else if (resid) k_finish_ws<T, true, 0><<<ws_fin_grid(g), FIN_THREADS, 0, g->stream>>>(p, thr, use_thr);
    else k_finish_ws<T, false, 0><<<ws_fin_grid(g), FIN_THREADS, 0, g->stream>>>(p, thr, use_thr);
    KERNEL_CHECK();
}
template <typename T>
void ws_launch_iteration(rwr_graph* g, const IterParams<T>& p, bool resid, double thr, int use_thr, const RestartSet* rs) {
    ws_launch_spmv_only<T>(g, p);
    ws_launch_finish_only<T>(g, p, resid, thr, use_thr, rs);
    g->pool.launches += 3;
}
template void ws_launch_iteration<double>(rwr_graph*, const IterParams<double>&, bool, double, int, const RestartSet*);
template void ws_launch_iteration<float>(rwr_graph*, const IterParams<float>&, bool, double, int, const RestartSet*);
template void ws_launch_spmv_only<double>(rwr_graph*, const IterParams<double>&);
template void ws_launch_spmv_only<float>(rwr_graph*, const IterParams<float>&);
template void ws_launch_finish_only<double>(rwr_graph*, const IterParams<double>&, bool, double, int, const RestartSet*);
template void ws_launch_finish_only<float>(rwr_graph*, const IterParams<float>&, bool, double, int, const RestartSet*);

#ifdef RWR_PROFILE_CLOCKS
extern "C" int rwr_debug_clocks_ws(unsigned long long* out16, int reset) {
    if (out16) cudaMemcpyFromSymbol(out16, g_clk_ws, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_clk_ws, z, sizeof(z)); }
    return 0;
}
#endif
