// graph.cu -- graph handle, transition-matrix construction (K1-K5) and parity probes.
//
// Restates Recommenders/RWRBased/Graph.cs:51-88 (buildGraph) on the device:
//   K1  explicit-link flags / out-degree count      Graph.cs:57-61
//   K2  exclusive scan -> row_ptr                   (implicit in `new ForwardLink[nExplicitLinks]`, Graph.cs:66)
//   K3  stable CSR scatter in insertion order       Graph.cs:71-77
//   K4  sequential row sums + IEEE division         Graph.cs:70, :75, :80-81
//   K5  pull layout: CSR of W^T (turns the push loop Model.cs:85-88 into a gather), rows and sources relabelled
//       by descending out-degree, sources inside a row kept in the reference's accumulation order.
#include <algorithm>
#include <chrono>

#include "graph.h"
#include "primitives.cuh"
#include "dist.h"
#include "stream.h"

// ------------------------------------------------------------------------------------------------ kernels
__global__ void k_i32_to_u8(const int32_t* __restrict__ in, u8* __restrict__ out, size_t n, int* bad) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        int32_t v = in[i];
        if (v < 0 || v > 255) *bad = 1;
        out[i] = (u8)v;
    }
}

// flags[0]: a source outside [0, n); flags[1]: sources not ascending
__global__ void k_check_src(const int32_t* __restrict__ src, size_t e0, int32_t n, int* flags) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < e0) {
        int32_t s = src[i];
        if (s < 0 || s >= n) flags[0] = 1;
        if (i > 0 && src[i - 1] > s) flags[1] = 1;
    }
}

__global__ void k_ptr_diff(const u32* __restrict__ ptr, int32_t n, u32* __restrict__ out) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = ptr[i + 1] - ptr[i];
}

__global__ void k_iota(u32* out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (u32)i;
}

template <typename T>
__global__ void k_gather(const T* __restrict__ in, const u32* __restrict__ idx, T* __restrict__ out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = in[idx[i]];
}

// ptr[s] = first position p with keys[p] >= s, for s in [0, n]   (keys ascending)
template <typename KeyT>
__global__ void k_lower_bounds(const KeyT* __restrict__ keys, size_t e, int32_t n, u32* __restrict__ ptr) {
    size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s > (size_t)n) return;
    size_t lo = 0, hi = e;
    while (lo < hi) {
        size_t mid = (lo + hi) >> 1;
        if ((size_t)keys[mid] < s) lo = mid + 1; else hi = mid;
    }
    ptr[s] = (u32)lo;
}

// K1: flag explicit links (type != UNDEFINED) and validate their targets (IndexOutOfRange at Model.cs:87)
// `mask`: bit t set = links of EdgeType t count as UNDEFINED (the methodology switches of Experiment.cs:84-101, which
// retype FRIENDSHIP links to UNDEFINED before buildGraph(), as one option instead of a rewrite of the link list)
__device__ __forceinline__ bool link_is_explicit(u8 t, u32 mask) { return t != RWR_EDGE_UNDEFINED && !(t < 32 && ((mask >> t) & 1u)); }
__device__ __forceinline__ bool type_in(u8 t, u32 mask) { return t < 32 && ((mask >> t) & 1u); }

// rwr_opts.zero_weight_type_mask (MENTION under methodology 15): DataLoader.addMentionCount2 gives a member mention links only
// when `allLinks` already holds an entry for it (DataLoader.cs:403-405) -- a member whose other relations were not loaded gets
// none and stays a dangling row, it does NOT become a row of zero weights (0 / 0 = NaN).  Hence: a link of a zero-weight type
// is in the matrix only if its source has an explicit link of another type (`carrier[source]`, null when no such type is set).
__device__ __forceinline__ bool link_in_matrix(u8 t, const int32_t* __restrict__ src, size_t i, u32 mask, u32 zero_mask,
                                               const u8* __restrict__ carrier) {
    if (!link_is_explicit(t, mask)) return false;
    if (carrier && type_in(t, zero_mask)) return carrier[src[i]] != 0;       // (src is only read on this path)
    return true;
}
__global__ void k_carrier_flags(const u8* __restrict__ type, const int32_t* __restrict__ src, size_t e0, int32_t n, u32 mask,
                                u32 zero_mask, u8* __restrict__ carrier) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < e0 && link_is_explicit(type[i], mask) && !type_in(type[i], zero_mask)) {
        const int32_t s = src[i];
        if (s >= 0 && s < n) carrier[s] = 1;
    }
}

__global__ void k_explicit_flags(const u8* __restrict__ type, const int32_t* __restrict__ src, const int32_t* __restrict__ dst,
                                 size_t e0, int32_t n, u32 mask, u32 zero_mask, const u8* __restrict__ carrier,
                                 u32* __restrict__ flags, int* bad) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < e0) {
        u32 f = link_in_matrix(type[i], src, i, mask, zero_mask, carrier);
        if (f) {
            int32_t d = dst[i];
            if (d < 0 || d >= n) *bad = 1;
        }
        flags[i] = f;
    }
}

// K3: stable compaction of the explicit links (insertion order kept: pos is an exclusive scan of the flags)
// `zero_mask`: links of these types keep their slot with weight 0.0 (rwr_opts.zero_weight_type_mask)
__global__ void k_compact(const u8* __restrict__ type, const u32* __restrict__ pos, const int32_t* __restrict__ src,
                          const int32_t* __restrict__ dst, const double* __restrict__ w, size_t e0, u32 mask, u32 zero_mask,
                          const u8* __restrict__ carrier, int32_t* __restrict__ src_of, int32_t* __restrict__ col,
                          double* __restrict__ wv) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < e0) {
        const u8 t = type[i];
        if (!link_in_matrix(t, src, i, mask, zero_mask, carrier)) return;
        u32 p = pos[i];
        src_of[p] = src[i];
        col[p] = dst[i];
        wv[p] = type_in(t, zero_mask) ? 0.0 : w[i];
    }
}

// `graph[i][k].type`: the types of the explicit links in CSR order
__global__ void k_compact_types(const u8* __restrict__ type, const int32_t* __restrict__ src, const u32* __restrict__ pos, size_t e0,
                                u32 mask, u32 zero_mask, const u8* __restrict__ carrier, int32_t* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < e0 && link_in_matrix(type[i], src, i, mask, zero_mask, carrier)) out[pos[i]] = (int32_t)type[i];
}

__global__ void k_row_ptr_from_pos(const u32* __restrict__ raw_ptr, const u32* __restrict__ pos, size_t e0, u32 nnz,
                                   int32_t n, u32* __restrict__ row_ptr) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= (size_t)n) {
        u32 r = raw_ptr[i];
        row_ptr[i] = (r >= e0) ? nnz : pos[r];
    }
}

struct BuildStats {
    int n_dangling;
    int all_uniform;
    u32 max_out;
    u32 max_in;
    int n_items;
};

// K4a: rows with <= 32 links, one thread per row, strictly sequential sum (Graph.cs:70-77 order)
// K4b: longer rows, one warp per row: all-ones rows sum exactly to their length, anything else is summed
//      sequentially by lane 0 to keep the reference's rounding.
constexpr u32 ROWSUM_SHORT = 32;
constexpr size_t WS_PAD_LINKS = 1 << 16;      // head-room of the 32-bit stream offsets (padding links, tile padding)

__device__ __forceinline__ void rowsum_finish(int32_t i, u32 deg, double sum, double w0, bool uniform, double* rowsum,
                                              double* w0norm, u8* uni, BuildStats* st) {
    rowsum[i] = sum;
    w0norm[i] = deg ? __ddiv_rn(w0, sum) : 0.0;
    uni[i] = uniform ? 1 : 0;
    if (deg == 0) atomicAdd(&st->n_dangling, 1);
    else if (!uniform) atomicAnd(&st->all_uniform, 0);
    atomicMax(&st->max_out, deg);
}

__global__ void k_rowsum_short(const u32* __restrict__ row_ptr, const double* __restrict__ wv, int32_t n,
                               double* __restrict__ rowsum, double* __restrict__ w0norm, u8* __restrict__ uni,
                               BuildStats* st) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 b = row_ptr[i], e = row_ptr[i + 1], deg = e - b;
    if (deg > ROWSUM_SHORT) return;
    double sum = 0.0, w0 = deg ? wv[b] : 0.0;
    bool uniform = true;
    for (u32 k = b; k < e; k++) {
        double w = wv[k];
        sum = __dadd_rn(sum, w);
        uniform = uniform && (w == w0);
    }
    rowsum_finish(i, deg, sum, w0, uniform, rowsum, w0norm, uni, st);
}

__global__ void k_rowsum_long(const u32* __restrict__ row_ptr, const double* __restrict__ wv, int32_t n,
                              double* __restrict__ rowsum, double* __restrict__ w0norm, u8* __restrict__ uni,
                              BuildStats* st) {
    int32_t i = (int32_t)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    int lane = threadIdx.x & 31;
    if (i >= n) return;
    u32 b = row_ptr[i], e = row_ptr[i + 1], deg = e - b;
    if (deg <= ROWSUM_SHORT) return;
    double w0 = wv[b];
    bool same = true;
    for (u32 k = b + lane; k < e; k += 32) same = same && (wv[k] == w0);
    bool uniform = __all_sync(0xffffffffu, same);
    if (lane == 0) {
        double sum;
        if (uniform && w0 == 1.0) {
            sum = (double)deg;                       // deg sequential additions of 1.0 are exact
        } else {
            sum = 0.0;
            for (u32 k = b; k < e; k++) sum = __dadd_rn(sum, wv[k]);
        }
        rowsum_finish(i, deg, sum, w0, uniform, rowsum, w0norm, uni, st);
    }
}

// K4c: Graph.cs:80-81
__global__ void k_normalise(const double* __restrict__ wv, const int32_t* __restrict__ src_of,
                            const double* __restrict__ rowsum, size_t nnz, double* __restrict__ val) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) val[i] = __ddiv_rn(wv[i], rowsum[src_of[i]]);
}

// per-node facts the relabel and the per-node arrays need: explicit out-degree, first out-neighbour (0 without links),
// common normalised weight (index-only layout) -- of the rows whose links this handle holds; a partitioned build sums the
// three arrays over the ranks (every node is owned by exactly one rank, the others contribute zeros)
__global__ void k_node_facts(const u32* __restrict__ row_ptr, const int32_t* __restrict__ col, const double* __restrict__ w0norm,
                             int32_t n, u32* __restrict__ deg, u32* __restrict__ first_nb, double* __restrict__ w0) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32 b = row_ptr[i], d = row_ptr[i + 1] - b;
    deg[i] = d;
    first_nb[i] = d ? (u32)col[b] : 0u;
    w0[i] = d ? w0norm[i] : 0.0;
}
__global__ void k_deg_stats(const u32* __restrict__ deg, int32_t n, BuildStats* st) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32 d = deg[i];
    if (d == 0) atomicAdd(&st->n_dangling, 1);
    atomicMax(&st->max_out, d);
}

__global__ void k_degree_keys(const u32* __restrict__ deg, int32_t n, u32 max_out, u32* __restrict__ keys,
                              u32* __restrict__ vals) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        keys[i] = max_out - deg[i];
        vals[i] = (u32)i;
    }
}

__global__ void k_invert_perm(const u32* __restrict__ old_of_new_u, int32_t n, int32_t* __restrict__ old_of_new,
                              int32_t* __restrict__ new_of_old) {
    int32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) {
        int32_t o = (int32_t)old_of_new_u[j];
        old_of_new[j] = o;
        new_of_old[o] = j;
    }
}

// cold == 1 <= out-degree < hot_min.  counts[0] = hot nodes, counts[1] = cold nodes
__global__ void k_cold_flags(const u32* __restrict__ degs, int32_t n, u32 hot_min, u32* __restrict__ flags, u32* counts) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32 deg = degs[i];
    const u32 cold = deg >= 1 && deg < hot_min;
    flags[i] = cold;
    if (deg >= hot_min) atomicAdd(&counts[0], 1u);
    else if (cold) atomicAdd(&counts[1], 1u);
}

// key of a cold node = label of its first out-neighbour when that one is hot, else n_hot + its original index
__global__ void k_cold_keys(const u32* __restrict__ degs, const u32* __restrict__ first_nb,
                            const int32_t* __restrict__ new_of_old, int32_t n, u32 hot_min, u32 n_hot,
                            const u32* __restrict__ pos, u32* __restrict__ keys, u32* __restrict__ vals) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u32 deg = degs[i];
    if (deg >= 1 && deg < hot_min) {
        const int32_t nb = (int32_t)first_nb[i];
        const u32 lab = (u32)new_of_old[nb];
        keys[pos[i]] = lab < n_hot ? lab : n_hot + (u32)nb;
        vals[pos[i]] = (u32)i;
    }
}

__global__ void k_assign_cold(const u32* __restrict__ sorted_ids, u32 n_cold, u32 n_hot, int32_t* __restrict__ new_of_old,
                              int32_t* __restrict__ old_of_new) {
    u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_cold) {
        const int32_t o = (int32_t)sorted_ids[p];
        new_of_old[o] = (int32_t)(n_hot + p);
        old_of_new[n_hot + p] = o;
    }
}

// Row-partitioned graphs: deal the label order over the P slices so that every contiguous slice of labels holds
// near-equal rows AND near-equal link counts.  The hot part of the order (degree-sorted) is dealt node by node --
// position i to slice i mod P -- so every slice gets every P-th hub; the cold part (low-degree nodes clustered next to
// their first neighbour) is dealt in blocks of DEAL_BLOCK positions, so that the siblings of a cluster stay adjacent
// and the row that gathers them still reads whole sectors.  Labels stay dense in [0, n); `start[r]` = first label of
// slice r, `hot_of[r]` = hot nodes in slice r.
constexpr int DEAL_BLOCK = 64;
struct DealPlan {
    int32_t start[17];
    int32_t hot_of[16];
    int32_t block;
};
__global__ void k_deal_labels(const int32_t* __restrict__ old_of_new_in, int32_t n, int32_t n_hot, int32_t parts, DealPlan plan,
                              int32_t* __restrict__ old_of_new, int32_t* __restrict__ new_of_old) {
    int32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int32_t lab;
    if (i < n_hot) {
        const int32_t r = i % parts;
        lab = plan.start[r] + i / parts;
    } else {
        const int32_t j = i - n_hot, blk = j / plan.block, r = blk % parts;
        lab = plan.start[r] + plan.hot_of[r] + (blk / parts) * plan.block + j % plan.block;
    }
    const int32_t o = old_of_new_in[i];
    old_of_new[lab] = o;
    new_of_old[o] = lab;
}

__global__ void k_identity_perm(int32_t n, int32_t* a, int32_t* b) {
    int32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) { a[j] = j; b[j] = j; }
}

__global__ void k_transpose_keys(const int32_t* __restrict__ col, const int32_t* __restrict__ new_of_old, size_t nnz,
                                 u32* __restrict__ keys, u32* __restrict__ vals) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nnz) {
        keys[i] = (u32)new_of_old[col[i]];
        vals[i] = (u32)i;
    }
}

__global__ void k_fill_pull(const u32* __restrict__ order, const int32_t* __restrict__ src_of,
                            const int32_t* __restrict__ new_of_old, const double* __restrict__ val, size_t nnz,
                            int32_t* __restrict__ in_src, double* __restrict__ in_val /* may be null */) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < nnz) {
        u32 e = order[p];
        in_src[p] = new_of_old[src_of[e]];
        if (in_val) in_val[p] = val[e];
    }
}

// ---- transpose of a partitioned build: every local link travels to the rank that owns its target row
__global__ void k_dest_keys(const int32_t* __restrict__ col, const int32_t* __restrict__ new_of_old, size_t nnz, int parts,
                            const int* __restrict__ part_rows, u32* __restrict__ keys, u32* __restrict__ vals, u32* __restrict__ cnt) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    int d = 64;                                      // lanes past the end: a bucket of their own
    if (i < nnz) {
        const int lab = new_of_old[col[i]];
        d = 0;
        for (int r = 1; r < parts; r++) d += (lab >= part_rows[r]);
        keys[i] = (u32)d;
        vals[i] = (u32)i;
    }
    const u32 peers = __match_any_sync(0xffffffffu, d);           // one atomic per bucket and warp
    if (d < 64 && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&cnt[d], (u32)__popc(peers));
}
// send buffers in destination order: (target label, original source id) [+ normalised weight]
__global__ void k_pack_links(const u32* __restrict__ order, const int32_t* __restrict__ col, const int32_t* __restrict__ src_of,
                             const int32_t* __restrict__ new_of_old, const double* __restrict__ val, size_t nnz,
                             uint2* __restrict__ out, double* __restrict__ out_val /* may be null */) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nnz) return;
    const u32 e = order[p];
    out[p] = make_uint2((u32)new_of_old[col[e]], (u32)src_of[e]);
    if (out_val) out_val[p] = val[e];
}
__global__ void k_pair_field(const uint2* __restrict__ pairs, const u32* __restrict__ idx /* may be null */, size_t n, int field,
                             u32* __restrict__ out, u32* __restrict__ iota /* may be null */) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint2 v = pairs[idx ? idx[i] : i];
    out[i] = field ? v.y : v.x;
    if (iota) iota[i] = (u32)i;
}
__global__ void k_fill_pull_recv(const u32* __restrict__ order, const uint2* __restrict__ pairs, const double* __restrict__ vals,
                                 const int32_t* __restrict__ new_of_old, size_t m, int32_t* __restrict__ in_src,
                                 double* __restrict__ in_val /* may be null */) {
    size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    const u32 e = order[p];
    in_src[p] = new_of_old[pairs[e].y];
    if (in_val) in_val[p] = vals[e];
}

__global__ void k_node_arrays(const int32_t* __restrict__ old_of_new, const u32* __restrict__ degs,
                              const double* __restrict__ w0,
                              const int64_t* __restrict__ node_id, const u8* __restrict__ node_type, int32_t n,
                              int index_layout, const u32* __restrict__ in_ptr, double* __restrict__ inv_orig,
                              double* __restrict__ inv_int, int64_t* __restrict__ id_int, u8* __restrict__ type_int,
                              BuildStats* st) {
    int32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int32_t o = old_of_new[j];
    u32 deg = degs[o];
    double inv = (deg == 0) ? 0.0 : (index_layout ? w0[o] : 1.0);
    inv_orig[o] = inv;
    inv_int[j] = inv;
    id_int[j] = node_id[o];
    u8 t = node_type[o];
    type_int[j] = t;
    if (t == RWR_NODE_ITEM) atomicAdd(&st->n_items, 1);
    atomicMax(&st->max_in, in_ptr[j + 1] - in_ptr[j]);
}

// ------------------------------------------------------------------------------------------------ host side
static inline unsigned grid_for(size_t n, int block = 256) { return n ? div_up(n, block) : 1; }

void graph_init_device(rwr_graph* g, const rwr_opts* opts) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        RWR_FAIL(RWR_E_CUDA, "no CUDA device: librwr_b200 has no CPU fallback");
    if (opts) g->opts = *opts; else { memset(&g->opts, 0, sizeof(g->opts)); g->opts.device = -1; g->opts.hub_entries = -1; }
    if (g->opts.device >= 0) {
        if (g->opts.device >= ndev) RWR_FAIL(RWR_E_INVALID, "device %d out of range (%d devices)", g->opts.device, ndev);
        CUDA_CHECK(cudaSetDevice(g->opts.device));
    }
    if (g->opts.kernel != 0) RWR_FAIL(RWR_E_INVALID, "rwr_opts.kernel is reserved and must be 0");
    CUDA_CHECK(cudaGetDevice(&g->device));
    // three attribute queries instead of cudaGetDeviceProperties (about a millisecond per call, and the reference
    // creates one graph per ego network)
    int major = 0, minor = 0, sms = 0, smem_optin = 0;
    CUDA_CHECK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, g->device));
    CUDA_CHECK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, g->device));
    CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, g->device));
    CUDA_CHECK(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, g->device));
    if (major < 10)
        RWR_FAIL(RWR_E_CUDA, "device %d is sm_%d%d; librwr_b200 is built for sm_100a only", g->device, major, minor);
    g->scratch.pool = &g->pool;
    g->sm_count = sms;
    g->max_smem_optin = smem_optin;
    if (g->opts.stream) {
        g->stream = (cudaStream_t)(uintptr_t)g->opts.stream;
        g->own_stream = false;
    } else {
        CUDA_CHECK(cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking));
        g->own_stream = true;
    }
    // keep up to 2 GB of freed blocks in the device's default memory pool (the default hands everything back at the next
    // synchronisation, which would make every build re-acquire its temporaries from the driver)
    cudaMemPool_t mp = nullptr;
    if (cudaDeviceGetDefaultMemPool(&mp, g->device) == cudaSuccess && mp) {
        uint64_t thr = 0;
        if (cudaMemPoolGetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &thr) == cudaSuccess && thr < ((uint64_t)2 << 30)) {
            thr = (uint64_t)2 << 30;
            cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    } else {
        cudaGetLastError();
    }
}

void graph_rebuild_raw_ptr(rwr_graph* g) {
    g->raw_ptr.alloc((size_t)g->n + 1, &g->pool);
    k_lower_bounds<int32_t><<<grid_for((size_t)g->n + 1), 256, 0, g->stream>>>(g->raw_src.p, (size_t)g->e0, g->n, g->raw_ptr.p);
    KERNEL_CHECK();
    CUDA_CHECK(cudaStreamSynchronize(g->stream));
}

// Canonicalise the raw links: stable sort by source when needed, then raw_ptr.
void graph_finish_create(rwr_graph* g) {
    cudaStream_t st = g->stream;
    const size_t e0 = (size_t)g->e0;
    DevBuf<int> flags;
    flags.alloc(2);
    CUDA_CHECK(cudaMemsetAsync(flags.p, 0, 2 * sizeof(int), st));
    if (e0) {
        k_check_src<<<grid_for(e0), 256, 0, st>>>(g->raw_src.p, e0, g->n, flags.p);
        KERNEL_CHECK();
    }
    int h[2];
    CUDA_CHECK(cudaMemcpyAsync(h, flags.p, sizeof(h), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    if (h[0]) RWR_FAIL(RWR_E_BADINDEX, "link source outside [0, %d)", g->n);
    if (h[1]) {
        // not source-ascending: stable sort by source keeps each source's insertion order
        prim::SortBuffers<u32> sb;
        sb.alloc(e0, true);
        CUDA_CHECK(cudaMemcpyAsync(sb.keys(), g->raw_src.p, e0 * sizeof(u32), cudaMemcpyDeviceToDevice, st));
        k_iota<<<grid_for(e0), 256, 0, st>>>(sb.vals(), e0);
        KERNEL_CHECK();
        sb.sort(e0, ceil_log2_u64((u64)g->n), st, &g->pool);
        DevBuf<int32_t> dst2; DevBuf<u8> type2; DevBuf<double> w2;
        dst2.alloc(e0, &g->pool); type2.alloc(e0, &g->pool); w2.alloc(e0, &g->pool);
        k_gather<int32_t><<<grid_for(e0), 256, 0, st>>>(g->raw_dst.p, sb.vals(), dst2.p, e0);
        k_gather<u8><<<grid_for(e0), 256, 0, st>>>(g->raw_type.p, sb.vals(), type2.p, e0);
        k_gather<double><<<grid_for(e0), 256, 0, st>>>(g->raw_w.p, sb.vals(), w2.p, e0);
        KERNEL_CHECK();
        CUDA_CHECK(cudaMemcpyAsync(g->raw_src.p, sb.keys(), e0 * sizeof(u32), cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        g->raw_dst = std::move(dst2);
        g->raw_type = std::move(type2);
        g->raw_w = std::move(w2);
    }
    graph_rebuild_raw_ptr(g);
}

// probe knob RWR_BUILD_TRACE=1: wall time of the build phases on stderr (each mark synchronises the stream)
struct BuildTrace {
    bool on = getenv("RWR_BUILD_TRACE") != nullptr;
    cudaStream_t st;
    int rank;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    BuildTrace(cudaStream_t s, int r) : st(s), rank(r) {}
    void mark(const char* what) {
        if (!on) return;
        cudaStreamSynchronize(st);
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[rwr build r%d] %-28s %8.1f ms\n", rank, what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

static void graph_build_impl(rwr_graph* g) {
    if (g->built) RWR_FAIL(RWR_E_ALREADY_BUILT, "buildGraph() called twice (ArgumentException at Graph.cs:86)");
    CUDA_CHECK(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    AllocStream alloc_on(st);
    const size_t e0 = (size_t)g->e0;
    const int32_t n = g->n;
    struct Events {                              // destroyed on every exit, including a failed build
        cudaEvent_t a = nullptr, b = nullptr;
        ~Events() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    } ev;
    CUDA_CHECK(cudaEventCreate(&ev.a));
    CUDA_CHECK(cudaEventCreate(&ev.b));
    CUDA_CHECK(cudaEventRecord(ev.a, st));

    DevBuf<BuildStats> stats;
    stats.alloc(1);
    BuildStats hs = {0, 1, 0, 0, 0};
    CUDA_CHECK(cudaMemcpyAsync(stats.p, &hs, sizeof(hs), cudaMemcpyHostToDevice, st));
    DevBuf<int> bad;
    bad.alloc(1);
    CUDA_CHECK(cudaMemsetAsync(bad.p, 0, sizeof(int), st));

    BuildTrace trace(st, dist_rank(g->comm));
    // ---- K1 + K2: explicit flags, exclusive scan
    DevBuf<u32> pos;
    pos.alloc(e0);
    DevBuf<u8> carrier;                    // sources that hold an explicit link of a type outside zero_weight_type_mask
    const u32 zero_mask = (u32)g->opts.zero_weight_type_mask;
    if (e0) {
        if (zero_mask) {
            carrier.alloc((size_t)std::max(n, 1));
            CUDA_CHECK(cudaMemsetAsync(carrier.p, 0, (size_t)std::max(n, 1), st));
            k_carrier_flags<<<grid_for(e0), 256, 0, st>>>(g->raw_type.p, g->raw_src.p, e0, n, (u32)g->opts.undefined_type_mask, zero_mask,
                                                         carrier.p);
        }
        k_explicit_flags<<<grid_for(e0), 256, 0, st>>>(g->raw_type.p, g->raw_src.p, g->raw_dst.p, e0, n, (u32)g->opts.undefined_type_mask,
                                                      zero_mask, carrier.p, pos.p, bad.p);
        KERNEL_CHECK();
    }
    int h_bad = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));   // complete once the scan returns
    const size_t nnz = prim::scan_total<u32>(pos.p, pos.p, e0, false, st, &g->pool);
    if (h_bad) RWR_FAIL(RWR_E_BADINDEX, "link target outside [0, %d) (IndexOutOfRangeException at Model.cs:87)", n);
    g->nnz = (int64_t)nnz;

    // ---- K3: stable scatter (skipped when no UNDEFINED link exists: the raw arrays already are the CSR)
    DevBuf<double> wv_own;
    const double* wv;
    if (nnz == e0 && g->opts.zero_weight_type_mask == 0) {
        g->compacted = false;
        g->row_ptr = g->raw_ptr.p;
        g->col = g->raw_dst.p;
        g->src_of = g->raw_src.p;
        wv = g->raw_w.p;
    } else {
        g->compacted = true;
        g->row_ptr_own.alloc((size_t)n + 1, &g->pool);
        g->col_own.alloc(nnz, &g->pool);
        g->src_of_own.alloc(nnz, &g->pool);
        wv_own.alloc(nnz);
        k_compact<<<grid_for(e0), 256, 0, st>>>(g->raw_type.p, pos.p, g->raw_src.p, g->raw_dst.p, g->raw_w.p, e0,
                                                (u32)g->opts.undefined_type_mask, zero_mask, carrier.p,
                                                g->src_of_own.p, g->col_own.p, wv_own.p);
        k_row_ptr_from_pos<<<grid_for((size_t)n + 1), 256, 0, st>>>(g->raw_ptr.p, pos.p, e0, (u32)nnz, n, g->row_ptr_own.p);
        KERNEL_CHECK();
        g->row_ptr = g->row_ptr_own.p;
        g->col = g->col_own.p;
        g->src_of = g->src_of_own.p;
        wv = wv_own.p;
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
    pos.release();
    carrier.release();

    trace.mark("K1-K3 flags/scan/compact");
    // ---- K4: row sums (sequential order), normalisation
    DevBuf<double> rowsum, w0norm;
    DevBuf<u8> uni;
    rowsum.alloc(n); w0norm.alloc(n); uni.alloc(n);
    if (n) {
        k_rowsum_short<<<grid_for(n), 256, 0, st>>>(g->row_ptr, wv, n, rowsum.p, w0norm.p, uni.p, stats.p);
        k_rowsum_long<<<grid_for((size_t)n * 32), 256, 0, st>>>(g->row_ptr, wv, n, rowsum.p, w0norm.p, uni.p, stats.p);
        KERNEL_CHECK();
    }
    g->val.alloc(nnz, &g->pool);
    if (nnz) {
        k_normalise<<<grid_for(nnz), 256, 0, st>>>(wv, g->src_of, rowsum.p, nnz, g->val.p);
        KERNEL_CHECK();
    }
    trace.mark("K4 row sums + normalise");
    // per-node facts (degree, first neighbour, common weight) of the rows this handle holds; a partitioned build makes them
    // global: every node is owned by one rank, the others add zeros
    const bool pb = g->part_build;
    DevBuf<u32> deg, first_nb;
    DevBuf<double> w0;
    deg.alloc((size_t)n + 1); first_nb.alloc((size_t)n + 1); w0.alloc((size_t)n + 1);
    if (n) {
        k_node_facts<<<grid_for(n), 256, 0, st>>>(g->row_ptr, g->col, w0norm.p, n, deg.p, first_nb.p, w0.p);
        KERNEL_CHECK();
    }
    if (pb) {
        // deg[n] carries "this rank saw a row with unequal weights"
        CUDA_CHECK(cudaMemcpyAsync(&hs, stats.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        const u32 flag = hs.all_uniform ? 0u : 1u;
        CUDA_CHECK(cudaMemcpyAsync(deg.p + n, &flag, sizeof(u32), cudaMemcpyHostToDevice, st));
        dist_allreduce_sum(g, deg.p, (size_t)n + 1, DIST_U32);
        dist_allreduce_sum(g, first_nb.p, (size_t)n, DIST_U32);
        dist_allreduce_sum(g, w0.p, (size_t)n, DIST_F64);
        BuildStats z = {0, 1, 0, 0, 0};
        CUDA_CHECK(cudaMemcpyAsync(stats.p, &z, sizeof(z), cudaMemcpyHostToDevice, st));
        if (n) k_deg_stats<<<grid_for(n), 256, 0, st>>>(deg.p, n, stats.p);
        KERNEL_CHECK();
        u32 any_nonuni = 0;
        CUDA_CHECK(cudaMemcpyAsync(&any_nonuni, deg.p + n, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(&hs, stats.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        hs.all_uniform = any_nonuni ? 0 : 1;
        int64_t counts[2] = {(int64_t)nnz, (int64_t)e0};
        DevBuf<int64_t> dc;
        dc.alloc(2);
        CUDA_CHECK(cudaMemcpyAsync(dc.p, counts, sizeof(counts), cudaMemcpyHostToDevice, st));
        dist_allreduce_sum(g, dc.p, 2, DIST_I64);
        CUDA_CHECK(cudaMemcpyAsync(counts, dc.p, sizeof(counts), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        g->nnz_global = counts[0];
        g->e0_global = counts[1];
        g->deg_all.alloc(n, &g->pool);
        if (n) CUDA_CHECK(cudaMemcpyAsync(g->deg_all.p, deg.p, (size_t)n * sizeof(u32), cudaMemcpyDeviceToDevice, st));
    } else {
        CUDA_CHECK(cudaMemcpyAsync(&hs, stats.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
    }
    wv_own.release();
    g->n_dangling = hs.n_dangling;
    g->all_uniform = hs.all_uniform != 0;
    g->max_out_degree = hs.max_out;

    int layout = g->opts.layout;
    if (layout == RWR_LAYOUT_AUTO) layout = g->all_uniform ? RWR_LAYOUT_INDEX : RWR_LAYOUT_VALUED;
    if (layout == RWR_LAYOUT_INDEX && !g->all_uniform)
        RWR_FAIL(RWR_E_UNSUPPORTED, "index-only layout needs one repeated weight per row of W (found non-uniform rows)");
    if (layout != RWR_LAYOUT_INDEX && layout != RWR_LAYOUT_VALUED) RWR_FAIL(RWR_E_INVALID, "unknown layout %d", layout);
    g->layout = layout;

    trace.mark("node facts (+ allReduce)");
    // ---- internal relabel (locality): [hot nodes by descending out-degree == how often x_i is gathered]
    //      ++ [cold nodes (out-degree < hot_min) clustered by their first out-neighbour, original order inside a
    //          cluster: the row of that neighbour then gathers them as one sequential run of x]
    //      ++ [nodes without explicit links: never gathered]
    g->new_of_old.alloc(n, &g->pool);
    g->old_of_new.alloc(n, &g->pool);
    g->relabelled = (g->opts.relabel == 0) && n > 1;
    g->n_hot = n;
    if (g->relabelled) {
        prim::SortBuffers<u32> sb;
        sb.alloc(n, true);
        k_degree_keys<<<grid_for(n), 256, 0, st>>>(deg.p, n, hs.max_out, sb.keys(), sb.vals());
        KERNEL_CHECK();
        sb.sort(n, ceil_log2_u64((u64)hs.max_out + 1), st, &g->pool);
        k_invert_perm<<<grid_for(n), 256, 0, st>>>(sb.vals(), n, g->old_of_new.p, g->new_of_old.p);
        KERNEL_CHECK();
        const u32 hot_min = g->opts.hot_min_degree > 0 ? (u32)g->opts.hot_min_degree : 8u;   // profiles/microbench/hotmin_sweep.py
        if (hot_min > 1) {
            DevBuf<u32> counts, pos;
            counts.alloc(2); pos.alloc(n);
            CUDA_CHECK(cudaMemsetAsync(counts.p, 0, 2 * sizeof(u32), st));
            k_cold_flags<<<grid_for(n), 256, 0, st>>>(deg.p, n, hot_min, pos.p, counts.p);
            KERNEL_CHECK();
            u32 hc[2] = {0, 0};
            CUDA_CHECK(cudaMemcpyAsync(hc, counts.p, sizeof(hc), cudaMemcpyDeviceToHost, st));   // complete once the scan returns
            const u32 n_cold = prim::scan_total<u32>(pos.p, pos.p, n, false, st, &g->pool);
            const u32 n_hot = hc[0];
            g->n_hot = (int32_t)n_hot;
            if (n_cold) {
                prim::SortBuffers<u32> cold;
                cold.alloc(n_cold, true);
                k_cold_keys<<<grid_for(n), 256, 0, st>>>(deg.p, first_nb.p, g->new_of_old.p, n, hot_min, n_hot, pos.p, cold.keys(),
                                                         cold.vals());
                KERNEL_CHECK();
                cold.sort(n_cold, ceil_log2_u64((u64)n_hot + (u64)n + 1), st, &g->pool);
                k_assign_cold<<<grid_for(n_cold), 256, 0, st>>>(cold.vals(), n_cold, n_hot, g->new_of_old.p, g->old_of_new.p);
                KERNEL_CHECK();
            }
        }
        CUDA_CHECK(cudaStreamSynchronize(st));
    } else if (n) {
        k_identity_perm<<<grid_for(n), 256, 0, st>>>(n, g->old_of_new.p, g->new_of_old.p);
        KERNEL_CHECK();
    }

    trace.mark("relabel");
    // ---- row-partitioned graph: deal the label order over the slices (see k_deal_labels)
    {
        const int parts = dist_n_ranks(g->comm);
        if (parts > 1 && n > 0) {
            if (parts > 16) RWR_FAIL(RWR_E_UNSUPPORTED, "more than 16 ranks");
            const int32_t n_hot = g->relabelled ? g->n_hot : n;       // without a relabel every position is dealt singly
            DealPlan plan;
            int32_t cold_of[16];
            const char* eb = getenv("RWR_DEAL_BLOCK");
            plan.block = eb ? std::max(1, atoi(eb)) : DEAL_BLOCK;
            const int32_t n_cold = n - n_hot, full_blocks = n_cold / plan.block, tail = n_cold % plan.block;
            for (int r = 0; r < parts; r++) {
                plan.hot_of[r] = n_hot / parts + (r < n_hot % parts ? 1 : 0);
                cold_of[r] = (full_blocks / parts + (r < full_blocks % parts ? 1 : 0)) * plan.block;
            }
            cold_of[full_blocks % parts] += tail;                      // the partial last block goes to the next slice in turn
            plan.start[0] = 0;
            for (int r = 0; r < parts; r++) plan.start[r + 1] = plan.start[r] + plan.hot_of[r] + cold_of[r];
            g->n_hot = n;                             // hotness is no longer a label prefix
            DevBuf<int32_t> tmp;
            tmp.alloc(n);
            CUDA_CHECK(cudaMemcpyAsync(tmp.p, g->old_of_new.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
            k_deal_labels<<<grid_for(n), 256, 0, st>>>(tmp.p, n, n_hot, parts, plan, g->old_of_new.p, g->new_of_old.p);
            KERNEL_CHECK();
            CUDA_CHECK(cudaStreamSynchronize(st));
            g->deal_rows.assign(plan.start, plan.start + parts + 1);
            g->part_hot.assign(plan.hot_of, plan.hot_of + parts);
            // ownership boundaries: the deal's, rounded down to 32 labels, so that a 128-byte line of x (32 floats, 16
            // doubles) belongs to ONE rank -- the overlapped exchange lets a rank gather from a slice while its neighbour's
            // slice is still arriving, and a line that spans both would be cached half stale
            g->part_rows.assign(plan.start, plan.start + parts + 1);
            for (int r = 1; r < parts; r++) g->part_rows[r] &= ~31;
        }
    }

    trace.mark("deal labels");
    // ---- K5: transpose to the pull layout with a stable sort keyed by the (relabelled) target
    g->in_ptr.alloc((size_t)n + 1, &g->pool);
    if (!pb) {
        g->nnz_in = (int64_t)nnz;
        g->in_src.alloc(nnz + IDX_PAD, &g->pool);
        CUDA_CHECK(cudaMemsetAsync(g->in_src.p, 0, (nnz + IDX_PAD) * sizeof(int32_t), st));
        if (layout == RWR_LAYOUT_VALUED) g->in_val64.alloc(nnz + IDX_PAD, &g->pool);   // k_spmm reads whole groups of 4
        prim::SortBuffers<u32> sb;
        sb.alloc(nnz, true);
        if (nnz) {
            k_transpose_keys<<<grid_for(nnz), 256, 0, st>>>(g->col, g->new_of_old.p, nnz, sb.keys(), sb.vals());
            KERNEL_CHECK();
        }
        sb.sort(nnz, ceil_log2_u64((u64)n), st, &g->pool);
        k_lower_bounds<u32><<<grid_for((size_t)n + 1), 256, 0, st>>>(sb.keys(), nnz, n, g->in_ptr.p);
        if (nnz)
            k_fill_pull<<<grid_for(nnz), 256, 0, st>>>(sb.vals(), g->src_of, g->new_of_old.p, g->val.p, nnz, g->in_src.p,
                                                      layout == RWR_LAYOUT_VALUED ? g->in_val64.p : nullptr);
        KERNEL_CHECK();
        CUDA_CHECK(cudaStreamSynchronize(st));
    } else {
        // Partitioned build: this rank holds the links of the SOURCES it owns and needs the links of the TARGET rows it
        // owns.  Links are bucketed by the rank of their target (one stable 3-bit pass), travel as (target label, original
        // source id [, weight]) through one grouped all-to-all, and are put into (target, original source, insertion) order
        // on arrival -- the accumulation order of the reference's push loop (Model.cs:80-88: i ascending).
        const int parts = dist_n_ranks(g->comm);
        const bool valued = layout == RWR_LAYOUT_VALUED;
        DevBuf<int> d_rows;
        DevBuf<u32> d_cnt;
        d_rows.alloc(parts + 1); d_cnt.alloc(16);
        CUDA_CHECK(cudaMemcpyAsync(d_rows.p, g->part_rows.data(), (size_t)(parts + 1) * sizeof(int), cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(d_cnt.p, 0, 16 * sizeof(u32), st));
        DevBuf<uint2> send_pairs;
        DevBuf<double> send_val;
        send_pairs.alloc(nnz);
        if (valued) send_val.alloc(nnz);
        {
            prim::SortBuffers<u32> sb;
            sb.alloc(nnz, true);
            if (nnz) {
                k_dest_keys<<<grid_for(nnz), 256, 0, st>>>(g->col, g->new_of_old.p, nnz, parts, d_rows.p, sb.keys(), sb.vals(), d_cnt.p);
                KERNEL_CHECK();
            }
            sb.sort(nnz, std::max(1, ceil_log2_u64((u64)parts)), st, &g->pool);
            if (nnz) {
                k_pack_links<<<grid_for(nnz), 256, 0, st>>>(sb.vals(), g->col, g->src_of, g->new_of_old.p, g->val.p, nnz,
                                                           send_pairs.p, valued ? send_val.p : nullptr);
                KERNEL_CHECK();
            }
            CUDA_CHECK(cudaStreamSynchronize(st));
        }
        trace.mark("K5 bucket by target rank");
        // counts matrix: every rank learns how many links it receives from every other rank
        std::vector<u32> h_send(16, 0);
        CUDA_CHECK(cudaMemcpyAsync(h_send.data(), d_cnt.p, 16 * sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        DevBuf<int64_t> d_mat;
        d_mat.alloc((size_t)parts * parts);
        std::vector<int64_t> h_mat((size_t)parts * parts, 0);
        const int me = dist_rank(g->comm);
        for (int d = 0; d < parts; d++) h_mat[(size_t)me * parts + d] = (int64_t)h_send[d];
        CUDA_CHECK(cudaMemcpyAsync(d_mat.p, h_mat.data(), h_mat.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        dist_allreduce_sum(g, d_mat.p, h_mat.size(), DIST_I64);
        CUDA_CHECK(cudaMemcpyAsync(h_mat.data(), d_mat.p, h_mat.size() * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        std::vector<size_t> s_off(parts), s_cnt(parts), r_off(parts), r_cnt(parts);
        size_t so = 0, ro = 0;
        for (int r = 0; r < parts; r++) {
            s_off[r] = so; s_cnt[r] = (size_t)h_mat[(size_t)me * parts + r]; so += s_cnt[r];
            r_off[r] = ro; r_cnt[r] = (size_t)h_mat[(size_t)r * parts + me]; ro += r_cnt[r];
        }
        const size_t m = ro;
        if (m + (size_t)n + WS_PAD_LINKS >= (1ull << 32)) RWR_FAIL(RWR_E_UNSUPPORTED, "more than 2^32 links in one rank's slice");
        DevBuf<uint2> recv_pairs;
        DevBuf<double> recv_val;
        recv_pairs.alloc(m);
        if (valued) recv_val.alloc(m);
        dist_alltoallv(g, send_pairs.p, s_off.data(), s_cnt.data(), recv_pairs.p, r_off.data(), r_cnt.data(), sizeof(uint2));
        if (valued) dist_alltoallv(g, send_val.p, s_off.data(), s_cnt.data(), recv_val.p, r_off.data(), r_cnt.data(), sizeof(double));
        CUDA_CHECK(cudaStreamSynchronize(st));
        send_pairs.release();
        send_val.release();
        trace.mark("K5 all-to-all");
        // (target label, original source, arrival) order: LSD, source id first, then a stable pass by target
        g->nnz_in = (int64_t)m;
        g->in_src.alloc(m + IDX_PAD, &g->pool);
        CUDA_CHECK(cudaMemsetAsync(g->in_src.p, 0, (m + IDX_PAD) * sizeof(int32_t), st));
        if (valued) g->in_val64.alloc(m + IDX_PAD, &g->pool);
        {
            prim::SortBuffers<u32> sb;
            sb.alloc(m, true);
            if (m) k_pair_field<<<grid_for(m), 256, 0, st>>>(recv_pairs.p, nullptr, m, 1, sb.keys(), sb.vals());
            KERNEL_CHECK();
            sb.sort(m, ceil_log2_u64((u64)n), st, &g->pool);
            u32* target_keys = sb.rekey();
            if (m) k_pair_field<<<grid_for(m), 256, 0, st>>>(recv_pairs.p, sb.vals(), m, 0, target_keys, nullptr);
            KERNEL_CHECK();
            sb.sort(m, ceil_log2_u64((u64)n), st, &g->pool);
            k_lower_bounds<u32><<<grid_for((size_t)n + 1), 256, 0, st>>>(sb.keys(), m, n, g->in_ptr.p);
            if (m)
                k_fill_pull_recv<<<grid_for(m), 256, 0, st>>>(sb.vals(), recv_pairs.p, valued ? recv_val.p : nullptr, g->new_of_old.p, m,
                                                             g->in_src.p, valued ? g->in_val64.p : nullptr);
            KERNEL_CHECK();
            CUDA_CHECK(cudaStreamSynchronize(st));
        }
    }

    trace.mark("K5 sort + pull arrays");
    // ---- per-node arrays in internal labels
    g->inv_orig.alloc(n, &g->pool);
    g->inv64.alloc(n, &g->pool);
    g->node_id_int.alloc(n, &g->pool);
    g->node_type_int.alloc(n, &g->pool);
    if (n) {
        k_node_arrays<<<grid_for(n), 256, 0, st>>>(g->old_of_new.p, deg.p, w0.p, g->node_id.p,
                                                   g->node_type.p, n, layout == RWR_LAYOUT_INDEX, g->in_ptr.p,
                                                   g->inv_orig.p, g->inv64.p, g->node_id_int.p, g->node_type_int.p, stats.p);
        KERNEL_CHECK();
    }
    CUDA_CHECK(cudaMemcpyAsync(&hs, stats.p, sizeof(hs), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    g->max_in_degree = hs.max_in;
    g->n_items = hs.n_items;

    trace.mark("node arrays");
    iterate_prepare(g);
    trace.mark("edge stream");
    dist_setup_p2p(g);
    trace.mark("peer mapping");

    CUDA_CHECK(cudaEventRecord(ev.b, st));
    CUDA_CHECK(cudaEventSynchronize(ev.b));
    CUDA_CHECK(cudaEventElapsedTime(&g->build_ms, ev.a, ev.b));
    g->built = true;
}

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

int rwr_graph_create_flat(int32_t n_nodes, const int64_t* node_id, const int32_t* node_type, int64_t n_links,
                          const int32_t* src, const int32_t* dst, const int32_t* etype, const double* w,
                          const rwr_opts* opts, rwr_comm* comm, rwr_graph** out);

int rwr_graph_create(int32_t n_nodes, const int64_t* node_id, const int32_t* node_type, int64_t n_links,
                     const int32_t* src, const int32_t* dst, const int32_t* etype, const double* w,
                     const rwr_opts* opts, rwr_graph** out) {
    return rwr_graph_create_flat(n_nodes, node_id, node_type, n_links, src, dst, etype, w, opts, nullptr, out);
}

// shared by rwr_graph_create and rwr_graph_create_partitioned (dist.cu): `comm` marks a row-partitioned graph
int rwr_graph_create_flat(int32_t n_nodes, const int64_t* node_id, const int32_t* node_type, int64_t n_links,
                          const int32_t* src, const int32_t* dst, const int32_t* etype, const double* w,
                          const rwr_opts* opts, rwr_comm* comm, rwr_graph** out) {
    rwr_graph* g = nullptr;
    RWR_API_BEGIN
    if (!out) RWR_FAIL(RWR_E_INVALID, "out is NULL");
    *out = nullptr;
    if (n_nodes < 0 || n_links < 0) RWR_FAIL(RWR_E_INVALID, "negative size");
    if ((n_nodes && (!node_id || !node_type)) || (n_links && (!src || !dst || !etype || !w)))
        RWR_FAIL(RWR_E_INVALID, "NULL input array");
    if ((u64)n_nodes >= (1ULL << 28)) RWR_FAIL(RWR_E_UNSUPPORTED, "more than 2^28-1 nodes");
    if ((u64)n_links >= (1ULL << 32) - 65536) RWR_FAIL(RWR_E_UNSUPPORTED, "more than 2^32-65537 links per device");
    g = new rwr_graph();
    graph_init_device(g, opts);
    g->comm = comm;
    cudaStream_t st = g->stream;
    AllocStream alloc_on(st);
    g->n = n_nodes;
    // Partitioned build: every rank is handed the same link list and uploads only the links of the sources it owns
    // (contiguous pieces of the node range), in their given order
    std::vector<int32_t> f_src, f_dst, f_et;
    std::vector<double> f_w;
    g->part_build = comm && dist_n_ranks(comm) > 1 && !dist_is_fake(comm) && !getenv("RWR_PART_REPLICATED");
    if (g->part_build) {
        OwnMap& own = g->own;
        own.parts = dist_n_ranks(comm); own.rank = dist_rank(comm); own.n_segs = 1;
        own.seg[0] = 0; own.seg[1] = std::max(1, n_nodes);
        for (int64_t i = 0; i < n_links; i++) {
            if (src[i] < 0 || src[i] >= n_nodes) RWR_FAIL(RWR_E_BADINDEX, "link source outside [0, %d)", n_nodes);
            if (own_rank(own, src[i]) != own.rank) continue;
            f_src.push_back(src[i]); f_dst.push_back(dst[i]); f_et.push_back(etype[i]); f_w.push_back(w[i]);
        }
        n_links = (int64_t)f_src.size();
        src = f_src.data(); dst = f_dst.data(); etype = f_et.data(); w = f_w.data();
    }
    g->e0 = n_links;
    const size_t n = (size_t)n_nodes, e0 = (size_t)n_links;
    g->node_id.alloc(n, &g->pool);
    g->node_type.alloc(n, &g->pool);
    g->raw_src.alloc(e0, &g->pool);
    g->raw_dst.alloc(e0, &g->pool);
    g->raw_type.alloc(e0, &g->pool);
    g->raw_w.alloc(e0, &g->pool);
    DevBuf<int32_t> tmp;
    tmp.alloc(std::max(n, e0));
    DevBuf<int> bad;
    bad.alloc(1);
    CUDA_CHECK(cudaMemsetAsync(bad.p, 0, sizeof(int), st));
    if (n) {
        CUDA_CHECK(cudaMemcpyAsync(g->node_id.p, node_id, n * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(tmp.p, node_type, n * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        k_i32_to_u8<<<grid_for(n), 256, 0, st>>>(tmp.p, g->node_type.p, n, bad.p);
        KERNEL_CHECK();
    }
    if (e0) {
        CUDA_CHECK(cudaMemcpyAsync(g->raw_src.p, src, e0 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(g->raw_dst.p, dst, e0 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(g->raw_w.p, w, e0 * sizeof(double), cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaStreamSynchronize(st));   // tmp is reused
        CUDA_CHECK(cudaMemcpyAsync(tmp.p, etype, e0 * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        k_i32_to_u8<<<grid_for(e0), 256, 0, st>>>(tmp.p, g->raw_type.p, e0, bad.p);
        KERNEL_CHECK();
    }
    int h_bad = 0;
    CUDA_CHECK(cudaMemcpyAsync(&h_bad, bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    if (h_bad) RWR_FAIL(RWR_E_INVALID, "node_type / etype value outside 0..255");
    graph_finish_create(g);
    *out = g;
    return RWR_OK;
    }
    catch (const RwrError& e__) { rwr_graph_destroy(g); return e__.code; }
    catch (const std::bad_alloc&) { rwr_graph_destroy(g); rwr_set_error("host allocation failed"); return RWR_E_OOM; }
    catch (...) { rwr_graph_destroy(g); rwr_set_error("unexpected exception"); return RWR_E_INVALID; }
}

int rwr_graph_build(rwr_graph* g) {
    RWR_API_BEGIN
    if (!g) RWR_FAIL(RWR_E_INVALID, "graph is NULL");
    graph_build_impl(g);
    return RWR_OK;
    RWR_API_END
}

int rwr_graph_get_info(rwr_graph* g, rwr_graph_info* info) {
    RWR_API_BEGIN
    if (!g || !info) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    memset(info, 0, sizeof(*info));
    info->n_nodes = g->n;
    info->built = g->built ? 1 : 0;
    info->n_links_raw = g->e0;          // a partitioned build: the links of the sources this rank owns
    info->nnz = g->built ? (g->part_build ? g->nnz_global : g->nnz) : 0;
    info->n_dangling = g->n_dangling;
    info->layout = g->built ? g->layout : 0;
    info->relabelled = g->relabelled ? 1 : 0;
    info->n_hot = g->n_hot;
    info->hub_entries_fp64 = g->built ? ws_hub_entries(g, RWR_FP64) : 0;
    info->hub_entries_fp32 = g->built ? ws_hub_entries(g, RWR_FP32) : 0;
    info->n_chunks = g->n_chunks;
    info->row_begin = g->row_begin;
    info->row_end = g->built ? g->row_end : 0;
    info->n_ranks = g->part_rows.empty() ? 1 : (int32_t)g->part_rows.size() - 1;
    info->x_blocks = g->x_blocks;
    info->max_in_degree = (int32_t)g->max_in_degree;
    info->max_out_degree = (int32_t)g->max_out_degree;
    info->build_ms = g->build_ms;
    info->synth_ms = g->synth_ms;
    info->device_bytes = g->pool.bytes;
    return RWR_OK;
    RWR_API_END
}

int rwr_graph_export_links(rwr_graph* g, int64_t* node_id, int32_t* node_type, int32_t* src, int32_t* dst,
                           int32_t* etype, double* w) {
    RWR_API_BEGIN
    if (!g) RWR_FAIL(RWR_E_INVALID, "graph is NULL");
    CUDA_CHECK(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    const size_t n = (size_t)g->n, e0 = (size_t)g->e0;
    if (node_id && n) CUDA_CHECK(cudaMemcpyAsync(node_id, g->node_id.p, n * 8, cudaMemcpyDeviceToHost, st));
    if (src && e0) CUDA_CHECK(cudaMemcpyAsync(src, g->raw_src.p, e0 * 4, cudaMemcpyDeviceToHost, st));
    if (dst && e0) CUDA_CHECK(cudaMemcpyAsync(dst, g->raw_dst.p, e0 * 4, cudaMemcpyDeviceToHost, st));
    if (w && e0) CUDA_CHECK(cudaMemcpyAsync(w, g->raw_w.p, e0 * 8, cudaMemcpyDeviceToHost, st));
    std::vector<u8> t8;
    if (node_type && n) {
        t8.resize(n);
        CUDA_CHECK(cudaMemcpyAsync(t8.data(), g->node_type.p, n, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (size_t i = 0; i < n; i++) node_type[i] = t8[i];
    }
    if (etype && e0) {
        t8.resize(e0);
        CUDA_CHECK(cudaMemcpyAsync(t8.data(), g->raw_type.p, e0, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (size_t i = 0; i < e0; i++) etype[i] = t8[i];
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
    return RWR_OK;
    RWR_API_END
}

int rwr_graph_get_csr(rwr_graph* g, int64_t* row_ptr, int32_t* col, double* val) {
    RWR_API_BEGIN
    if (!g) RWR_FAIL(RWR_E_INVALID, "graph is NULL");
    if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
    if (g->part_build) RWR_FAIL(RWR_E_UNSUPPORTED, "row-partitioned handle: every rank holds the rows of W of the sources it owns only");
    CUDA_CHECK(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    const size_t n = (size_t)g->n, nnz = (size_t)g->nnz;
    if (col && nnz) CUDA_CHECK(cudaMemcpyAsync(col, g->col, nnz * 4, cudaMemcpyDeviceToHost, st));
    if (val && nnz) CUDA_CHECK(cudaMemcpyAsync(val, g->val.p, nnz * 8, cudaMemcpyDeviceToHost, st));
    if (row_ptr) {
        std::vector<u32> rp(n + 1);
        CUDA_CHECK(cudaMemcpyAsync(rp.data(), g->row_ptr, (n + 1) * 4, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (size_t i = 0; i <= n; i++) row_ptr[i] = (int64_t)rp[i];
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
    return RWR_OK;
    RWR_API_END
}

int rwr_graph_get_csr_types(rwr_graph* g, int32_t* etype) {
    RWR_API_BEGIN
    if (!g || !etype) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
    if (g->part_build) RWR_FAIL(RWR_E_UNSUPPORTED, "row-partitioned handle: every rank holds the rows of W of the sources it owns only");
    CUDA_CHECK(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    AllocStream alloc_on(st);
    const size_t e0 = (size_t)g->e0, nnz = (size_t)g->nnz;
    if (nnz == 0) return RWR_OK;
    DevBuf<u32> pos;
    DevBuf<int> bad;
    DevBuf<int32_t> out;
    pos.alloc(e0); bad.alloc(1); out.alloc(nnz);
    DevBuf<u8> carrier;
    const u32 zero_mask = (u32)g->opts.zero_weight_type_mask;
    if (zero_mask) {
        carrier.alloc((size_t)std::max(g->n, 1));
        CUDA_CHECK(cudaMemsetAsync(carrier.p, 0, (size_t)std::max(g->n, 1), st));
        k_carrier_flags<<<grid_for(e0), 256, 0, st>>>(g->raw_type.p, g->raw_src.p, e0, g->n, (u32)g->opts.undefined_type_mask, zero_mask,
                                                     carrier.p);
    }
    k_explicit_flags<<<grid_for(e0), 256, 0, st>>>(g->raw_type.p, g->raw_src.p, g->raw_dst.p, e0, g->n, (u32)g->opts.undefined_type_mask,
                                                  zero_mask, carrier.p, pos.p, bad.p);
    KERNEL_CHECK();
    prim::exclusive_scan<u32>(pos.p, pos.p, e0, nullptr, st, &g->pool);
    k_compact_types<<<grid_for(e0), 256, 0, st>>>(g->raw_type.p, g->raw_src.p, pos.p, e0, (u32)g->opts.undefined_type_mask, zero_mask,
                                                 carrier.p, out.p);
    KERNEL_CHECK();
    CUDA_CHECK(cudaMemcpyAsync(etype, out.p, nnz * 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    return RWR_OK;
    RWR_API_END
}

int rwr_graph_get_degrees(rwr_graph* g, int32_t* out_degree, int32_t* raw_degree) {
    RWR_API_BEGIN
    if (!g) RWR_FAIL(RWR_E_INVALID, "graph is NULL");
    CUDA_CHECK(cudaSetDevice(g->device));
    const size_t n = (size_t)g->n;
    std::vector<u32> rp(n + 1);
    if (g->part_build) {
        // every rank holds the links of its own sources only: the per-node counts are summed over the ranks (collective call)
        AllocStream alloc_on(g->stream);
        DevBuf<u32> d;
        d.alloc(n + 1);
        std::vector<u32> h(n);
        for (int which = 0; which < 2; which++) {
            int32_t* out = which ? raw_degree : out_degree;
            if (!out) continue;
            if (!which && !g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
            if (n) k_ptr_diff<<<grid_for(n), 256, 0, g->stream>>>(which ? g->raw_ptr.p : g->row_ptr, (int32_t)n, d.p);
            KERNEL_CHECK();
            dist_allreduce_sum(g, d.p, n, DIST_U32);
            CUDA_CHECK(cudaMemcpyAsync(h.data(), d.p, n * 4, cudaMemcpyDeviceToHost, g->stream));
            CUDA_CHECK(cudaStreamSynchronize(g->stream));
            for (size_t i = 0; i < n; i++) out[i] = (int32_t)h[i];
        }
        return RWR_OK;
    }
    if (out_degree) {
        if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
        CUDA_CHECK(cudaMemcpyAsync(rp.data(), g->row_ptr, (n + 1) * 4, cudaMemcpyDeviceToHost, g->stream));
        CUDA_CHECK(cudaStreamSynchronize(g->stream));
        for (size_t i = 0; i < n; i++) out_degree[i] = (int32_t)(rp[i + 1] - rp[i]);
    }
    if (raw_degree) {
        CUDA_CHECK(cudaMemcpyAsync(rp.data(), g->raw_ptr.p, (n + 1) * 4, cudaMemcpyDeviceToHost, g->stream));
        CUDA_CHECK(cudaStreamSynchronize(g->stream));
        for (size_t i = 0; i < n; i++) raw_degree[i] = (int32_t)(rp[i + 1] - rp[i]);
    }
    return RWR_OK;
    RWR_API_END
}

void rwr_graph_destroy(rwr_graph* g) {
    if (!g) return;
    cudaSetDevice(g->device);
    if (g->stream) cudaStreamSynchronize(g->stream);
    dist_release_p2p(g);
    for (auto& ig : g->iter_graph) if (ig.exec) cudaGraphExecDestroy(ig.exec);
    const cudaStream_t st = g->stream;
    const bool own = g->own_stream;
    delete g;                                    // the buffers go back to the pool on the stream ...
    if (st) cudaStreamSynchronize(st);
    if (own && st) cudaStreamDestroy(st);        // ... which is destroyed last
}

}  // extern "C"
