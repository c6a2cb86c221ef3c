// select.cu -- per-seed candidate filtering, top-k (K9) and full ranking.
//
// Restates Recommenders/RWRBased/Recommender.cs:
//   :19-24  exclusion list = targets of the seed's raw LIKE links            -> k_mark_excluded (bitmap)
//           (a restart set: the union over its nodes)                        -> k_mark_excluded_set
//   :27-31  candidates = ITEM nodes not excluded, as (node.id, rank[i])       -> filter inside the scan
//   :34-38  order by score descending, ties by id descending                 -> 64-bit order-preserving score key, id
//   :42-51  first topN of that order                                         -> k_topk_scan + k_topk_merge (k <= 16)
//   :14-40  the full ranking (what Experiment.cs:121-128 walks)               -> stable LSD radix sort over items that
//                                                                               are pre-ordered by id descending
#include <algorithm>
#include <unordered_set>

#include "dist.h"
#include "iterate.h"
#include "primitives.cuh"

constexpr int TOPK_MAX = 16;
constexpr int TOPK_THREADS = 256;

struct Cand {
    u64 key;       // order-preserving image of the score (NaN lowest, like System.Double.CompareTo)
    int64_t id;
    int idx;       // internal node index, -1: empty
};

__device__ __forceinline__ u64 score_key(double s) {
    if (s != s) return 0ULL;                         // NaN sorts below everything
    if (s == 0.0) s = 0.0;                           // -0.0 == +0.0 for CompareTo
    const u64 b = (u64)__double_as_longlong(s);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}

__device__ __forceinline__ bool better(const Cand& a, const Cand& b) {   // a ranks before b
    if (a.idx < 0) return false;
    if (b.idx < 0) return true;
    if (a.key != b.key) return a.key > b.key;
    return a.id > b.id;
}

__device__ __forceinline__ void list_insert(Cand (&list)[TOPK_MAX], const Cand& c) {
    if (!better(c, list[TOPK_MAX - 1])) return;
    list[TOPK_MAX - 1] = c;
#pragma unroll
    for (int i = TOPK_MAX - 1; i > 0; i--) {
        if (better(list[i], list[i - 1])) {
            Cand t = list[i]; list[i] = list[i - 1]; list[i - 1] = t;
        }
    }
}

__device__ __forceinline__ Cand cand_shfl_down(const Cand& c, int o) {
    Cand r;
    r.key = __shfl_down_sync(0xffffffffu, c.key, o);
    r.id = __shfl_down_sync(0xffffffffu, c.id, o);
    r.idx = __shfl_down_sync(0xffffffffu, c.idx, o);
    return r;
}

// k rounds of block-wide arg-best over the heads of the per-thread sorted lists; winners go to out[0..k)
__device__ void block_extract(Cand (&list)[TOPK_MAX], int k, Cand* out, Cand* sm_best /*[warps]*/, int* sm_owner /*[warps+1]*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int round = 0; round < k; round++) {
        Cand best = list[0];
        int owner = threadIdx.x;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            Cand other = cand_shfl_down(best, o);
            int oo = __shfl_down_sync(0xffffffffu, owner, o);
            if (better(other, best)) { best = other; owner = oo; }
        }
        if (lane == 0) { sm_best[warp] = best; sm_owner[warp] = owner; }
        __syncthreads();
        if (threadIdx.x == 0) {
            Cand b = sm_best[0];
            int ow = sm_owner[0];
            for (int w = 1; w < TOPK_THREADS / 32; w++)
                if (better(sm_best[w], b)) { b = sm_best[w]; ow = sm_owner[w]; }
            out[round] = b;
            sm_owner[TOPK_THREADS / 32] = (b.idx < 0) ? -1 : ow;
        }
        __syncthreads();
        const int win = sm_owner[TOPK_THREADS / 32];
        if (win == (int)threadIdx.x) {
#pragma unroll
            for (int i = 0; i < TOPK_MAX - 1; i++) list[i] = list[i + 1];
            list[TOPK_MAX - 1].idx = -1;
        }
        __syncthreads();
    }
}

// Pass 1 of the top-k: the best candidate key of every block's share.  The k-th largest of these block maxima is a
// lower bound of the k-th best score overall (k distinct candidates reach it), so pass 2 only has to look at the few
// candidates at or above it -- exact, and on the skewed score vectors of a random walk it skips almost everything.
constexpr int TOPK_MAX_GRID = 1024;
template <typename T>
__global__ void __launch_bounds__(TOPK_THREADS) k_topk_bound(const T* __restrict__ y, int ld, const u8* __restrict__ type_int,
                                                             const u32* __restrict__ excl, int n, u64* __restrict__ block_max) {
    __shared__ u64 sm[TOPK_THREADS / 32];
    u64 best = 0;
    for (int j = blockIdx.x * TOPK_THREADS + threadIdx.x; j < n; j += gridDim.x * TOPK_THREADS) {
        if (type_int[j] != RWR_NODE_ITEM) continue;
        if ((excl[j >> 5] >> (j & 31)) & 1u) continue;
        const u64 key = score_key((double)y[(size_t)j * ld]);
        best = key > best ? key : best;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { const u64 t = __shfl_xor_sync(0xffffffffu, best, o); best = t > best ? t : best; }
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < TOPK_THREADS / 32; w++) best = sm[w] > best ? sm[w] : best;
        block_max[blockIdx.x] = best;
    }
}

// y is read with a stride of `ld` elements: ld == 1 for one rank vector, ld == B for a column of a row-major tile
template <typename T>
__global__ void __launch_bounds__(TOPK_THREADS) k_topk_scan(const T* __restrict__ y, int ld, const u8* __restrict__ type_int,
                                                            const int64_t* __restrict__ id_int, const u32* __restrict__ excl,
                                                            int n, int k, const u64* __restrict__ block_max,
                                                            Cand* __restrict__ block_out) {
    __shared__ Cand sm_best[TOPK_THREADS / 32];
    __shared__ int sm_owner[TOPK_THREADS / 32 + 1];
    __shared__ u64 sm_max[TOPK_MAX_GRID];
    __shared__ u64 sm_bound;
    // the k-th largest block maximum (rank counting, ties by index); 0 == no bound when there are fewer than k blocks
    const int nb = (int)gridDim.x;
    for (int i = threadIdx.x; i < nb; i += TOPK_THREADS) sm_max[i] = block_max[i];
    if (threadIdx.x == 0) sm_bound = 0;
    __syncthreads();
    if (nb >= k) {
        for (int i = threadIdx.x; i < nb; i += TOPK_THREADS) {
            const u64 v = sm_max[i];
            int rank = 0;
            for (int j = 0; j < nb; j++) rank += (sm_max[j] > v) || (sm_max[j] == v && j < i);
            if (rank == k - 1) sm_bound = v;
        }
    }
    __syncthreads();
    const u64 bound = sm_bound;
    Cand list[TOPK_MAX];
#pragma unroll
    for (int i = 0; i < TOPK_MAX; i++) { list[i].key = 0; list[i].id = 0; list[i].idx = -1; }
    for (int j = blockIdx.x * TOPK_THREADS + threadIdx.x; j < n; j += gridDim.x * TOPK_THREADS) {
        if (type_int[j] != RWR_NODE_ITEM) continue;
        Cand c;
        c.key = score_key((double)y[(size_t)j * ld]);
        if (c.key < bound) continue;
        if ((excl[j >> 5] >> (j & 31)) & 1u) continue;
        c.idx = j;
        const Cand& worst = list[TOPK_MAX - 1];
        if (worst.idx >= 0 && c.key < worst.key) continue;       // cheap reject before touching the id
        c.id = id_int[j];
        list_insert(list, c);
    }
    block_extract(list, k, block_out + (size_t)blockIdx.x * k, sm_best, sm_owner);
}

template <typename T>
__global__ void __launch_bounds__(TOPK_THREADS) k_topk_merge(const Cand* __restrict__ cands, int n_cands, int k,
                                                             const T* __restrict__ y, int ld, int64_t* __restrict__ out_ids,
                                                             double* __restrict__ out_scores, int* __restrict__ out_count) {
    __shared__ Cand sm_best[TOPK_THREADS / 32];
    __shared__ int sm_owner[TOPK_THREADS / 32 + 1];
    __shared__ Cand result[TOPK_MAX];
    Cand list[TOPK_MAX];
#pragma unroll
    for (int i = 0; i < TOPK_MAX; i++) { list[i].key = 0; list[i].id = 0; list[i].idx = -1; }
    for (int j = threadIdx.x; j < n_cands; j += TOPK_THREADS) {
        Cand c = cands[j];
        if (c.idx >= 0) list_insert(list, c);
    }
    block_extract(list, k, result, sm_best, sm_owner);
    __syncthreads();
    if (threadIdx.x == 0) {
        int cnt = 0;
        for (int i = 0; i < k; i++) {
            if (result[i].idx < 0) break;
            out_ids[i] = result[i].id;
            out_scores[i] = (double)y[(size_t)result[i].idx * ld];
            cnt++;
        }
        *out_count = cnt;
    }
}

// Recommender.cs:20-24 -- targets of the seed's RAW links of type LIKE (original labels -> internal bitmap)
__global__ void k_mark_excluded(const int32_t* __restrict__ raw_dst, const u8* __restrict__ raw_type, u32 begin, u32 end,
                                const int32_t* __restrict__ new_of_old, int n, u32* __restrict__ excl) {
    const u32 e = begin + blockIdx.x * blockDim.x + threadIdx.x;
    if (e < end && raw_type[e] == RWR_EDGE_LIKE) {
        const int32_t d = raw_dst[e];
        if (d >= 0 && d < n) {
            const int j = new_of_old[d];
            atomicOr(&excl[j >> 5], 1u << (j & 31));
        }
    }
}

// A restart set (rwr_run_*_restart): Recommender.cs:20-24 for each listed node, one warp per node -- the union of the
// targets of their raw LIKE links
__global__ void k_mark_excluded_set(const int32_t* __restrict__ raw_dst, const u8* __restrict__ raw_type, const u32* __restrict__ raw_ptr,
                                    const int32_t* __restrict__ nodes /* original labels */, int m, const int32_t* __restrict__ new_of_old,
                                    int n, u32* __restrict__ excl) {
    const int k = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (k >= m) return;
    const int node = nodes[k];
    const u32 b = raw_ptr[node], e = raw_ptr[node + 1];
    for (u32 i = b + lane; i < e; i += 32) {
        if (raw_type[i] == RWR_EDGE_LIKE) {
            const int32_t d = raw_dst[i];
            if (d >= 0 && d < n) {
                const int j = new_of_old[d];
                atomicOr(&excl[j >> 5], 1u << (j & 31));
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ top-k of a whole seed tile
// The batched path keeps the ranks of B seeds row-major, Y[n, B].  Scanning one column at a time reads every 32-byte
// sector of Y once per column and pass; these kernels handle all B columns of a row at once (coalesced), with the same
// exact scheme as k_topk_bound / k_topk_scan: per-column lower bound from block maxima, then only the candidates at or
// above the bound are kept -- here appended to a per-column list (they are few) that k_topk_merge reduces.
constexpr int TILE_MAXB = 16;
constexpr int TILE_CAND_CAP = 1 << 16;          // candidates kept per column; more (e.g. everything ties at 0) -> per-column path

__global__ void k_mark_excluded_tile(const int32_t* __restrict__ raw_dst, const u8* __restrict__ raw_type,
                                     const u32* __restrict__ raw_ptr, const int32_t* __restrict__ seeds /* original labels */,
                                     const int32_t* __restrict__ new_of_old, int n, size_t words, u32* __restrict__ excl,
                                     int* __restrict__ no_links) {
    const int col = blockIdx.y;
    const int seed = seeds[col];
    const u32 b = raw_ptr[seed], e = raw_ptr[seed + 1];
    if (b == e && blockIdx.x == 0 && threadIdx.x == 0) no_links[col] = 1;      // KeyNotFoundException, Recommender.cs:21
    u32* ex = excl + (size_t)col * words;
    for (u32 i = b + blockIdx.x * blockDim.x + threadIdx.x; i < e; i += gridDim.x * blockDim.x) {
        if (raw_type[i] == RWR_EDGE_LIKE) {
            const int32_t d = raw_dst[i];
            if (d >= 0 && d < n) {
                const int j = new_of_old[d];
                atomicOr(&ex[j >> 5], 1u << (j & 31));
            }
        }
    }
}

template <typename T, int B>
__global__ void __launch_bounds__(TOPK_THREADS) k_topk_bound_tile(const T* __restrict__ y, const u8* __restrict__ type_int,
                                                                  const u32* __restrict__ excl, size_t words, int n, int cols,
                                                                  u64* __restrict__ block_max /* [grid][B] */) {
    __shared__ u64 sm[TOPK_THREADS];
    const int col = threadIdx.x % B, rlane = threadIdx.x / B;
    constexpr int RPB = TOPK_THREADS / B;                    // rows per block step
    u64 best = 0;
    if (col < cols) {
        const u32* ex = excl + (size_t)col * words;
        for (int j = blockIdx.x * RPB + rlane; j < n; j += gridDim.x * RPB) {
            if (type_int[j] != RWR_NODE_ITEM) continue;
            const u64 key = score_key((double)y[(size_t)j * B + col]);
            if (key <= best) continue;
            if ((ex[j >> 5] >> (j & 31)) & 1u) continue;
            best = key;
        }
    }
    sm[threadIdx.x] = best;
    __syncthreads();
    if (threadIdx.x < B) {
        u64 m = 0;
        for (int i = threadIdx.x; i < TOPK_THREADS; i += B) m = sm[i] > m ? sm[i] : m;
        block_max[(size_t)blockIdx.x * B + threadIdx.x] = m;
    }
}

// k-th largest block maximum of every column (rank counting, ties by index); 0 when there are fewer than k blocks
template <int B>
__global__ void __launch_bounds__(TOPK_THREADS) k_topk_bounds_tile(const u64* __restrict__ block_max, int nb, int k,
                                                                   u64* __restrict__ bound /* [B] */) {
    __shared__ u64 sm[TOPK_MAX_GRID];
    const int col = blockIdx.x;
    for (int i = threadIdx.x; i < nb; i += TOPK_THREADS) sm[i] = block_max[(size_t)i * B + col];
    if (threadIdx.x == 0) bound[col] = 0;
    __syncthreads();
    if (nb < k) return;
    for (int i = threadIdx.x; i < nb; i += TOPK_THREADS) {
        const u64 v = sm[i];
        int rank = 0;
        for (int j = 0; j < nb; j++) rank += (sm[j] > v) || (sm[j] == v && j < i);
        if (rank == k - 1) bound[col] = v;
    }
}

template <typename T, int B>
__global__ void __launch_bounds__(TOPK_THREADS) k_topk_scan_tile(const T* __restrict__ y, const u8* __restrict__ type_int,
                                                                 const int64_t* __restrict__ id_int, const u32* __restrict__ excl,
                                                                 size_t words, int n, int cols, const u64* __restrict__ bound,
                                                                 Cand* __restrict__ cand /* [B][CAP] */, int* __restrict__ cnt) {
    const int col = threadIdx.x % B, rlane = threadIdx.x / B;
    constexpr int RPB = TOPK_THREADS / B;
    if (col >= cols) return;
    const u64 bd = bound[col];
    const u32* ex = excl + (size_t)col * words;
    for (int j = blockIdx.x * RPB + rlane; j < n; j += gridDim.x * RPB) {
        if (type_int[j] != RWR_NODE_ITEM) continue;
        const u64 key = score_key((double)y[(size_t)j * B + col]);
        if (key < bd) continue;
        if ((ex[j >> 5] >> (j & 31)) & 1u) continue;
        const int slot = atomicAdd(&cnt[col], 1);
        if (slot < TILE_CAND_CAP) {
            Cand c;
            c.key = key; c.id = id_int[j]; c.idx = j;
            cand[(size_t)col * TILE_CAND_CAP + slot] = c;
        }
    }
}

// one block per column: the k best of the column's candidate list
template <typename T>
__global__ void __launch_bounds__(TOPK_THREADS) k_topk_merge_tile(const Cand* __restrict__ cand, const int* __restrict__ cnt, int k,
                                                                  const T* __restrict__ y, int ld, int64_t* __restrict__ out_ids,
                                                                  double* __restrict__ out_scores, int* __restrict__ out_count) {
    __shared__ Cand sm_best[TOPK_THREADS / 32];
    __shared__ int sm_owner[TOPK_THREADS / 32 + 1];
    __shared__ Cand result[TOPK_MAX];
    const int col = blockIdx.x;
    const int n_cands = min(cnt[col], TILE_CAND_CAP);
    const Cand* cands = cand + (size_t)col * TILE_CAND_CAP;
    Cand list[TOPK_MAX];
#pragma unroll
    for (int i = 0; i < TOPK_MAX; i++) { list[i].key = 0; list[i].id = 0; list[i].idx = -1; }
    for (int j = threadIdx.x; j < n_cands; j += TOPK_THREADS) list_insert(list, cands[j]);
    block_extract(list, k, result, sm_best, sm_owner);
    __syncthreads();
    if (threadIdx.x == 0) {
        int c = 0;
        for (int i = 0; i < k; i++) {
            if (result[i].idx < 0) break;
            out_ids[(size_t)col * k + i] = result[i].id;
            out_scores[(size_t)col * k + i] = (double)y[(size_t)result[i].idx * ld + col];
            c++;
        }
        out_count[col] = c;
    }
}

__global__ void k_lookup(const int32_t* __restrict__ table, const int32_t* __restrict__ keys, int n, int32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = table[keys[i]];
}

// ---- full ranking helpers
__global__ void k_item_flags(const u8* __restrict__ type_int, int n, u32* __restrict__ flags) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) flags[j] = type_int[j] == RWR_NODE_ITEM;
}
__global__ void k_item_keys(const u8* __restrict__ type_int, const int64_t* __restrict__ id_int, const u32* __restrict__ pos,
                            int n, u64* __restrict__ keys, u32* __restrict__ vals) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n && type_int[j] == RWR_NODE_ITEM) {
        const u64 asc = (u64)id_int[j] ^ 0x8000000000000000ULL;   // signed order -> unsigned order
        keys[pos[j]] = ~asc;                                      // ascending sort == id descending
        vals[pos[j]] = (u32)j;
    }
}
__global__ void k_cand_flags(const int32_t* __restrict__ items, int n_items, const u32* __restrict__ excl, u32* __restrict__ flags) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_items) {
        const int j = items[p];
        flags[p] = !((excl[j >> 5] >> (j & 31)) & 1u);
    }
}
template <typename T>
__global__ void k_cand_keys(const int32_t* __restrict__ items, int n_items, const u32* __restrict__ excl,
                            const u32* __restrict__ pos, const T* __restrict__ y, u64* __restrict__ keys, u32* __restrict__ vals) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_items) {
        const int j = items[p];
        if (!((excl[j >> 5] >> (j & 31)) & 1u)) {
            keys[pos[p]] = ~score_key((double)y[j]);              // ascending sort == score descending
            vals[pos[p]] = (u32)j;
        }
    }
}
template <typename T>
__global__ void k_emit_ranking(const u32* __restrict__ order, size_t count, const T* __restrict__ y,
                               const int64_t* __restrict__ id_int, int64_t* __restrict__ ids, double* __restrict__ scores) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < count) {
        const u32 j = order[p];
        ids[p] = id_int[j];
        scores[p] = (double)y[j];
    }
}

// ------------------------------------------------------------------------------------------------ host side
static void seed_raw_range(rwr_graph* g, int seed, u32* begin, u32* end) {
    u32 rp[2];
    CUDA_CHECK(cudaMemcpyAsync(rp, g->raw_ptr.p + seed, 2 * sizeof(u32), cudaMemcpyDeviceToHost, g->stream));
    CUDA_CHECK(cudaStreamSynchronize(g->stream));
    *begin = rp[0];
    *end = rp[1];
}

static void mark_excluded(rwr_graph* g, int seed, u32* excl, size_t words) {
    if (seed == -1) RWR_FAIL(RWR_E_INVALID, "a uniform-restart Model (seed -1) has no target user: Recommendation() needs one (Recommender.cs:14)");
    if (seed < 0 || seed >= g->n) RWR_FAIL(RWR_E_BADSEED, "seed %d has no `edges` entry (KeyNotFoundException, Recommender.cs:21)", seed);
    u32 b, e;
    seed_raw_range(g, seed, &b, &e);
    if (g->part_build) {
        // the raw links of the seed live on the rank that owns it: that rank marks the bitmap (and, in the spare last word,
        // "the seed has links"), the others contribute zeros, one sum over the ranks gives everybody the same bitmap
        CUDA_CHECK(cudaMemsetAsync(excl, 0, words * sizeof(u32), g->stream));
        if (e > b) {
            k_mark_excluded<<<div_up(e - b, 256), 256, 0, g->stream>>>(g->raw_dst.p, g->raw_type.p, b, e, g->new_of_old.p, g->n, excl);
            KERNEL_CHECK();
            const u32 one = 1;
            CUDA_CHECK(cudaMemcpyAsync(excl + words - 1, &one, sizeof(u32), cudaMemcpyHostToDevice, g->stream));
        }
        dist_allreduce_sum(g, excl, words, DIST_U32);
        u32 has = 0;
        CUDA_CHECK(cudaMemcpyAsync(&has, excl + words - 1, sizeof(u32), cudaMemcpyDeviceToHost, g->stream));
        CUDA_CHECK(cudaMemsetAsync(excl + words - 1, 0, sizeof(u32), g->stream));
        CUDA_CHECK(cudaStreamSynchronize(g->stream));
        if (!has && !g->opts.empty_seed_ok)
            RWR_FAIL(RWR_E_BADSEED, "seed %d has no `edges` entry (KeyNotFoundException, Recommender.cs:21)", seed);
        g->pool.launches += 1;
        return;
    }
    if (b == e && !g->opts.empty_seed_ok) RWR_FAIL(RWR_E_BADSEED, "seed %d has no `edges` entry (KeyNotFoundException, Recommender.cs:21)", seed);
    CUDA_CHECK(cudaMemsetAsync(excl, 0, words * sizeof(u32), g->stream));
    if (e > b) k_mark_excluded<<<div_up(e - b, 256), 256, 0, g->stream>>>(g->raw_dst.p, g->raw_type.p, b, e, g->new_of_old.p, g->n, excl);
    KERNEL_CHECK();
    g->pool.launches += 1;
}

// the exclusion bitmap of a result: its seed's LIKE targets, or the union over the nodes of a restart set
static void mark_excluded_for(rwr_graph* g, const rwr_result* r, int slot, u32* excl, size_t words) {
    if (r->restart_nodes.empty()) { mark_excluded(g, r->seeds[slot], excl, words); return; }
    const int m = (int)r->restart_nodes.size();
    Scratch<int32_t> nodes;
    nodes.alloc(&g->scratch, m);
    CUDA_CHECK(cudaMemcpyAsync(nodes.p, r->restart_nodes.data(), (size_t)m * sizeof(int32_t), cudaMemcpyHostToDevice, g->stream));
    CUDA_CHECK(cudaMemsetAsync(excl, 0, words * sizeof(u32), g->stream));
    k_mark_excluded_set<<<div_up((size_t)m * 32, 256), 256, 0, g->stream>>>(g->raw_dst.p, g->raw_type.p, g->raw_ptr.p, nodes.p, m,
                                                                           g->new_of_old.p, g->n, excl);
    KERNEL_CHECK();
    CUDA_CHECK(cudaStreamSynchronize(g->stream));          // the host list is the caller's until the copy has run
    g->pool.launches += 1;
}

// blocks of the top-k scans over a rank vector or a seed tile
static int topk_grid(const rwr_graph* g) {
    return std::max(1, std::min(std::min(g->sm_count * 4, TOPK_MAX_GRID), (int)div_up((size_t)std::max(g->n, 1), TOPK_THREADS)));
}

// Scratch of the k <= 16 top-k of `lists` rank vectors: the exclusion bitmap and the block candidates serve one list after
// the other; the results of all lists are zeroed up front (the slots past a short list's count read 0) and go out together.
struct TopkScratch {
    const size_t words;         // exclusion bitmap, + 1 spare word (a partitioned build's "the seed has links" flag)
    const int grid, k, lists;
    Scratch<u32> excl;
    Scratch<Cand> block_out;
    Scratch<int64_t> ids;
    Scratch<double> scores;
    Scratch<int> counts;
    TopkScratch(rwr_graph* g, int k_, int lists_) : words(((size_t)g->n + 31) / 32 + 1), grid(topk_grid(g)), k(k_), lists(lists_) {
        excl.alloc(&g->scratch, words); block_out.alloc(&g->scratch, (size_t)grid * k);
        ids.alloc(&g->scratch, (size_t)lists * k); scores.alloc(&g->scratch, (size_t)lists * k); counts.alloc(&g->scratch, lists);
        CUDA_CHECK(cudaMemsetAsync(ids.p, 0, (size_t)lists * k * 8, g->stream));
        CUDA_CHECK(cudaMemsetAsync(scores.p, 0, (size_t)lists * k * 8, g->stream));
    }
    // enqueues the copies of every list's result; the caller synchronises
    void copy_out(cudaStream_t st, int64_t* out_ids, double* out_scores, int32_t* out_counts) const {
        CUDA_CHECK(cudaMemcpyAsync(out_ids, ids.p, (size_t)lists * k * 8, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(out_scores, scores.p, (size_t)lists * k * 8, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(out_counts, counts.p, (size_t)lists * 4, cudaMemcpyDeviceToHost, st));
    }
};

// top-k of the rank vector y (stride ld) into result `list` of ts
template <typename T>
static void topk_one(rwr_graph* g, TopkScratch& ts, int list, const T* y, int ld, int seed, bool marked = false) {
    if (!marked) mark_excluded(g, seed, ts.excl.p, ts.words);
    Scratch<u64> block_max;
    block_max.alloc(&g->scratch, (size_t)ts.grid);
    k_topk_bound<T><<<ts.grid, TOPK_THREADS, 0, g->stream>>>(y, ld, g->node_type_int.p, ts.excl.p, g->n, block_max.p);
    k_topk_scan<T><<<ts.grid, TOPK_THREADS, 0, g->stream>>>(y, ld, g->node_type_int.p, g->node_id_int.p, ts.excl.p, g->n, ts.k,
                                                            block_max.p, ts.block_out.p);
    k_topk_merge<T><<<1, TOPK_THREADS, 0, g->stream>>>(ts.block_out.p, ts.grid * ts.k, ts.k, y, ld, ts.ids.p + (size_t)list * ts.k,
                                                       ts.scores.p + (size_t)list * ts.k, ts.counts.p + list);
    KERNEL_CHECK();
    g->pool.launches += 3;
}

static void ensure_items_by_id(rwr_graph* g) {
    if (g->items_by_id_desc.p) return;
    cudaStream_t st = g->stream;
    const int n = g->n;
    DevBuf<u32> pos;
    pos.alloc(n);
    if (n) k_item_flags<<<div_up(n, 256), 256, 0, st>>>(g->node_type_int.p, n, pos.p);
    KERNEL_CHECK();
    const u32 m = prim::scan_total<u32>(pos.p, pos.p, n, false, st, &g->pool);
    prim::SortBuffers<u64> sb;
    sb.alloc(m, true);
    if (n) k_item_keys<<<div_up(n, 256), 256, 0, st>>>(g->node_type_int.p, g->node_id_int.p, pos.p, n, sb.keys(), sb.vals());
    KERNEL_CHECK();
    sb.sort(m, 64, st, &g->pool);
    g->items_by_id_desc.alloc(m, &g->pool);
    if (m) CUDA_CHECK(cudaMemcpyAsync(g->items_by_id_desc.p, sb.vals(), (size_t)m * 4, cudaMemcpyDeviceToDevice, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    g->n_items = (int)m;
}

// Full ranking of one seed on the device; returns the candidate count, fills up to `cap` pairs on the host.
// (rset: a restart-set result, whose exclusion is the union over its nodes; seed is then unused)
template <typename T>
static int64_t rank_all_one(rwr_graph* g, const T* y, int seed, int64_t* ids, double* scores, int64_t cap,
                            const rwr_result* rset = nullptr) {
    cudaStream_t st = g->stream;
    ensure_items_by_id(g);
    const size_t words = ((size_t)g->n + 31) / 32 + 1;
    DevBuf<u32> excl;
    excl.alloc(words);
    if (rset) mark_excluded_for(g, rset, 0, excl.p, words);
    else mark_excluded(g, seed, excl.p, words);
    const int m = g->n_items;
    DevBuf<u32> pos;
    pos.alloc(m);
    if (m) k_cand_flags<<<div_up(m, 256), 256, 0, st>>>(g->items_by_id_desc.p, m, excl.p, pos.p);
    KERNEL_CHECK();
    const u32 cnt = prim::scan_total<u32>(pos.p, pos.p, m, false, st, &g->pool);
    if (cnt == 0) return 0;
    prim::SortBuffers<u64> sb;
    sb.alloc(cnt, true);
    k_cand_keys<T><<<div_up(m, 256), 256, 0, st>>>(g->items_by_id_desc.p, m, excl.p, pos.p, y, sb.keys(), sb.vals());
    KERNEL_CHECK();
    sb.sort(cnt, 64, st, &g->pool);
    const size_t emit = (size_t)std::min<int64_t>(cap, (int64_t)cnt);
    if (emit && ids && scores) {
        DevBuf<int64_t> d_ids;
        DevBuf<double> d_sc;
        d_ids.alloc(emit); d_sc.alloc(emit);
        k_emit_ranking<T><<<div_up(emit, 256), 256, 0, st>>>(sb.vals(), emit, y, g->node_id_int.p, d_ids.p, d_sc.p);
        KERNEL_CHECK();
        CUDA_CHECK(cudaMemcpyAsync(ids, d_ids.p, emit * 8, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaMemcpyAsync(scores, d_sc.p, emit * 8, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
    }
    g->pool.launches += 3;
    return (int64_t)cnt;
}

extern "C" {

int rwr_topk(rwr_result* r, int32_t k, int64_t* out_ids, double* out_scores, int32_t* out_counts) {
    RWR_API_BEGIN
    if (!r || !out_ids || !out_scores || !out_counts) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (k <= 0) RWR_FAIL(RWR_E_INVALID, "k must be positive (Recommendation(.., topN <= 0) returns the full list: use rwr_rank_all)");
    rwr_graph* g = r->g;
    CUDA_CHECK(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    const int S = r->n_seeds;
    const rwr_result* rset = r->restart_nodes.empty() ? nullptr : r;
    if (k > TOPK_MAX) {                                  // large k: truncate the full ranking
        for (int s = 0; s < S; s++) {
            int64_t cnt = (r->precision == RWR_FP64)
                ? rank_all_one<double>(g, r->y64.p + (size_t)s * r->ld, r->seeds[s], out_ids + (size_t)s * k, out_scores + (size_t)s * k, k, rset)
                : rank_all_one<float>(g, r->y32.p + (size_t)s * r->ld, r->seeds[s], out_ids + (size_t)s * k, out_scores + (size_t)s * k, k, rset);
            out_counts[s] = (int32_t)std::min<int64_t>(cnt, k);
        }
        return RWR_OK;
    }
    TopkScratch ts(g, k, S);
    for (int s = 0; s < S; s++) {
        if (rset) mark_excluded_for(g, r, s, ts.excl.p, ts.words);
        if (r->precision == RWR_FP64) topk_one<double>(g, ts, s, r->y64.p + (size_t)s * r->ld, 1, r->seeds[s], rset != nullptr);
        else topk_one<float>(g, ts, s, r->y32.p + (size_t)s * r->ld, 1, r->seeds[s], rset != nullptr);
    }
    ts.copy_out(st, out_ids, out_scores, out_counts);
    CUDA_CHECK(cudaStreamSynchronize(st));
    return RWR_OK;
    RWR_API_END
}

int rwr_rank_all(rwr_result* r, int32_t seed_slot, int64_t* ids, double* scores, int64_t cap, int64_t* count) {
    RWR_API_BEGIN
    if (!r || !count) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (seed_slot < 0 || seed_slot >= r->n_seeds) RWR_FAIL(RWR_E_INVALID, "seed slot %d outside [0, %d)", seed_slot, r->n_seeds);
    rwr_graph* g = r->g;
    CUDA_CHECK(cudaSetDevice(g->device));
    if (cap < 0) cap = 0;
    const rwr_result* rset = r->restart_nodes.empty() ? nullptr : r;
    *count = (r->precision == RWR_FP64)
        ? rank_all_one<double>(g, r->y64.p + (size_t)seed_slot * r->ld, r->seeds[seed_slot], ids, scores, cap, rset)
        : rank_all_one<float>(g, r->y32.p + (size_t)seed_slot * r->ld, r->seeds[seed_slot], ids, scores, cap, rset);
    return RWR_OK;
    RWR_API_END
}

}  // extern "C"

// n_seeds x Recommendation(seed, c, nIter, k).  Seeds are processed in SpMM tiles of B columns (8 FP64 / 16 FP32):
// one pass over the matrix serves B seeds; the ranks of a tile are dropped once its top-k lists are out.
template <typename T>
void spmm_run_tile(rwr_graph* g, const int* seeds_int, int n_active, double c, int n_iter, T* y_out, int64_t* launches);
int spmm_tile_width(int precision);
void ensure_fp32_arrays(rwr_graph* g);

template <typename T>
void iterate_single_into(rwr_graph* g, int seed_orig, double c, int n_iter, T* y_out, float* iter_ms, int64_t* launches,
                         cudaEvent_t ext0, cudaEvent_t ext1);

// What a fixed-count run of n_seeds seeds reports (no residual: no convergence test ran)
template <typename T>
static void fill_info(rwr_run_info* info, const rwr_graph* g, int n_seeds, int n_iter, float iterate_ms, float total_ms,
                      int64_t launches) {
    if (!info) return;
    info->n_seeds = n_seeds; info->n_nodes = g->n; info->precision = sizeof(T) == 4 ? RWR_FP32 : RWR_FP64;
    info->iterations = n_iter; info->residual = NAN; info->iterate_ms = iterate_ms; info->total_ms = total_ms;
    info->kernel_launches = launches;
}

// The internal labels of a seed list (for the SpMM tiles), and its original labels copied to d_orig (the tile kernels
// read the seeds' raw link ranges)
static std::vector<int32_t> seed_labels(rwr_graph* g, const int32_t* seeds, int n_seeds, Scratch<int32_t>& d_orig) {
    cudaStream_t st = g->stream;
    std::vector<int32_t> internal((size_t)n_seeds);
    d_orig.alloc(&g->scratch, n_seeds);
    Scratch<int32_t> d_int;
    d_int.alloc(&g->scratch, n_seeds);
    CUDA_CHECK(cudaMemcpyAsync(d_orig.p, seeds, (size_t)n_seeds * 4, cudaMemcpyHostToDevice, st));
    k_lookup<<<div_up((size_t)n_seeds, 256), 256, 0, st>>>(g->new_of_old.p, d_orig.p, n_seeds, d_int.p);
    KERNEL_CHECK();
    CUDA_CHECK(cudaMemcpyAsync(internal.data(), d_int.p, (size_t)n_seeds * 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    return internal;
}

// seeds one by one through the single-column kernel (k <= 16): no result objects, scratch from the handle's pool
template <typename T>
static void recommend_singles(rwr_graph* g, const int32_t* seeds, int n_seeds, double c, int n_iter, int k, int64_t* out_ids,
                              double* out_scores, int32_t* out_counts, rwr_run_info* info) {
    cudaStream_t st = g->stream;
    const size_t n = (size_t)g->n;
    Scratch<T> y;
    y.alloc(&g->scratch, n + 8);
    TopkScratch ts(g, k, n_seeds);
    float it_ms = 0.f;
    int64_t launches = 0;
    struct Events {                                 // destroyed on every exit path (a seed without links throws)
        cudaEvent_t e[4] = {nullptr, nullptr, nullptr, nullptr};
        ~Events() { for (auto& x : e) if (x) cudaEventDestroy(x); }
    } evs;
    cudaEvent_t &e0 = evs.e[0], &e1 = evs.e[1], &i0 = evs.e[2], &i1 = evs.e[3];
    CUDA_CHECK(cudaEventCreate(&e0)); CUDA_CHECK(cudaEventCreate(&e1));
    // one request (the usual case): the exclusion list first (its host round trip happens before any kernel is queued),
    // then iterations and top-k enqueued back to back with a single synchronisation at the end
    const bool one = n_seeds == 1;
    if (one) { CUDA_CHECK(cudaEventCreate(&i0)); CUDA_CHECK(cudaEventCreate(&i1)); }
    CUDA_CHECK(cudaEventRecord(e0, st));
    for (int s = 0; s < n_seeds; s++) {
        if (one) mark_excluded(g, seeds[s], ts.excl.p, ts.words);
        iterate_single_into<T>(g, seeds[s], c, n_iter, y.p, &it_ms, &launches, i0, i1);
        topk_one<T>(g, ts, s, y.p, 1, seeds[s], /*marked=*/one);
        launches += 3;
    }
    ts.copy_out(st, out_ids, out_scores, out_counts);
    CUDA_CHECK(cudaEventRecord(e1, st));
    CUDA_CHECK(cudaEventSynchronize(e1));
    float tot = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&tot, e0, e1));
    if (one) CUDA_CHECK(cudaEventElapsedTime(&it_ms, i0, i1));
    fill_info<T>(info, g, n_seeds, n_iter, it_ms, tot, launches);
}

template <typename T>
static void recommend_tiles(rwr_graph* g, const int32_t* seeds, int n_seeds, double c, int n_iter, int k, int64_t* out_ids,
                            double* out_scores, int32_t* out_counts, rwr_run_info* info) {
    cudaStream_t st = g->stream;
    const int B = spmm_tile_width(sizeof(T) == 4 ? RWR_FP32 : RWR_FP64);
    const size_t n = (size_t)g->n;
    if (sizeof(T) == 4) ensure_fp32_arrays(g);
    Scratch<int32_t> d_seeds_all;
    const std::vector<int32_t> n2o = seed_labels(g, seeds, n_seeds, d_seeds_all);
    Scratch<T> y;
    y.alloc(&g->scratch, n * B + 16);
    TopkScratch ts(g, k, n_seeds);
    const size_t words = ts.words;
    const int grid = ts.grid;
    Scratch<u32> excl_t;                           // [B][words] exclusion bitmaps of a tile
    Scratch<u64> tile_max, tile_bound;             // [grid][B] block maxima, [B] bounds
    Scratch<Cand> tile_cand;                       // [B][TILE_CAND_CAP]
    Scratch<int> tile_cnt;                         // [TILE_MAXB] candidate counts | [TILE_MAXB] seeds without links
    excl_t.alloc(&g->scratch, (size_t)B * words); tile_max.alloc(&g->scratch, (size_t)grid * B); tile_bound.alloc(&g->scratch, TILE_MAXB);
    tile_cand.alloc(&g->scratch, (size_t)B * TILE_CAND_CAP); tile_cnt.alloc(&g->scratch, 2 * TILE_MAXB);
    DevEvent e0, e1, e2;
    int64_t launches = 0;
    float it_ms = 0.f, tot_ms = 0.f;
    for (int s0 = 0; s0 < n_seeds; s0 += B) {
        const int cnt = std::min(B, n_seeds - s0);
        CUDA_CHECK(cudaEventRecord(e0, st));
        spmm_run_tile<T>(g, n2o.data() + s0, cnt, c, n_iter, y.p, &launches);
        CUDA_CHECK(cudaEventRecord(e1, st));
        // top-k of the whole tile in one pass over Y per step (bound, scan), then one merge block per column
        CUDA_CHECK(cudaMemsetAsync(excl_t.p, 0, (size_t)B * words * sizeof(u32), st));
        CUDA_CHECK(cudaMemsetAsync(tile_cnt.p, 0, 2 * TILE_MAXB * sizeof(int), st));
        k_mark_excluded_tile<<<dim3(8, cnt), 256, 0, st>>>(g->raw_dst.p, g->raw_type.p, g->raw_ptr.p, d_seeds_all.p + s0,
                                                          g->new_of_old.p, g->n, words, excl_t.p, tile_cnt.p + TILE_MAXB);
        if (B == 8) {
            k_topk_bound_tile<T, 8><<<grid, TOPK_THREADS, 0, st>>>(y.p, g->node_type_int.p, excl_t.p, words, g->n, cnt, tile_max.p);
            k_topk_bounds_tile<8><<<cnt, TOPK_THREADS, 0, st>>>(tile_max.p, grid, k, tile_bound.p);
            k_topk_scan_tile<T, 8><<<grid, TOPK_THREADS, 0, st>>>(y.p, g->node_type_int.p, g->node_id_int.p, excl_t.p, words, g->n, cnt,
                                                                 tile_bound.p, tile_cand.p, tile_cnt.p);
        } else {
            k_topk_bound_tile<T, 16><<<grid, TOPK_THREADS, 0, st>>>(y.p, g->node_type_int.p, excl_t.p, words, g->n, cnt, tile_max.p);
            k_topk_bounds_tile<16><<<cnt, TOPK_THREADS, 0, st>>>(tile_max.p, grid, k, tile_bound.p);
            k_topk_scan_tile<T, 16><<<grid, TOPK_THREADS, 0, st>>>(y.p, g->node_type_int.p, g->node_id_int.p, excl_t.p, words, g->n, cnt,
                                                                  tile_bound.p, tile_cand.p, tile_cnt.p);
        }
        k_topk_merge_tile<T><<<cnt, TOPK_THREADS, 0, st>>>(tile_cand.p, tile_cnt.p, k, y.p, B, ts.ids.p + (size_t)s0 * k,
                                                          ts.scores.p + (size_t)s0 * k, ts.counts.p + s0);
        KERNEL_CHECK();
        launches += 5;
        int h_cnt[2 * TILE_MAXB];
        CUDA_CHECK(cudaMemcpyAsync(h_cnt, tile_cnt.p, sizeof(h_cnt), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaEventRecord(e2, st));
        CUDA_CHECK(cudaEventSynchronize(e2));
        for (int j = 0; j < cnt; j++) {
            if (h_cnt[TILE_MAXB + j] && !g->opts.empty_seed_ok)
                RWR_FAIL(RWR_E_BADSEED, "seed %d has no `edges` entry (KeyNotFoundException, Recommender.cs:21)", seeds[s0 + j]);
            if (h_cnt[j] > TILE_CAND_CAP) {              // too many candidates at the bound (ties): exact per-column path
                topk_one<T>(g, ts, s0 + j, y.p + j, B, seeds[s0 + j]);
                launches += 4;
            }
        }
        float a = 0.f, b = 0.f;
        CUDA_CHECK(cudaEventElapsedTime(&a, e0, e1));
        CUDA_CHECK(cudaEventElapsedTime(&b, e0, e2));
        it_ms += a; tot_ms += b;
    }
    ts.copy_out(st, out_ids, out_scores, out_counts);
    CUDA_CHECK(cudaStreamSynchronize(st));
    fill_info<T>(info, g, n_seeds, n_iter, it_ms, tot_ms, launches);
}

extern "C" {

int rwr_recommend(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, int32_t n_iter, int32_t precision,
                  int32_t k, int64_t* out_ids, double* out_scores, int32_t* out_counts, rwr_run_info* info) {
    RWR_API_BEGIN
    if (!g || !out_ids || !out_scores || !out_counts || (n_seeds && !seeds)) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (k <= 0) RWR_FAIL(RWR_E_INVALID, "k must be positive");
    if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
    if (precision != RWR_FP64 && precision != RWR_FP32) RWR_FAIL(RWR_E_INVALID, "unknown precision %d", precision);
    if (info) memset(info, 0, sizeof(*info));
    if (n_seeds == 0) return RWR_OK;
    if (n_iter < 0) n_iter = 0;
    CUDA_CHECK(cudaSetDevice(g->device));
    AllocStream alloc_on(g->stream);
    for (int s = 0; s < n_seeds; s++) {
        // Recommendation(idxTargetUser, ..) always has a target user; the uniform constructor (seed -1) is a Model-only path
        if (seeds[s] == -1) RWR_FAIL(RWR_E_INVALID, "seed -1 (uniform restart) is not a target user: use rwr_run_fixed + rwr_scores");
        if (seeds[s] < 0 || seeds[s] >= g->n) RWR_FAIL(RWR_E_BADSEED, "seed %d outside [0, %d)", seeds[s], g->n);
    }
    // a row slice of a partitioned graph has no whole-graph pull CSR: seeds run one at a time through the edge stream
    if (k <= TOPK_MAX && (n_seeds < 2 || g->opts.batch_width == 1 || g->comm)) {
        if (precision == RWR_FP64) recommend_singles<double>(g, seeds, n_seeds, c, n_iter, k, out_ids, out_scores, out_counts, info);
        else recommend_singles<float>(g, seeds, n_seeds, c, n_iter, k, out_ids, out_scores, out_counts, info);
        return RWR_OK;
    }
    if (k > TOPK_MAX) {
        // result-object path per seed (k > 16 needs the full ranking)
        for (int s = 0; s < n_seeds; s++) {
            rwr_result* res = nullptr;
            int rc = rwr_run_fixed(g, seeds + s, 1, c, n_iter, precision, &res);
            if (rc != RWR_OK) return rc;
            rc = rwr_topk(res, k, out_ids + (size_t)s * k, out_scores + (size_t)s * k, out_counts + s);
            if (info) {
                info->n_seeds = n_seeds; info->n_nodes = g->n; info->precision = precision; info->iterations = n_iter;
                info->residual = NAN; info->iterate_ms += res->iterate_ms; info->total_ms += res->total_ms;
                info->kernel_launches += res->launches + 3;
            }
            rwr_result_destroy(res);
            if (rc != RWR_OK) return rc;
        }
        return RWR_OK;
    }
    if (precision == RWR_FP64) recommend_tiles<double>(g, seeds, n_seeds, c, n_iter, k, out_ids, out_scores, out_counts, info);
    else recommend_tiles<float>(g, seeds, n_seeds, c, n_iter, k, out_ids, out_scores, out_counts, info);
    return RWR_OK;
    RWR_API_END
}

}  // extern "C"

// The ranks of the batched request path, tile by tile as recommend_tiles / evaluate_tiles compose them, unpermuted and
// widened on the host (not timed: no kernel of its own)
template <typename T>
static void probe_tiles(rwr_graph* g, const int32_t* seeds, int n_seeds, double c, int n_iter, double* out) {
    cudaStream_t st = g->stream;
    const int B = spmm_tile_width(sizeof(T) == 4 ? RWR_FP32 : RWR_FP64);
    const size_t n = (size_t)g->n;
    if (sizeof(T) == 4) ensure_fp32_arrays(g);
    Scratch<int32_t> d_seeds_all;
    const std::vector<int32_t> n2o = seed_labels(g, seeds, n_seeds, d_seeds_all);
    Scratch<T> y;
    y.alloc(&g->scratch, n * B + 16);
    std::vector<T> h_y(n * B);
    std::vector<int32_t> new_of_old(n);
    CUDA_CHECK(cudaMemcpyAsync(new_of_old.data(), g->new_of_old.p, n * 4, cudaMemcpyDeviceToHost, st));
    int64_t launches = 0;
    for (int s0 = 0; s0 < n_seeds; s0 += B) {
        const int cnt = std::min(B, n_seeds - s0);
        spmm_run_tile<T>(g, n2o.data() + s0, cnt, c, n_iter, y.p, &launches);
        CUDA_CHECK(cudaMemcpyAsync(h_y.data(), y.p, n * B * sizeof(T), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        for (int j = 0; j < cnt; j++)
            for (size_t i = 0; i < n; i++) out[(size_t)(s0 + j) * n + i] = (double)h_y[(size_t)new_of_old[i] * B + j];
    }
}

extern "C" {

int rwr_probe_tile_ranks(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, int32_t n_iter, int32_t precision,
                         double* out) {
    RWR_API_BEGIN
    if (!g || (n_seeds && (!seeds || !out)) || n_seeds < 0) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
    if (precision != RWR_FP64 && precision != RWR_FP32) RWR_FAIL(RWR_E_INVALID, "unknown precision %d", precision);
    for (int s = 0; s < n_seeds; s++) {
        if (seeds[s] == -1) RWR_FAIL(RWR_E_INVALID, "seed -1 (uniform restart) is not a target user: use rwr_run_fixed + rwr_scores");
        if (seeds[s] < 0 || seeds[s] >= g->n) RWR_FAIL(RWR_E_BADSEED, "seed %d outside [0, %d)", seeds[s], g->n);
    }
    if (g->comm) RWR_FAIL(RWR_E_UNSUPPORTED, "the seed tiles need the whole pull CSR: a row-partitioned handle has a slice of it");
    if (n_seeds == 0) return RWR_OK;
    if (n_iter < 0) n_iter = 0;
    CUDA_CHECK(cudaSetDevice(g->device));
    AllocStream alloc_on(g->stream);
    if (precision == RWR_FP64) probe_tiles<double>(g, seeds, n_seeds, c, n_iter, out);
    else probe_tiles<float>(g, seeds, n_seeds, c, n_iter, out);
    return RWR_OK;
    RWR_API_END
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------ N1: evaluation on the device
// Experiment.cs:121-128 walks the full ranking and, for every test item it meets, adds nHits / (i + 1).  The ranking is a
// total order (score desc, id desc: Recommender.cs:34-38), so the position of a test item is 1 + the number of candidates
// that rank before it -- a count, no sort.  One pass over the rank tile Y[n, B] serves all B users of the tile.
struct EvalItem {
    u64 key;        // score key of the test item (0 with idx < 0: not a candidate)
    int64_t id;
    int idx;        // internal label, -1: the id is not a candidate of this user
    u32 before;     // candidates ranking before it
};

// unsigned-order image of a node id
__device__ __forceinline__ u64 id_key(int64_t id) { return (u64)id ^ 0x8000000000000000ULL; }

__global__ void k_ev_id_keys(const int64_t* __restrict__ id_int, int n, u64* __restrict__ keys, u32* __restrict__ vals) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) { keys[j] = id_key(id_int[j]); vals[j] = (u32)j; }
}

// items of the tile: column `col` owns items [iptr[col], iptr[col + 1]); resolve id -> label, candidate test, score key
template <typename T>
__global__ void k_ev_resolve(const int64_t* __restrict__ test_ids, const int* __restrict__ iptr, int cols, int B,
                             const u64* __restrict__ ids_sorted, const u32* __restrict__ label_of_sorted, int n,
                             const u8* __restrict__ type_int, const u32* __restrict__ excl, size_t words,
                             const T* __restrict__ y, EvalItem* __restrict__ items) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= iptr[cols]) return;
    int col = 0;
    while (col + 1 < cols && iptr[col + 1] <= i) col++;
    const int64_t id = test_ids[i];
    const u64 k = id_key(id);
    int lo = 0, hi = n;
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ids_sorted[mid] < k) lo = mid + 1; else hi = mid; }
    EvalItem it;
    it.key = 0; it.id = id; it.idx = -1; it.before = 0;
    if (lo < n && ids_sorted[lo] == k) {
        const int j = (int)label_of_sorted[lo];
        const u32* ex = excl + (size_t)col * words;
        if (type_int[j] == RWR_NODE_ITEM && !((ex[j >> 5] >> (j & 31)) & 1u)) {
            it.idx = j;
            it.key = score_key((double)y[(size_t)j * B + col]);
        }
    }
    items[i] = it;
}

// The candidates that rank before a test item are counted with one pass over the rank tile, whatever the number of test
// items: per column the valid items are sorted ascending by (score key, id); a candidate row finds by binary search how
// many items it beats (ip = items strictly below it) and adds one to bucket ip of the column's histogram; the number of
// candidates before sorted item j is then the sum of the buckets above j.
constexpr int EV_SMEM_ITEMS = 2048;              // tile items whose sorted keys and buckets fit the block's shared memory

__device__ __forceinline__ bool ev_less(u64 ka, int64_t ia, u64 kb, int64_t ib) { return ka < kb || (ka == kb && ia < ib); }

// one block per column: rank-sort the valid items; sorted[] gets (key, id), sptr[col + 1] the valid count (prefix-summed by
// the caller's layout: sorted items of column `col` live at [iptr[col], iptr[col] + nvalid[col]))
__global__ void __launch_bounds__(TOPK_THREADS) k_ev_sort(const EvalItem* __restrict__ items, const int* __restrict__ iptr,
                                                          u64* __restrict__ skey, int64_t* __restrict__ sid, int* __restrict__ nvalid) {
    const int col = blockIdx.x, b = iptr[col], e = iptr[col + 1];
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    for (int i = b + threadIdx.x; i < e; i += TOPK_THREADS) {
        if (items[i].idx < 0) continue;
        const u64 k = items[i].key;
        const int64_t id = items[i].id;
        int r = 0;
        for (int j = b; j < e; j++)
            if (items[j].idx >= 0 && (ev_less(items[j].key, items[j].id, k, id) || (items[j].key == k && items[j].id == id && j < i))) r++;
        skey[b + r] = k;
        sid[b + r] = id;
        atomicAdd(&cnt, 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) nvalid[col] = cnt;
}

// thread (row lane, column): bucket of every candidate row.  hist[iptr[col] + col + ip], ip in [0, nvalid[col]]
template <typename T, int B, bool SMEM>
__global__ void __launch_bounds__(TOPK_THREADS) k_ev_hist(const T* __restrict__ y, const u8* __restrict__ type_int,
                                                          const int64_t* __restrict__ id_int, const u32* __restrict__ excl,
                                                          size_t words, int n, int cols, const int* __restrict__ iptr,
                                                          const int* __restrict__ nvalid, const u64* __restrict__ skey,
                                                          const int64_t* __restrict__ sid, u32* __restrict__ hist) {
    __shared__ u64 s_key[SMEM ? EV_SMEM_ITEMS : 1];
    __shared__ int64_t s_id[SMEM ? EV_SMEM_ITEMS : 1];
    __shared__ u32 s_hist[SMEM ? EV_SMEM_ITEMS + TILE_MAXB : 1];
    const int total = iptr[cols];
    if (SMEM) {
        for (int i = threadIdx.x; i < total; i += TOPK_THREADS) { s_key[i] = skey[i]; s_id[i] = sid[i]; }
        for (int i = threadIdx.x; i < total + cols; i += TOPK_THREADS) s_hist[i] = 0;
        __syncthreads();
    }
    const int col = threadIdx.x % B, rlane = threadIdx.x / B;
    constexpr int RPB = TOPK_THREADS / B;
    if (col < cols && nvalid[col] > 0) {
        const int base = iptr[col], m = nvalid[col];
        const u64* kk = SMEM ? s_key + base : skey + base;
        const int64_t* ii = SMEM ? s_id + base : sid + base;
        u32* hh = (SMEM ? s_hist : hist) + base + col;
        const u32* ex = excl + (size_t)col * words;
        const u64 kmin = kk[0];
        for (int j = blockIdx.x * RPB + rlane; j < n; j += gridDim.x * RPB) {
            if (type_int[j] != RWR_NODE_ITEM) continue;
            const u64 key = score_key((double)y[(size_t)j * B + col]);
            if (key < kmin) continue;                                   // beats nothing: bucket 0 is never read
            if ((ex[j >> 5] >> (j & 31)) & 1u) continue;
            const int64_t id = id_int[j];
            int lo = 0, hi = m;                                         // ip = first sorted item that is not below the row
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (ev_less(kk[mid], ii[mid], key, id)) lo = mid + 1; else hi = mid;
            }
            if (lo > 0) atomicAdd(hh + lo, 1u);
        }
    }
    if (SMEM) {
        __syncthreads();
        for (int i = threadIdx.x; i < total + cols; i += TOPK_THREADS)
            if (s_hist[i]) atomicAdd(hist + i, s_hist[i]);
    }
}

// one thread per column: the reference's loop (Experiment.cs:121-128) over the test items in ranking order -- sorted item
// m-1 comes first -- with position = number of candidates above it
__global__ void k_ev_finish(const int* __restrict__ iptr, const int* __restrict__ nvalid, const u32* __restrict__ hist, int cols,
                            int k, int* __restrict__ hits, double* __restrict__ ap, int* __restrict__ hits_at_k) {
    const int col = blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= cols) return;
    const int m = nvalid[col];
    const u32* hh = hist + iptr[col] + col;
    int nHits = 0, atk = 0;
    double sumPrecision = 0.0;
    u32 above = 0;                                        // candidates that beat sorted item j: buckets j+1 .. m
    for (int j = m - 1; j >= 0; j--) {
        above += hh[j + 1];
        // the (m - 1 - j) test items above j are candidates themselves and are counted in `above` already
        const u32 i0 = above;                             // zero-based index in the recommendation list
        nHits += 1;
        sumPrecision += (double)nHits / (double)(i0 + 1);  // Experiment.cs:126
        if ((int)i0 < k) atk++;
    }
    hits[col] = nHits;
    ap[col] = nHits == 0 ? 0.0 : sumPrecision / nHits;     // Experiment.cs:136
    hits_at_k[col] = atk;
}

static void ensure_id_lookup(rwr_graph* g) {
    if (g->ids_sorted.p) return;
    cudaStream_t st = g->stream;
    const int n = g->n;
    prim::SortBuffers<u64> sb;
    sb.alloc(n, true);
    if (n) k_ev_id_keys<<<div_up(n, 256), 256, 0, st>>>(g->node_id_int.p, n, sb.keys(), sb.vals());
    KERNEL_CHECK();
    sb.sort(n, 64, st, &g->pool);
    g->ids_sorted.alloc(n, &g->pool);
    g->label_of_sorted.alloc(n, &g->pool);
    if (n) {
        CUDA_CHECK(cudaMemcpyAsync(g->ids_sorted.p, sb.keys(), (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(g->label_of_sorted.p, sb.vals(), (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
}

template <typename T>
static void evaluate_tiles(rwr_graph* g, const int32_t* users, int n_users, const int64_t* test_ptr, const int64_t* test_ids,
                           double c, int n_iter, int k, int32_t* hits, double* avg_precision, int32_t* hits_at_k,
                           rwr_run_info* info) {
    cudaStream_t st = g->stream;
    const int B = spmm_tile_width(sizeof(T) == 4 ? RWR_FP32 : RWR_FP64);
    const size_t n = (size_t)g->n;
    if (sizeof(T) == 4) ensure_fp32_arrays(g);
    ensure_id_lookup(g);
    Scratch<int32_t> d_users;
    const std::vector<int32_t> n2o = seed_labels(g, users, n_users, d_users);
    const int64_t total_items = test_ptr[n_users];
    Scratch<int64_t> d_test;
    d_test.alloc(&g->scratch, (size_t)std::max<int64_t>(total_items, 1));
    if (total_items) CUDA_CHECK(cudaMemcpyAsync(d_test.p, test_ids, (size_t)total_items * 8, cudaMemcpyHostToDevice, st));
    int64_t max_tile_items = 1;
    for (int s0 = 0; s0 < n_users; s0 += B)
        max_tile_items = std::max(max_tile_items, test_ptr[std::min(n_users, s0 + B)] - test_ptr[s0]);
    Scratch<T> y;
    y.alloc(&g->scratch, n * B + 16);
    const size_t words = (n + 31) / 32 + 1;
    const int grid = topk_grid(g);
    Scratch<u32> excl_t, hist;
    Scratch<EvalItem> items;
    Scratch<u64> skey;
    Scratch<int64_t> sid;
    Scratch<int> d_iptr, no_links, d_hits, d_atk, d_nvalid;
    Scratch<double> d_ap;
    excl_t.alloc(&g->scratch, (size_t)B * words);
    items.alloc(&g->scratch, (size_t)max_tile_items); hist.alloc(&g->scratch, (size_t)max_tile_items + TILE_MAXB);
    skey.alloc(&g->scratch, (size_t)max_tile_items); sid.alloc(&g->scratch, (size_t)max_tile_items);
    d_iptr.alloc(&g->scratch, TILE_MAXB + 1); no_links.alloc(&g->scratch, TILE_MAXB); d_nvalid.alloc(&g->scratch, TILE_MAXB);
    d_hits.alloc(&g->scratch, n_users); d_atk.alloc(&g->scratch, n_users); d_ap.alloc(&g->scratch, n_users);
    DevEvent e0, e1, e2;
    int64_t launches = 0;
    float it_ms = 0.f, tot_ms = 0.f;
    for (int s0 = 0; s0 < n_users; s0 += B) {
        const int cnt = std::min(B, n_users - s0);
        CUDA_CHECK(cudaEventRecord(e0, st));
        spmm_run_tile<T>(g, n2o.data() + s0, cnt, c, n_iter, y.p, &launches);
        CUDA_CHECK(cudaEventRecord(e1, st));
        int h_iptr[TILE_MAXB + 1];
        for (int j = 0; j <= TILE_MAXB; j++) h_iptr[j] = (int)(test_ptr[s0 + std::min(j, cnt)] - test_ptr[s0]);
        const int tile_items = h_iptr[cnt];
        CUDA_CHECK(cudaMemcpyAsync(d_iptr.p, h_iptr, sizeof(h_iptr), cudaMemcpyHostToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(excl_t.p, 0, (size_t)B * words * sizeof(u32), st));
        CUDA_CHECK(cudaMemsetAsync(no_links.p, 0, TILE_MAXB * sizeof(int), st));
        k_mark_excluded_tile<<<dim3(8, cnt), 256, 0, st>>>(g->raw_dst.p, g->raw_type.p, g->raw_ptr.p, d_users.p + s0, g->new_of_old.p,
                                                          g->n, words, excl_t.p, no_links.p);
        CUDA_CHECK(cudaMemsetAsync(d_nvalid.p, 0, TILE_MAXB * sizeof(int), st));
        if (tile_items) {
            k_ev_resolve<T><<<div_up((size_t)tile_items, 256), 256, 0, st>>>(d_test.p + test_ptr[s0], d_iptr.p, cnt, B, g->ids_sorted.p,
                                                                            g->label_of_sorted.p, g->n, g->node_type_int.p, excl_t.p,
                                                                            words, y.p, items.p);
            k_ev_sort<<<cnt, TOPK_THREADS, 0, st>>>(items.p, d_iptr.p, skey.p, sid.p, d_nvalid.p);
            CUDA_CHECK(cudaMemsetAsync(hist.p, 0, ((size_t)tile_items + TILE_MAXB) * sizeof(u32), st));
            const bool sm = tile_items <= EV_SMEM_ITEMS;
#define EV_HIST(BB, SM) k_ev_hist<T, BB, SM><<<grid, TOPK_THREADS, 0, st>>>(y.p, g->node_type_int.p, g->node_id_int.p, excl_t.p, words, \
                                                                            g->n, cnt, d_iptr.p, d_nvalid.p, skey.p, sid.p, hist.p)
            if (B == 8) { if (sm) EV_HIST(8, true); else EV_HIST(8, false); }
            else { if (sm) EV_HIST(16, true); else EV_HIST(16, false); }
#undef EV_HIST
            launches += 3;
        }
        k_ev_finish<<<1, 32, 0, st>>>(d_iptr.p, d_nvalid.p, hist.p, cnt, k, d_hits.p + s0, d_ap.p + s0, d_atk.p + s0);
        KERNEL_CHECK();
        launches += 2;
        int h_no[TILE_MAXB];
        CUDA_CHECK(cudaMemcpyAsync(h_no, no_links.p, sizeof(h_no), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaEventRecord(e2, st));
        CUDA_CHECK(cudaEventSynchronize(e2));
        for (int j = 0; j < cnt; j++)
            if (h_no[j] && !g->opts.empty_seed_ok) RWR_FAIL(RWR_E_BADSEED, "user %d has no `edges` entry (KeyNotFoundException, Recommender.cs:21)", users[s0 + j]);
        float a = 0.f, b = 0.f;
        CUDA_CHECK(cudaEventElapsedTime(&a, e0, e1));
        CUDA_CHECK(cudaEventElapsedTime(&b, e0, e2));
        it_ms += a; tot_ms += b;
    }
    CUDA_CHECK(cudaMemcpyAsync(hits, d_hits.p, (size_t)n_users * 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaMemcpyAsync(hits_at_k, d_atk.p, (size_t)n_users * 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaMemcpyAsync(avg_precision, d_ap.p, (size_t)n_users * 8, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    fill_info<T>(info, g, n_users, n_iter, it_ms, tot_ms, launches);
}

extern "C" {

int rwr_evaluate_users(rwr_graph* g, const int32_t* users, int32_t n_users, const int64_t* test_ptr, const int64_t* test_ids,
                       double c, int32_t n_iter, int32_t precision, int32_t k, int32_t* hits, double* avg_precision,
                       int32_t* hits_at_k, int32_t* n_test_of_user, rwr_run_info* info) {
    RWR_API_BEGIN
    if (!g || !hits || !avg_precision || !hits_at_k) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
    if (g->comm) RWR_FAIL(RWR_E_UNSUPPORTED, "evaluation runs on seed tiles: use a replicated graph and shard the users over the ranks");
    if (precision != RWR_FP64 && precision != RWR_FP32) RWR_FAIL(RWR_E_INVALID, "unknown precision %d", precision);
    if (info) memset(info, 0, sizeof(*info));
    if (!users) {                                   // the users and test sets rwr_graph_hold_out stored
        if (test_ptr || test_ids) RWR_FAIL(RWR_E_INVALID, "test sets without a user list");
        if (n_users != (int32_t)g->held_users.size()) RWR_FAIL(RWR_E_INVALID, "n_users %d != %zu held-out users", n_users, g->held_users.size());
        users = g->held_users.data();
    }
    if (!test_ptr) {
        if (n_users != (int32_t)g->held_users.size() || !std::equal(users, users + n_users, g->held_users.begin()))
            RWR_FAIL(RWR_E_INVALID, "no test sets given and the user list is not the one of rwr_graph_hold_out");
        test_ptr = g->held_ptr.data();
        test_ids = g->held_ids.data();
    }
    if (n_users < 0 || (n_users && test_ptr[n_users] && !test_ids)) RWR_FAIL(RWR_E_INVALID, "bad test sets");
    for (int s = 0; s < n_users; s++) {
        if (users[s] < 0 || users[s] >= g->n) RWR_FAIL(RWR_E_BADSEED, "user %d outside [0, %d)", users[s], g->n);
        if (test_ptr[s + 1] < test_ptr[s]) RWR_FAIL(RWR_E_INVALID, "test_ptr is not ascending");
        if (n_test_of_user) n_test_of_user[s] = (int32_t)(test_ptr[s + 1] - test_ptr[s]);
    }
    if (n_users == 0) return RWR_OK;
    if (n_iter < 0) n_iter = 0;
    if (k < 0) k = 0;
    CUDA_CHECK(cudaSetDevice(g->device));
    AllocStream alloc_on(g->stream);
    if (precision == RWR_FP64) evaluate_tiles<double>(g, users, n_users, test_ptr, test_ids, c, n_iter, k, hits, avg_precision, hits_at_k, info);
    else evaluate_tiles<float>(g, users, n_users, test_ptr, test_ids, c, n_iter, k, hits, avg_precision, hits_at_k, info);
    return RWR_OK;
    RWR_API_END
}

// Experiment.cs:121-128 (+ :136): hits and average precision of a ranking against the held-out set
int rwr_evaluate(const int64_t* ranked_ids, int64_t n, const int64_t* test_ids, int64_t n_test, int32_t* hits,
                 double* avg_precision) {
    RWR_API_BEGIN
    if ((n && !ranked_ids) || (n_test && !test_ids) || !hits || !avg_precision || n < 0 || n_test < 0)
        RWR_FAIL(RWR_E_INVALID, "bad argument");
    std::unordered_set<int64_t> test(test_ids, test_ids + n_test);
    int nHits = 0;
    double sumPrecision = 0;
    for (int64_t i = 0; i < n; i++) {
        if (test.count(ranked_ids[i])) {
            nHits += 1;
            sumPrecision += (double)nHits / (double)(i + 1);
        }
    }
    *hits = nHits;
    *avg_precision = nHits == 0 ? 0.0 : sumPrecision / nHits;
    return RWR_OK;
    RWR_API_END
}

}  // extern "C"
