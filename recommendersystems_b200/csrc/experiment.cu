// experiment.cu -- the callers' side of the hot path (SURVEY section 8f, rows N2 and N3) on the device.
//
//   N3  rwr_methodology_masks   TweetRecommender/DataLoader.cs:142-219 (Methodology -> List<Feature>), Experiment.cs:84-101
//                               (FRIENDSHIP "temporarily included", then retyped UNDEFINED) as link-type masks of rwr_opts
//   N2  rwr_graph_hold_out      DataLoader.splitLikeHistory (DataLoader.cs:122-140) + the LIKE links of the test fold that
//                               never reach `edges` (DataLoader.cs:287-298), for many test users of one graph at once:
//                               candidate likes -> stable LSD sort by (user, tweet id) -> fold window -> both directions of
//                               every held-out like leave the raw link list (stable compaction, insertion order kept).
//                               A held-out tweet that no LIKE link reaches any more is no node of the reference's graph at
//                               all (DataLoader creates tweet nodes while it walks somebody's likes, :291-303, and
//                               addAuthorship skips tweets that are not nodes, :355-356): its remaining links leave too and
//                               its node type becomes UNDEFINED, so it is no candidate (Recommender.cs:29) and never a hit
//                               (Experiment.cs:124); the node index itself stays, indices do not shift
// The evaluation itself (N1, Experiment.cs:121-128) lives next to the top-k kernels in select.cu.
#include <algorithm>
#include <vector>

#include "graph.h"
#include "primitives.cuh"

// ------------------------------------------------------------------------------------------------ N3
// Feature bits (Experiment.cs:16)
enum { F_FRIENDSHIP = 1, F_FOLLOW3P = 2, F_AUTHORSHIP = 4, F_MENTION = 8 };

extern "C" int rwr_methodology_masks(int32_t methodology, int32_t* feature_mask, int32_t* undefined_type_mask,
                                     int32_t* zero_weight_type_mask) {
    // DataLoader.cs:144-214, in the order of the Methodology enum (Experiment.cs:7-15); `tmp`: the friendship links are
    // loaded ("temporarily included", they set the MENTION weights) and retyped UNDEFINED at Experiment.cs:84-101
    static const struct { int features; bool friendship_tmp; } table[16] = {
        {0, false},                                                        //  0 BASELINE
        {F_FRIENDSHIP, false},                                             //  1 INCL_FRIENDSHIP
        {F_FOLLOW3P, false},                                               //  2 INCL_FOLLOWSHIP_ON_THIRDPARTY
        {F_AUTHORSHIP, false},                                             //  3 INCL_AUTHORSHIP
        {F_FRIENDSHIP | F_MENTION, true},                                  //  4 INCL_MENTIONCOUNT
        {F_FRIENDSHIP | F_FOLLOW3P, false},                                //  5 INCL_ALLFOLLOWSHIP
        {F_FRIENDSHIP | F_AUTHORSHIP, false},                              //  6 INCL_FRIENDSHIP_AUTHORSHIP
        {F_FRIENDSHIP | F_MENTION, false},                                 //  7 INCL_FRIENDSHIP_MENTIONCOUNT
        {F_FRIENDSHIP | F_FOLLOW3P | F_AUTHORSHIP | F_MENTION, false},     //  8 ALL
        {F_FRIENDSHIP | F_FOLLOW3P | F_AUTHORSHIP | F_MENTION, true},      //  9 EXCL_FRIENDSHIP
        {F_FRIENDSHIP | F_AUTHORSHIP | F_MENTION, false},                  // 10 EXCL_FOLLOWSHIP_ON_THIRDPARTY
        {F_FRIENDSHIP | F_FOLLOW3P | F_MENTION, false},                    // 11 EXCL_AUTHORSHIP
        {F_FRIENDSHIP | F_FOLLOW3P | F_AUTHORSHIP, false},                 // 12 EXCL_MENTIONCOUNT
        {F_FOLLOW3P | F_AUTHORSHIP, false},                                // 13 INCL_FOLLOWSHIP_ON_THIRDPARTY_AND_AUTHORSHIP
        {F_FRIENDSHIP | F_FOLLOW3P | F_MENTION, true},                     // 14 INCL_FOLLOWSHIP_ON_THIRDPARTY_AND_MENTIONCOUNT
        {F_AUTHORSHIP | F_MENTION, false},                                 // 15 INCL_AUTHORSHIP_AND_MENTIONCOUNT
    };
    if (methodology < 0 || methodology > 15) {
        rwr_set_error("methodology %d outside 0..15 (Experiment.cs:7-15)", methodology);
        return RWR_E_INVALID;
    }
    const int f = table[methodology].features;
    int undef = 0, zero = 0;
    if (!(f & F_FRIENDSHIP) || table[methodology].friendship_tmp) undef |= 1 << RWR_EDGE_FRIENDSHIP;
    if (!(f & F_FOLLOW3P)) undef |= 1 << RWR_EDGE_FOLLOW;
    if (!(f & F_AUTHORSHIP)) undef |= 1 << RWR_EDGE_AUTHORSHIP;
    if (!(f & F_MENTION)) undef |= 1 << RWR_EDGE_MENTION;
    // mention weights are nFriendhips * ln(cnt) / sum(ln cnt) with nFriendhips counted in allLinks (DataLoader.cs:423-434):
    // without the FRIENDSHIP feature no such link was loaded and every MENTION weight is exactly 0.0
    if ((f & F_MENTION) && !(f & F_FRIENDSHIP)) zero |= 1 << RWR_EDGE_MENTION;
    if (feature_mask) *feature_mask = f;
    if (undefined_type_mask) *undefined_type_mask = undef;
    if (zero_weight_type_mask) *zero_weight_type_mask = zero;
    return RWR_OK;
}

// ------------------------------------------------------------------------------------------------ N2
namespace {

constexpr u64 HS_EMPTY = ~0ULL;

__device__ __forceinline__ u32 hs_hash(u64 k) {
    k ^= k >> 33; k *= 0xff51afd7ed558ccdULL; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL; k ^= k >> 33;
    return (u32)k;
}
__device__ __forceinline__ void hs_insert(u64* tab, u32 mask, u64 key) {
    u32 h = hs_hash(key) & mask;
    while (true) {
        const u64 prev = atomicCAS((unsigned long long*)&tab[h], (unsigned long long)HS_EMPTY, (unsigned long long)key);
        if (prev == HS_EMPTY || prev == key) return;
        h = (h + 1) & mask;
    }
}
__device__ __forceinline__ bool hs_has(const u64* __restrict__ tab, u32 mask, u64 key) {
    u32 h = hs_hash(key) & mask;
    while (true) {
        const u64 v = tab[h];
        if (v == key) return true;
        if (v == HS_EMPTY) return false;
        h = (h + 1) & mask;
    }
}

__device__ __forceinline__ bool is_like_of_item(u8 t, int32_t d, const u8* __restrict__ node_type, int n) {
    return t == RWR_EDGE_LIKE && d >= 0 && d < n && node_type[d] == RWR_NODE_ITEM;
}

// likes(u): one warp per test user counts / lists the user's raw LIKE links to ITEM nodes (insertion order kept)
__global__ void k_ho_count(const int32_t* __restrict__ users, int n_users, const u32* __restrict__ raw_ptr,
                           const int32_t* __restrict__ raw_dst, const u8* __restrict__ raw_type,
                           const u8* __restrict__ node_type, int n, u32* __restrict__ cnt) {
    const int w = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= n_users) return;
    const int u = users[w];
    const u32 b = raw_ptr[u], e = raw_ptr[u + 1];
    u32 c = 0;
    for (u32 i = b + lane; i < e; i += 32) c += is_like_of_item(raw_type[i], raw_dst[i], node_type, n);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if (lane == 0) cnt[w] = c;
}

__global__ void k_ho_fill(const int32_t* __restrict__ users, int n_users, const u32* __restrict__ raw_ptr,
                          const int32_t* __restrict__ raw_dst, const u8* __restrict__ raw_type,
                          const u8* __restrict__ node_type, const int64_t* __restrict__ node_id, int n,
                          const u32* __restrict__ off, u64* __restrict__ key_id, u32* __restrict__ pos_iota,
                          u32* __restrict__ link, u32* __restrict__ slot) {
    const int w = (int)(((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (w >= n_users) return;
    const int u = users[w];
    const u32 b = raw_ptr[u], e = raw_ptr[u + 1];
    u32 run = off[w];
    const u32 lt = (1u << lane) - 1u;
    for (u32 base = b; base < e; base += 32) {
        const u32 i = base + lane;
        const bool ok = i < e && is_like_of_item(raw_type[i], raw_dst[i], node_type, n);
        const u32 m = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            const u32 p = run + __popc(m & lt);
            key_id[p] = (u64)node_id[raw_dst[i]] ^ 0x8000000000000000ULL;      // signed order -> unsigned order
            pos_iota[p] = p;
            link[p] = i;
            slot[p] = (u32)w;
        }
        run += __popc(m);
    }
}

__global__ void k_ho_slot_keys(const u32* __restrict__ perm1, const u32* __restrict__ slot, size_t m, u32* __restrict__ keys2) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) keys2[i] = slot[perm1[i]];
}

// DataLoader.cs:131-133: unitSize = likes.Count / nFolds; the last fold takes the remainder
__device__ __forceinline__ void fold_window(u32 cnt, int n_folds, int fold, u32* lo, u32* hi) {
    const u32 unit = cnt / (u32)n_folds;
    *lo = unit * (u32)fold;
    *hi = (fold < n_folds - 1) ? unit * (u32)(fold + 1) : cnt;
}

__global__ void k_ho_tcount(const u32* __restrict__ off, int n_users, int n_folds, int fold, u32* __restrict__ tcnt) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_users) return;
    u32 lo, hi;
    fold_window(off[s + 1] - off[s], n_folds, fold, &lo, &hi);
    tcnt[s] = hi - lo;
}

// q-th entry of the (user slot, tweet id) order: held out iff its position inside the user's likes is in the fold window
__global__ void k_ho_select(const u32* __restrict__ perm2, const u32* __restrict__ slot, const u32* __restrict__ link,
                            const u32* __restrict__ off, const u32* __restrict__ toff, const int32_t* __restrict__ users,
                            const int32_t* __restrict__ raw_dst, const int64_t* __restrict__ node_id, size_t m, int n_folds,
                            int fold, u8* __restrict__ removed, int64_t* __restrict__ test_ids, u64* __restrict__ tab, u32 mask) {
    const size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const u32 p = perm2[q], s = slot[p];
    const u32 idx = (u32)q - off[s];
    u32 lo, hi;
    fold_window(off[s + 1] - off[s], n_folds, fold, &lo, &hi);
    if (idx < lo || idx >= hi) return;
    const u32 e = link[p];
    const int32_t t = raw_dst[e];
    removed[e] = 1;                                              // u -> t never added (DataLoader.cs:293 not executed)
    test_ids[toff[s] + (idx - lo)] = node_id[t];
    hs_insert(tab, mask, ((u64)(u32)t << 32) | (u64)(u32)users[s]);   // t -> u goes too (DataLoader.cs:294)
}

__global__ void k_ho_reverse(const int32_t* __restrict__ raw_src, const int32_t* __restrict__ raw_dst,
                             const u8* __restrict__ raw_type, const u8* __restrict__ node_type, size_t e0,
                             const u64* __restrict__ tab, u32 mask, u8* __restrict__ removed) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= e0) return;
    if (raw_type[e] != RWR_EDGE_LIKE) return;
    const int32_t s = raw_src[e];
    if (node_type[s] != RWR_NODE_ITEM) return;
    if (hs_has(tab, mask, ((u64)(u32)s << 32) | (u64)(u32)raw_dst[e])) removed[e] = 1;
}

// ---- held-out tweets nobody likes any more (see the header) ----------------------------------------------------------
// remaining LIKE links into ITEM nodes, per target
__global__ void k_ho_like_in(const int32_t* __restrict__ raw_dst, const u8* __restrict__ raw_type, const u8* __restrict__ node_type,
                             int n, size_t e0, const u8* __restrict__ removed, u32* __restrict__ like_in) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= e0 || removed[e]) return;
    if (is_like_of_item(raw_type[e], raw_dst[e], node_type, n)) atomicAdd(&like_in[raw_dst[e]], 1u);
}
// a removed LIKE link into an ITEM is the u -> t half of a held-out like: t is an orphan when nothing is left in like_in[t]
__global__ void k_ho_orphans(const int32_t* __restrict__ raw_dst, const u8* __restrict__ raw_type, const u8* __restrict__ node_type,
                             int n, size_t e0, const u8* __restrict__ removed, const u32* __restrict__ like_in,
                             u8* __restrict__ orphan, u32* __restrict__ any) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= e0 || !removed[e]) return;
    if (is_like_of_item(raw_type[e], raw_dst[e], node_type, n) && like_in[raw_dst[e]] == 0) {
        orphan[raw_dst[e]] = 1;
        *any = 1u;
    }
}
__global__ void k_ho_drop_orphan_links(const int32_t* __restrict__ raw_src, const int32_t* __restrict__ raw_dst, int n, size_t e0,
                                       const u8* __restrict__ orphan, u8* __restrict__ removed) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= e0) return;
    const int32_t s = raw_src[e], d = raw_dst[e];
    if (((u32)s < (u32)n && orphan[s]) || ((u32)d < (u32)n && orphan[d])) removed[e] = 1;
}
__global__ void k_ho_retype_orphans(const u8* __restrict__ orphan, int n, u8* __restrict__ node_type) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n && orphan[j]) node_type[j] = RWR_NODE_UNDEFINED;
}

__global__ void k_ho_keep_flags(const u8* __restrict__ removed, size_t e0, u32* __restrict__ flags) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < e0) flags[e] = removed[e] ? 0u : 1u;
}

__global__ void k_ho_compact(const u8* __restrict__ removed, const u32* __restrict__ pos, const int32_t* __restrict__ src,
                             const int32_t* __restrict__ dst, const u8* __restrict__ type, const double* __restrict__ w,
                             size_t e0, int32_t* __restrict__ src2, int32_t* __restrict__ dst2, u8* __restrict__ type2,
                             double* __restrict__ w2) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < e0 && !removed[e]) {
        const u32 p = pos[e];
        src2[p] = src[e]; dst2[p] = dst[e]; type2[p] = type[e]; w2[p] = w[e];
    }
}

__global__ void k_fill_u64(u64* p, size_t n, u64 v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

inline unsigned grid_of(size_t n, int block = 256) { return n ? div_up(n, block) : 1; }

}  // namespace

void graph_rebuild_raw_ptr(rwr_graph* g);      // graph.cu

extern "C" int rwr_graph_hold_out(rwr_graph* g, const int32_t* users, int32_t n_users, int32_t n_folds, int32_t fold,
                                  int64_t* test_ptr, int64_t* test_ids, int64_t cap, int64_t* n_test) {
    RWR_API_BEGIN
    if (!g || (n_users && !users) || n_users < 0) RWR_FAIL(RWR_E_INVALID, "bad argument");
    if (g->built) RWR_FAIL(RWR_E_ALREADY_BUILT, "hold-out edits `edges`: call it before buildGraph()");
    if (g->comm) RWR_FAIL(RWR_E_UNSUPPORTED, "hold-out on a row-partitioned handle: evaluate on replicated graphs, users sharded over the ranks");
    if (n_folds < 1 || fold < 0 || fold >= n_folds) RWR_FAIL(RWR_E_INVALID, "fold %d of %d", fold, n_folds);
    for (int i = 0; i < n_users; i++)
        if (users[i] < 0 || users[i] >= g->n) RWR_FAIL(RWR_E_BADSEED, "user %d outside [0, %d)", users[i], g->n);
    {
        std::vector<int32_t> sorted(users, users + n_users);
        std::sort(sorted.begin(), sorted.end());
        if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end()) RWR_FAIL(RWR_E_INVALID, "a test user is listed twice");
    }
    CUDA_CHECK(cudaSetDevice(g->device));
    cudaStream_t st = g->stream;
    AllocStream alloc_on(st);
    const size_t e0 = (size_t)g->e0;
    const int n = g->n;
    g->held_users.assign(users, users + n_users);
    g->held_ptr.assign((size_t)n_users + 1, 0);
    g->held_ids.clear();
    if (n_test) *n_test = 0;
    if (test_ptr) std::fill(test_ptr, test_ptr + n_users + 1, (int64_t)0);
    if (n_users == 0 || e0 == 0) return RWR_OK;

    DevBuf<int32_t> d_users;
    DevBuf<u32> off, toff;
    d_users.alloc(n_users); off.alloc((size_t)n_users + 1); toff.alloc((size_t)n_users + 1);
    CUDA_CHECK(cudaMemcpyAsync(d_users.p, users, (size_t)n_users * 4, cudaMemcpyHostToDevice, st));
    const unsigned wgrid = grid_of((size_t)n_users * 32);
    k_ho_count<<<wgrid, 256, 0, st>>>(d_users.p, n_users, g->raw_ptr.p, g->raw_dst.p, g->raw_type.p, g->node_type.p, n, off.p);
    KERNEL_CHECK();
    const size_t m = prim::scan_total<u32>(off.p, off.p, n_users, true, st, &g->pool);
    if (m == 0) return RWR_OK;

    // ---- (user slot, tweet id) order of the candidate likes: LSD sort by id, then a stable pass by slot
    prim::SortBuffers<u64> by_id;
    DevBuf<u32> link, slot;
    by_id.alloc(m, true); link.alloc(m); slot.alloc(m);
    k_ho_fill<<<wgrid, 256, 0, st>>>(d_users.p, n_users, g->raw_ptr.p, g->raw_dst.p, g->raw_type.p, g->node_type.p, g->node_id.p, n,
                                     off.p, by_id.keys(), by_id.vals(), link.p, slot.p);
    KERNEL_CHECK();
    by_id.sort(m, 64, st, &g->pool);
    prim::SortBuffers<u32> by_slot;
    by_slot.alloc(m, true);
    k_ho_slot_keys<<<grid_of(m), 256, 0, st>>>(by_id.vals(), slot.p, m, by_slot.keys());
    KERNEL_CHECK();
    CUDA_CHECK(cudaMemcpyAsync(by_slot.vals(), by_id.vals(), m * 4, cudaMemcpyDeviceToDevice, st));
    by_slot.sort(m, std::max(1, ceil_log2_u64((u64)n_users)), st, &g->pool);
    const u32* perm2 = by_slot.vals();

    // ---- fold windows -> test sets, removed flags, reverse links
    k_ho_tcount<<<grid_of(n_users), 256, 0, st>>>(off.p, n_users, n_folds, fold, toff.p);
    KERNEL_CHECK();
    const size_t held = prim::scan_total<u32>(toff.p, toff.p, n_users, true, st, &g->pool);
    std::vector<u32> h_toff((size_t)n_users + 1);
    CUDA_CHECK(cudaMemcpyAsync(h_toff.data(), toff.p, ((size_t)n_users + 1) * 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    for (int i = 0; i <= n_users; i++) g->held_ptr[i] = (int64_t)h_toff[i];
    if (test_ptr) std::copy(g->held_ptr.begin(), g->held_ptr.end(), test_ptr);
    if (n_test) *n_test = (int64_t)held;
    if (held == 0) return RWR_OK;

    u32 cap_tab = 64;
    while ((size_t)cap_tab < 2 * held + 16) cap_tab <<= 1;
    DevBuf<u64> tab;
    DevBuf<u8> removed;
    DevBuf<int64_t> d_test;
    tab.alloc(cap_tab); removed.alloc(e0); d_test.alloc(held);
    k_fill_u64<<<grid_of(cap_tab), 256, 0, st>>>(tab.p, cap_tab, HS_EMPTY);
    CUDA_CHECK(cudaMemsetAsync(removed.p, 0, e0, st));
    k_ho_select<<<grid_of(m), 256, 0, st>>>(perm2, slot.p, link.p, off.p, toff.p, d_users.p, g->raw_dst.p, g->node_id.p, m, n_folds,
                                           fold, removed.p, d_test.p, tab.p, cap_tab - 1);
    k_ho_reverse<<<grid_of(e0), 256, 0, st>>>(g->raw_src.p, g->raw_dst.p, g->raw_type.p, g->node_type.p, e0, tab.p, cap_tab - 1,
                                             removed.p);
    KERNEL_CHECK();
    g->held_ids.resize(held);
    CUDA_CHECK(cudaMemcpyAsync(g->held_ids.data(), d_test.p, held * 8, cudaMemcpyDeviceToHost, st));

    // ---- held-out tweets that no LIKE link reaches any more leave the graph (their other links, their candidacy)
    {
        DevBuf<u32> like_in, any;
        DevBuf<u8> orphan;
        like_in.alloc((size_t)n); any.alloc(1); orphan.alloc((size_t)n);
        CUDA_CHECK(cudaMemsetAsync(like_in.p, 0, (size_t)n * sizeof(u32), st));
        CUDA_CHECK(cudaMemsetAsync(any.p, 0, sizeof(u32), st));
        CUDA_CHECK(cudaMemsetAsync(orphan.p, 0, (size_t)n, st));
        k_ho_like_in<<<grid_of(e0), 256, 0, st>>>(g->raw_dst.p, g->raw_type.p, g->node_type.p, n, e0, removed.p, like_in.p);
        k_ho_orphans<<<grid_of(e0), 256, 0, st>>>(g->raw_dst.p, g->raw_type.p, g->node_type.p, n, e0, removed.p, like_in.p, orphan.p,
                                                 any.p);
        KERNEL_CHECK();
        u32 h_any = 0;
        CUDA_CHECK(cudaMemcpyAsync(&h_any, any.p, sizeof(u32), cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
        if (h_any) {
            k_ho_drop_orphan_links<<<grid_of(e0), 256, 0, st>>>(g->raw_src.p, g->raw_dst.p, n, e0, orphan.p, removed.p);
            k_ho_retype_orphans<<<grid_of((size_t)n), 256, 0, st>>>(orphan.p, n, g->node_type.p);
            KERNEL_CHECK();
            g->pool.launches += 2;
        }
        g->pool.launches += 2;
    }

    // ---- stable compaction of `edges`
    DevBuf<u32> pos;
    pos.alloc(e0);
    k_ho_keep_flags<<<grid_of(e0), 256, 0, st>>>(removed.p, e0, pos.p);
    KERNEL_CHECK();
    const u32 kept = prim::scan_total<u32>(pos.p, pos.p, e0, false, st, &g->pool);
    DevBuf<int32_t> src2, dst2;
    DevBuf<u8> type2;
    DevBuf<double> w2;
    src2.alloc(kept, &g->pool); dst2.alloc(kept, &g->pool); type2.alloc(kept, &g->pool); w2.alloc(kept, &g->pool);
    k_ho_compact<<<grid_of(e0), 256, 0, st>>>(removed.p, pos.p, g->raw_src.p, g->raw_dst.p, g->raw_type.p, g->raw_w.p, e0, src2.p,
                                             dst2.p, type2.p, w2.p);
    KERNEL_CHECK();
    CUDA_CHECK(cudaStreamSynchronize(st));
    g->raw_src = std::move(src2);
    g->raw_dst = std::move(dst2);
    g->raw_type = std::move(type2);
    g->raw_w = std::move(w2);
    g->e0 = (int64_t)kept;
    graph_rebuild_raw_ptr(g);
    g->pool.launches += 9;
    if (test_ids && cap > 0) std::copy(g->held_ids.begin(), g->held_ids.begin() + std::min<size_t>(held, (size_t)cap), test_ids);
    return RWR_OK;
    RWR_API_END
}
