// synth.cu -- K0: deterministic synthetic graph generator on the device.
//
// Replaces the SQLite-sourced graph assembly of TweetRecommender/DataLoader.cs:256-436 (member nodes, tweet nodes +
// bidirectional LIKE, FRIENDSHIP / FOLLOW, AUTHORSHIP, MENTION weights) and its (target, type) dedup on insert
// (DataLoader.cs:60-77).  Spec: include/rwr_b200.h `rwr_synth_spec`.  Integer-only and counter-based, so the CPU
// generator of the oracle produces the same links bit for bit:
//   relation j -> endpoints by per-bit Bernoulli draws on mix64 hashes (R-MAT-style skew), optional scramble;
//   every relation emits up to two 64-bit keys (src << 31 | class << 28 | dst); sort, unique, drop the sentinel;
//   canonical "insertion order" of a source = (class: LIKE, FRIENDSHIP, FOLLOW, AUTHORSHIP, MENTION; then target).
#include <algorithm>

#include "dist.h"
#include "graph.h"
#include "primitives.cuh"

namespace {

__host__ __device__ __forceinline__ u64 mix64(u64 z) {
    z ^= z >> 30; z *= 0xbf58476d1ce4e5b9ULL;
    z ^= z >> 27; z *= 0x94d049bb133111ebULL;
    z ^= z >> 31;
    return z;
}
__device__ __forceinline__ u64 hashH(u64 seed, u64 j, u64 k) {
    return mix64(mix64(seed + 0x9E3779B97F4A7C15ULL * (j + 1)) + 0xD1B54A32D192ED03ULL * (k + 1));
}

struct SynthDev {
    u64 seed;
    u64 U, T, X;
    int LU, LT, LX;           // ceil(log2(range))
    u64 offU, offT;           // scramble offsets, mix64(seed ^ salt) % range
    int scramble;
    u32 p1;
    u32 auth_pm, undef_pm;
    u64 r_like, r_friend, r_follow, r_mention, nrel;
};

constexpr u64 SALT_U = 0x1111111111111111ULL, SALT_T = 0x2222222222222222ULL;
constexpr u64 SALT_UNDEF = 0xF1E2D3C4B5A69788ULL, SALT_MENTION = 0xA5A5A5A55A5A5A5AULL;
constexpr u64 INVALID_KEY = ~0ULL;
enum { CLS_LIKE = 0, CLS_FRIEND = 1, CLS_FOLLOW = 2, CLS_AUTHOR = 3, CLS_MENTION = 4 };

__device__ __forceinline__ u64 draw(const SynthDev& s, u64 j, int which, u64 range, int L) {
    u64 v = 0, h = 0;
    for (int l = 0; l < L; l++) {
        if ((l & 7) == 0) h = hashH(s.seed, j, (u64)(which * 4 + (l >> 3)));
        const u64 byte = (h >> (8 * (l & 7))) & 255;
        v |= (u64)(byte < (u64)s.p1) << l;
    }
    return v % range;
}
__device__ __forceinline__ u64 permU(const SynthDev& s, u64 x) { return s.scramble ? (x * 2654435761ULL + s.offU) % s.U : x; }
__device__ __forceinline__ u64 permT(const SynthDev& s, u64 x) { return s.scramble ? (x * 2654435761ULL + s.offT) % s.T : x; }
__device__ __forceinline__ u64 make_key(u64 src, int cls, u64 dst) { return (src << 31) | ((u64)cls << 28) | dst; }

// the (up to) two keys of relation j
__device__ __forceinline__ void relation_keys(const SynthDev& s, u64 j, u64& k0, u64& k1) {
    k0 = INVALID_KEY; k1 = INVALID_KEY;
    if (j < s.r_like) {
        if ((hashH(s.seed, j, 15) % 1000) < (u64)s.auth_pm) {
            const u64 a = permU(s, draw(s, j, 0, s.U, s.LU)), it = s.U + j;
            k0 = make_key(a, CLS_AUTHOR, it);
            k1 = make_key(it, CLS_AUTHOR, a);
        }
    } else if (j < s.r_friend) {
        const u64 u = permU(s, draw(s, j, 0, s.U, s.LU)), it = s.U + permT(s, draw(s, j, 1, s.T, s.LT));
        k0 = make_key(u, CLS_LIKE, it);
        k1 = make_key(it, CLS_LIKE, u);
    } else if (j < s.r_follow) {
        const u64 u = permU(s, draw(s, j, 0, s.U, s.LU)), v = permU(s, draw(s, j, 1, s.U, s.LU));
        if (u != v) {
            k0 = make_key(u, CLS_FRIEND, v);
            k1 = make_key(v, CLS_FRIEND, u);
        }
    } else if (j < s.r_mention) {
        const u64 u = permU(s, draw(s, j, 0, s.U, s.LU)), x = s.U + s.T + draw(s, j, 1, s.X, s.LX);
        k0 = make_key(u, CLS_FOLLOW, x);
        k1 = make_key(x, CLS_FOLLOW, u);
    } else {
        const u64 u = permU(s, draw(s, j, 0, s.U, s.LU)), v = permU(s, draw(s, j, 1, s.U, s.LU));
        if (u != v) k0 = make_key(u, CLS_MENTION, v);
    }
}

__global__ void k_synth_keys(const SynthDev s, u64* __restrict__ keys) {
    const u64 j = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= s.nrel) return;
    u64 k0, k1;
    relation_keys(s, j, k0, k1);
    keys[2 * j] = k0;
    keys[2 * j + 1] = k1;
}

// Partitioned build: only the keys whose SOURCE this rank owns.  Pass 1 (keys == null) counts them, pass 2 appends them in
// any order (the sort that follows makes the order canonical); one atomic per warp.
__global__ void k_synth_keys_owned(const SynthDev s, const OwnMap own, u64 j0, u64 j1, u64* __restrict__ keys,
                                   unsigned long long* __restrict__ counter) {
    const u64 j = j0 + (u64)blockIdx.x * blockDim.x + threadIdx.x;
    u64 k0 = INVALID_KEY, k1 = INVALID_KEY;
    if (j < j1) relation_keys(s, j, k0, k1);
    const bool m0 = k0 != INVALID_KEY && own_rank(own, (long long)(k0 >> 31)) == own.rank;
    const bool m1 = k1 != INVALID_KEY && own_rank(own, (long long)(k1 >> 31)) == own.rank;
    const int mine = (int)m0 + (int)m1;
    const int lane = threadIdx.x & 31;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    unsigned long long base = 0;
    if (lane == 31 && total) base = atomicAdd(counter, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 31);
    if (keys) {
        unsigned long long p = base + (unsigned long long)(incl - mine);
        if (m0) keys[p++] = k0;
        if (m1) keys[p] = k1;
    }
}

__global__ void k_unique_flags(const u64* __restrict__ keys, size_t n, u32* __restrict__ flags) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const u64 k = keys[i];
        flags[i] = (k != INVALID_KEY) && (i == 0 || keys[i - 1] != k);
    }
}

__global__ void k_emit_links(const SynthDev s, const u64* __restrict__ keys, const u32* __restrict__ pos, size_t n,
                             int32_t* __restrict__ src, int32_t* __restrict__ dst, u8* __restrict__ type, double* __restrict__ w) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 k = keys[i];
    if (k == INVALID_KEY || (i > 0 && keys[i - 1] == k)) return;
    const u64 sN = k >> 31, dN = k & ((1ULL << 28) - 1);
    const int cls = (int)((k >> 28) & 7);
    int et = RWR_EDGE_UNDEFINED;
    double wt = 1.0;
    switch (cls) {
        case CLS_LIKE: et = RWR_EDGE_LIKE; break;
        case CLS_FRIEND: {
            const u64 lo = sN < dN ? sN : dN, hi = sN < dN ? dN : sN;
            const bool undef = (mix64(s.seed ^ SALT_UNDEF ^ ((lo << 32) | hi)) % 1000) < (u64)s.undef_pm;
            et = undef ? RWR_EDGE_UNDEFINED : RWR_EDGE_FRIENDSHIP;
        } break;
        case CLS_FOLLOW: et = RWR_EDGE_FOLLOW; break;
        case CLS_AUTHOR: et = RWR_EDGE_AUTHORSHIP; break;
        default:
            et = RWR_EDGE_MENTION;
            wt = (double)(1 + (mix64(s.seed ^ SALT_MENTION ^ ((sN << 32) | dN)) & 127)) / 32.0;
            break;
    }
    const u32 p = pos[i];
    src[p] = (int32_t)sN; dst[p] = (int32_t)dN; type[p] = (u8)et; w[p] = wt;
}

__global__ void k_synth_nodes(u64 U, u64 T, u64 N, int64_t* __restrict__ id, u8* __restrict__ type) {
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    if (i < U) { id[i] = 1000000000LL + (int64_t)i; type[i] = RWR_NODE_USER; }
    else if (i < U + T) { id[i] = 5000000000000LL + (int64_t)(i - U); type[i] = RWR_NODE_ITEM; }
    else { id[i] = 2000000000LL + (int64_t)(i - U - T); type[i] = RWR_NODE_ETC; }
}

}  // namespace

// Generates the canonical link list on g's device.  Shared by rwr_synth_create and the partitioned variant.
void synth_generate_device(rwr_graph* g, const rwr_synth_spec* spec) {
    cudaStream_t st = g->stream;
    if (spec->n_users < 1 || spec->n_items < 0 || spec->n_third < 0 || spec->n_like < 0 || spec->n_friend < 0 ||
        spec->n_follow < 0 || spec->n_mention < 0)
        RWR_FAIL(RWR_E_INVALID, "bad synthetic spec");
    SynthDev s;
    s.seed = spec->seed;
    s.U = (u64)spec->n_users; s.T = (u64)spec->n_items; s.X = (u64)spec->n_third;
    const u64 N = s.U + s.T + s.X;
    if (N >= (1ULL << 28)) RWR_FAIL(RWR_E_UNSUPPORTED, "more than 2^28-1 nodes");
    if ((spec->n_like > 0 && s.T == 0) || (spec->n_follow > 0 && s.X == 0)) RWR_FAIL(RWR_E_INVALID, "relations need nodes");
    s.LU = ceil_log2_u64(s.U); s.LT = ceil_log2_u64(std::max<u64>(s.T, 1)); s.LX = ceil_log2_u64(std::max<u64>(s.X, 1));
    s.offU = mix64(s.seed ^ SALT_U) % s.U;
    s.offT = s.T ? mix64(s.seed ^ SALT_T) % s.T : 0;
    s.scramble = spec->scramble;
    s.p1 = (u32)spec->p1_byte;
    s.auth_pm = (u32)spec->authorship_per_mille;
    s.undef_pm = (u32)spec->undefined_per_mille;
    s.r_like = s.T;
    s.r_friend = s.r_like + (u64)spec->n_like;
    s.r_follow = s.r_friend + (u64)spec->n_friend;
    s.r_mention = s.r_follow + (u64)spec->n_follow;
    s.nrel = s.r_mention + (u64)spec->n_mention;
    size_t slots = (size_t)(2 * s.nrel);
    const bool owned = g->part_build;
    if (owned) {
        // who holds which source: users, items and third-party users are three populations with very different degrees, so
        // each of them is dealt evenly over the ranks (ids inside a class carry no locality when `scramble` is on)
        OwnMap& own = g->own;
        own.parts = dist_n_ranks(g->comm);
        own.rank = dist_rank(g->comm);
        own.n_segs = 0;
        own.seg[0] = 0;
        for (u64 len : {s.U, s.T, s.X})
            if (len) { own.seg[own.n_segs + 1] = own.seg[own.n_segs] + (long long)len; own.n_segs++; }
    } else if (slots >= (1ULL << 32) - 65536) {
        RWR_FAIL(RWR_E_UNSUPPORTED, "more than 2^32-65537 link slots per device");
    }

    DevEvent ev0, ev1;
    CUDA_CHECK(cudaEventRecord(ev0, st));

    g->n = (int32_t)N;
    g->node_id.alloc(N, &g->pool);
    g->node_type.alloc(N, &g->pool);
    k_synth_nodes<<<div_up(N, 256), 256, 0, st>>>(s.U, s.T, N, g->node_id.p, g->node_type.p);
    KERNEL_CHECK();

    prim::SortBuffers<u64> sb;
    if (owned) {
        DevBuf<unsigned long long> counter;
        counter.alloc(1);
        const u64 CH = 1ULL << 30;                        // relations per launch (grid size limit)
        unsigned long long mine = 0;
        for (int pass = 0; pass < 2; pass++) {
            CUDA_CHECK(cudaMemsetAsync(counter.p, 0, sizeof(unsigned long long), st));
            for (u64 j0 = 0; j0 < s.nrel; j0 += CH) {
                const u64 j1 = std::min(s.nrel, j0 + CH);
                k_synth_keys_owned<<<div_up((size_t)(j1 - j0), 256), 256, 0, st>>>(s, g->own, j0, j1, pass ? sb.keys() : nullptr, counter.p);
                KERNEL_CHECK();
            }
            if (pass == 0) {
                CUDA_CHECK(cudaMemcpyAsync(&mine, counter.p, sizeof(mine), cudaMemcpyDeviceToHost, st));
                CUDA_CHECK(cudaStreamSynchronize(st));
                if (mine >= (1ULL << 32) - 65536) RWR_FAIL(RWR_E_UNSUPPORTED, "more than 2^32-65537 link slots on one rank");
                slots = (size_t)mine;
                sb.alloc(slots, false);
            }
        }
    } else {
        sb.alloc(slots, false);
        if (s.nrel) {
            k_synth_keys<<<div_up((size_t)s.nrel, 256), 256, 0, st>>>(s, sb.keys());
            KERNEL_CHECK();
        }
    }
    // the all-ones sentinel must sort last: include every bit when any slot can be invalid
    sb.sort(slots, 64, st, &g->pool);
    sb.release_spare();
    const u64* sorted = sb.keys();
    DevBuf<u32> pos;
    pos.alloc(slots);
    if (slots) {
        k_unique_flags<<<div_up(slots, 256), 256, 0, st>>>(sorted, slots, pos.p);
        KERNEL_CHECK();
    }
    const u32 e0 = prim::scan_total<u32>(pos.p, pos.p, slots, false, st, &g->pool);
    g->e0 = (int64_t)e0;
    g->raw_src.alloc(e0, &g->pool);
    g->raw_dst.alloc(e0, &g->pool);
    g->raw_type.alloc(e0, &g->pool);
    g->raw_w.alloc(e0, &g->pool);
    if (slots) {
        k_emit_links<<<div_up(slots, 256), 256, 0, st>>>(s, sorted, pos.p, slots, g->raw_src.p, g->raw_dst.p, g->raw_type.p, g->raw_w.p);
        KERNEL_CHECK();
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
    g->pool.launches += 4;
    pos.release();
    sb.release();
    graph_finish_create(g);     // already source-ascending: only raw_ptr is built
    CUDA_CHECK(cudaEventRecord(ev1, st));
    CUDA_CHECK(cudaEventSynchronize(ev1));
    CUDA_CHECK(cudaEventElapsedTime(&g->synth_ms, ev0, ev1));
}

extern "C" int rwr_synth_create(const rwr_synth_spec* spec, const rwr_opts* opts, rwr_graph** out) {
    rwr_graph* g = nullptr;
    try {
        if (!out || !spec) RWR_FAIL(RWR_E_INVALID, "NULL argument");
        *out = nullptr;
        g = new rwr_graph();
        graph_init_device(g, opts);
        AllocStream alloc_on(g->stream);
        synth_generate_device(g, spec);
        *out = g;
        return RWR_OK;
    } catch (const RwrError& e) {
        rwr_graph_destroy(g);
        return e.code;
    } catch (...) {
        rwr_graph_destroy(g);
        rwr_set_error("unexpected exception");
        return RWR_E_INVALID;
    }
}
