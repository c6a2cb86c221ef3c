// frontier.cu -- the sparse prefix of a single-seed fixed-count run: iterations pushed from the frontier.
//
// x_0 of a seeded run has one nonzero entry, x_1 a handful: the first iterations read a tiny share of the links that the
// edge stream of stream.cu walks in full.  For iteration k, with the frontier F (the nonzero entries of x_{k-1}, original
// labels ascending):
//   extract  the frontier bitmap (original labels) -> F and the out-degrees of F; the bitmap is cleared on the way
//   scan     exclusive prefix of the degrees -> push links L; L > budget clears ctl->sparse: the run is dense from here
//   expand   one (target internal label, product) entry per push link, in the reference's accumulation order (F
//            ascending, then the links of a source in push-CSR order, Model.cs:85-88), plus a zero entry for the seed row
//   sort     stable LSD radix sort by target, as many 8-bit passes as n needs
//   sum      each target's run added in order in double from 0.0, then exactly the per-row epilogue of k_finish_ws, the
//            restart mass reduced through per-block slots in a fixed order; the active rows with inv != 0 go into the
//            bitmap for the next iteration
// No floating-point atomics: a run is bit-reproducible.  Every kernel returns at once when ctl->sparse is clear, so the
// launches can be captured in the iteration graph of any seed; the dense kernels skip the iterations counted in
// ctl->sparse_iters.  Grids and buffers are sized for the budget on the host; the counts live on the device.
#include <cmath>
#include <cstdlib>

#include "frontier.h"
#include "iterate_dev.cuh"
#include "primitives.cuh"
#include "stream.h"
#include "dist.h"

constexpr int FR_THREADS = 256;
constexpr int FR_ITEMS = 8;
constexpr int FR_TILE = FR_THREADS * FR_ITEMS;   // 2048
constexpr int FR_WARPS = FR_THREADS / 32;

struct FrDev {
    IterCtl* ctl;
    u32* sc;
    const u32* row_ptr;
    const int32_t* col;
    const double* val;              // valued layout: normalised weights of the push CSR; null: index-only
    const int32_t* new_of_old;
    const int32_t* old_of_new;
    int n;
    u32 words;
    u64 nnz, budget;
    u32 *bits, *fid, *fdeg, *foff, *bsum, *table;
};

// Only k_fr_extract and k_fr_expand clear the flag; no other kernel sees it change while it runs.
__device__ __forceinline__ bool fr_off(const FrDev& d) { return d.ctl->sparse == 0; }

// sum of bsum[0, b) over the block (result in every thread)
__device__ __forceinline__ u32 fr_prefix(const u32* bsum, int b, u32* red /* FR_WARPS + 1 */) {
    u32 s = 0;
    for (int i = threadIdx.x; i < b; i += FR_THREADS) s += bsum[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        u32 t = 0;
        for (int w = 0; w < FR_WARPS; w++) t += red[w];
        red[FR_WARPS] = t;
    }
    __syncthreads();
    const u32 r = red[FR_WARPS];
    __syncthreads();
    return r;
}

// ------------------------------------------------------------------------------------------------ frontier
__global__ void __launch_bounds__(FR_THREADS) k_fr_count(const FrDev d) {
    __shared__ u32 sm[9];
    if (fr_off(d)) return;
    const size_t base = (size_t)blockIdx.x * FR_TILE + (size_t)threadIdx.x * FR_ITEMS;
    u32 c = 0;
#pragma unroll
    for (int k = 0; k < FR_ITEMS; k++)
        if (base + k < d.words) c += __popc(d.bits[base + k]);
    u32 total;
    prim::block_exclusive_scan_256(c, &total, sm);
    if (threadIdx.x == 0) d.bsum[blockIdx.x] = total;
}

// bitmap -> frontier list (ascending) and out-degrees; clears the bitmap
// This kernel may clear ctl->sparse itself: every block reads the flag once, behind a barrier, so that all its threads
// agree and reach the barriers below together.
__global__ void __launch_bounds__(FR_THREADS) k_fr_extract(const FrDev d) {
    __shared__ u32 sm[9];
    __shared__ u32 red[FR_WARPS + 1];
    __shared__ int off;
    if (threadIdx.x == 0) off = fr_off(d);
    __syncthreads();
    if (off) return;
    const u32 nf = fr_prefix(d.bsum, gridDim.x, red);
    if (nf > d.budget) {                       // a frontier that large has more links than the budget
        if (blockIdx.x == 0 && threadIdx.x == 0) d.ctl->sparse = 0;
        return;
    }
    const u32 pre = fr_prefix(d.bsum, blockIdx.x, red);
    if (blockIdx.x == 0 && threadIdx.x == 0) d.sc[0] = nf;
    const size_t base = (size_t)blockIdx.x * FR_TILE + (size_t)threadIdx.x * FR_ITEMS;
    u32 w[FR_ITEMS];
    u32 c = 0;
#pragma unroll
    for (int k = 0; k < FR_ITEMS; k++) {
        w[k] = (base + k < d.words) ? d.bits[base + k] : 0u;
        c += __popc(w[k]);
    }
    u32 total;
    u32 pos = prim::block_exclusive_scan_256(c, &total, sm) + pre;
#pragma unroll
    for (int k = 0; k < FR_ITEMS; k++) {
        u32 m = w[k];
        if (!m) continue;
        d.bits[base + k] = 0u;
        while (m) {
            const u32 id = (u32)(base + k) * 32u + (u32)(__ffs(m) - 1);
            m &= m - 1;
            if (!RWR_CHK(id < (u32)d.n, d.ctl, 5)) continue;
            d.fid[pos] = id;
            d.fdeg[pos] = d.row_ptr[id + 1] - d.row_ptr[id];
            pos++;
        }
    }
}

// ------------------------------------------------------------------------------------------------ device-sized scan
// Exclusive scan of in[0, *len) into out (in place allowed), out[*len] = total.  Pass A: one sum per 2048-entry block;
// pass B: every block adds the sums of the blocks before it.
__global__ void __launch_bounds__(FR_THREADS) k_fr_scan_a(const FrDev d, const u32* __restrict__ in, const u32* len_ptr) {
    __shared__ u32 sm[9];
    if (fr_off(d)) return;
    const u32 len = *len_ptr;
    const size_t base = (size_t)blockIdx.x * FR_TILE + (size_t)threadIdx.x * FR_ITEMS;
    if ((size_t)blockIdx.x * FR_TILE >= len) return;
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < FR_ITEMS; k++)
        if (base + k < len) s += in[base + k];
    u32 total;
    prim::block_exclusive_scan_256(s, &total, sm);
    if (threadIdx.x == 0) d.bsum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(FR_THREADS) k_fr_scan_b(const FrDev d, const u32* in, u32* out, const u32* len_ptr) {
    __shared__ u32 sm[9];
    __shared__ u32 red[FR_WARPS + 1];
    if (fr_off(d)) return;
    const u32 len = *len_ptr;
    if (len == 0) {
        if (blockIdx.x == 0 && threadIdx.x == 0) out[0] = 0;
        return;
    }
    if ((size_t)blockIdx.x * FR_TILE >= len) return;
    const u32 pre = fr_prefix(d.bsum, blockIdx.x, red);
    const size_t base = (size_t)blockIdx.x * FR_TILE + (size_t)threadIdx.x * FR_ITEMS;
    u32 v[FR_ITEMS];
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < FR_ITEMS; k++) {
        v[k] = (base + k < len) ? in[base + k] : 0u;
        s += v[k];
    }
    u32 total;
    u32 ex = prim::block_exclusive_scan_256(s, &total, sm) + pre;
#pragma unroll
    for (int k = 0; k < FR_ITEMS; k++) {
        if (base + k < len) out[base + k] = ex;
        ex += v[k];
    }
    if (threadIdx.x == 0 && (size_t)(blockIdx.x + 1) * FR_TILE >= len) out[len] = pre + total;
}

// ------------------------------------------------------------------------------------------------ expand
// Entry i < L: the (i - foff[j])-th push link of frontier source j, the largest j with foff[j] <= i.  Entry L: the seed
// row with 0.0 (adding +0.0 to a sum of nonnegative terms changes no bit; it makes the seed row active).
template <typename T>
__global__ void __launch_bounds__(FR_THREADS) k_fr_expand(const FrDev d, const T* __restrict__ x, u32* __restrict__ key,
                                                         T* __restrict__ prod) {
    if (fr_off(d)) return;
    const u32 nf = d.sc[0];
    const u32 L = d.foff[nf];
    if (L > d.budget) {
        if (blockIdx.x == 0 && threadIdx.x == 0) d.ctl->sparse = 0;
        return;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) d.sc[1] = L + 1;
    const int seed = d.ctl->seed;               // from the device: a captured graph serves every seed
    for (u32 i = blockIdx.x * FR_THREADS + threadIdx.x; i <= L; i += gridDim.x * FR_THREADS) {
        if (i == L) { key[i] = (u32)seed; prod[i] = (T)0; continue; }
        u32 lo = 0, hi = nf;                 // foff[lo] <= i < foff[hi]
        while (hi - lo > 1) {
            const u32 mid = (lo + hi) >> 1;
            if (d.foff[mid] <= i) lo = mid; else hi = mid;
        }
        const u32 src = d.fid[lo];
        const u64 link = (u64)d.row_ptr[src] + (i - d.foff[lo]);
        if (!RWR_CHK(link < d.nnz, d.ctl, 5)) { key[i] = (u32)seed; prod[i] = (T)0; continue; }
        const int tgt = d.new_of_old[d.col[link]];
        const T xs = x[d.new_of_old[src]];
        key[i] = (u32)tgt;
        prod[i] = d.val ? mul_rn(xs, (T)d.val[link]) : xs;        // what k_spmv_ws forms for this link
    }
}

// ------------------------------------------------------------------------------------------------ radix sort
// One stable 8-bit pass of an LSD sort over the sc[1] entries (the same scheme as prim::SortBuffers, with the count on the
// device).  The digit table is digit-major over the tiles that hold entries.
__global__ void __launch_bounds__(FR_THREADS) k_fr_hist(const FrDev d, const u32* __restrict__ keys, int shift) {
    __shared__ u32 h[256];
    if (fr_off(d)) return;
    const u32 ne = d.sc[1];
    const u32 tiles = (ne + FR_TILE - 1) / FR_TILE;
    if (blockIdx.x >= tiles) return;
    if (blockIdx.x == 0 && threadIdx.x == 0) d.sc[2] = 256u * tiles;
    h[threadIdx.x] = 0;
    __syncthreads();
    const size_t base = (size_t)blockIdx.x * FR_TILE;
#pragma unroll
    for (int k = 0; k < FR_ITEMS; k++) {
        const size_t i = base + (size_t)k * FR_THREADS + threadIdx.x;
        if (i < ne) atomicAdd(&h[(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    d.table[(size_t)threadIdx.x * tiles + blockIdx.x] = h[threadIdx.x];
}

template <typename T>
__global__ void __launch_bounds__(FR_THREADS) k_fr_scatter(const FrDev d, const u32* __restrict__ keys_in, u32* __restrict__ keys_out,
                                                          const T* __restrict__ vals_in, T* __restrict__ vals_out, int shift) {
    __shared__ u32 wh[FR_WARPS][256];
    if (fr_off(d)) return;
    const u32 ne = d.sc[1];
    const u32 tiles = (ne + FR_TILE - 1) / FR_TILE;
    if (blockIdx.x >= tiles) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < FR_WARPS * 256; i += FR_THREADS) (&wh[0][0])[i] = 0;
    __syncthreads();
    // element order inside a tile is (warp, round, lane): ranking in that order keeps the sort stable
    const size_t wbase = (size_t)blockIdx.x * FR_TILE + (size_t)warp * (32 * FR_ITEMS);
    u32 key[FR_ITEMS], rank[FR_ITEMS];
    const u32 lt = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < FR_ITEMS; r++) {
        const size_t i = wbase + (size_t)r * 32 + lane;
        const bool valid = i < ne;
        key[r] = valid ? keys_in[i] : 0u;
        const u32 dg = valid ? ((key[r] >> shift) & 255u) : 256u;
        const u32 peers = __match_any_sync(0xffffffffu, dg);
        const int leader = __ffs(peers) - 1;
        u32 b = 0;
        if (valid && lane == leader) {
            b = wh[warp][dg];
            wh[warp][dg] = b + __popc(peers);
        }
        b = __shfl_sync(0xffffffffu, b, leader);
        rank[r] = b + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();
    {
        u32 run = d.table[(size_t)threadIdx.x * tiles + blockIdx.x];
#pragma unroll
        for (int w = 0; w < FR_WARPS; w++) {
            const u32 t = wh[w][threadIdx.x];
            wh[w][threadIdx.x] = run;
            run += t;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < FR_ITEMS; r++) {
        const size_t i = wbase + (size_t)r * 32 + lane;
        if (i < ne) {
            const u32 pos = wh[warp][(key[r] >> shift) & 255u] + rank[r];
            keys_out[pos] = key[r];
            vals_out[pos] = vals_in[i];
        }
    }
}

// ------------------------------------------------------------------------------------------------ sum + epilogue
// One thread per run of equal targets: the run added in storage order (= the reference's order), then what k_finish_ws
// does for the row.  Rows outside the runs keep y = 0 and x_next = 0 from earlier iterations (active sets only grow).
template <typename T>
__global__ void __launch_bounds__(FR_THREADS) k_fr_sum(const FrDev d, const u32* __restrict__ key, const T* __restrict__ prod,
                                                      const IterParams<T> p, int emit) {
    __shared__ double scratch[2 * FR_WARPS];
    __shared__ int is_last;
    IterCtl* ctl = p.ctl;
    if (fr_off(d)) return;
    const u32 ne = d.sc[1];
    const double S = ctl->S;
    const int seed = ctl->seed;
    double accS = 0.0, unused = 0.0;
    for (u32 i = blockIdx.x * FR_THREADS + threadIdx.x; i < ne; i += gridDim.x * FR_THREADS) {
        const u32 row = key[i];
        if (i > 0 && key[i - 1] == row) continue;
        double acc = 0.0;
        u32 j = i;
        do { acc = __dadd_rn(acc, (double)prod[j]); j++; } while (j < ne && key[j] == row);
        if (!RWR_CHK(row < (u32)p.n, ctl, 5)) continue;
        T y = (T)acc;
        if ((int)row == seed) y = (T)__dadd_rn((double)y, S);
        p.y[row] = y;
        const T invr = p.inv[row];
        const T rw = mul_rn(p.omc, y);
        p.x_next[row] = mul_rn(rw, invr);
        accS += (invr == (T)0) ? (double)y : (double)sub_rn(y, rw);
        if (emit && invr != (T)0) {
            const u32 o = (u32)d.old_of_new[row];
            atomicOr(&d.bits[o >> 5], 1u << (o & 31));
        }
    }
    block_sum2<FR_THREADS>(accS, unused, scratch);
    if (threadIdx.x == 0) {
        p.slot_S[blockIdx.x] = accS;
        __threadfence();
        const unsigned tk = atomicAdd(&ctl->ticket, 1u);
        is_last = (tk == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        double a = 0.0, b = 0.0;
        for (int i = threadIdx.x; i < (int)gridDim.x; i += FR_THREADS) a += __ldcg(p.slot_S + i);
        __syncthreads();
        block_sum2<FR_THREADS>(a, b, scratch);
        if (threadIdx.x == 0) {
            ctl->S = a;
            ctl->iters += 1;
            ctl->sparse_iters += 1;               // the dense kernels of this iteration return at once
            ctl->ticket = 0;
        }
    }
}

// ------------------------------------------------------------------------------------------------ build-time check
__global__ void k_fr_finite(const double* __restrict__ a, size_t n, int* bad) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && !isfinite(a[i])) *bad = 1;
}

void frontier_prepare(rwr_graph* g) {
    g->fr_finite = false;
    if (dist_n_ranks(g->comm) > 1 || !g->n) return;
    cudaStream_t st = g->stream;
    DevBuf<int> bad;
    bad.alloc(1);
    CUDA_CHECK(cudaMemsetAsync(bad.p, 0, sizeof(int), st));
    k_fr_finite<<<div_up((size_t)g->n, 256), 256, 0, st>>>(g->inv64.p, (size_t)g->n, bad.p);
    if (g->nnz && g->val.p) k_fr_finite<<<div_up((size_t)g->nnz, 256), 256, 0, st>>>(g->val.p, (size_t)g->nnz, bad.p);
    KERNEL_CHECK();
    int h = 1;
    CUDA_CHECK(cudaMemcpyAsync(&h, bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    g->fr_finite = h == 0;
}

// ------------------------------------------------------------------------------------------------ host side
u64 frontier_budget(const rwr_graph* g) {
    if (!g->fr_finite || dist_n_ranks(g->comm) > 1 || g->x_blocks > 1 || g->n < 1 || g->nnz < 1) return 0;
    const char* off = getenv("RWR_NO_FRONTIER");
    if (off && atoi(off) != 0) return 0;
    u64 b = 0;
    if (const char* e = getenv("RWR_FRONTIER_BUDGET")) b = strtoull(e, nullptr, 10);   // probe knob: links per sparse iteration
    else if (g->nnz >= FR_MIN_LINKS) b = (u64)g->nnz / 64;
    return std::min<u64>(b, (u64)INT32_MAX - 4);
}

static size_t fr_align(size_t b) { return (b + 255) & ~(size_t)255; }

size_t frontier_carve(const rwr_graph* g, u64 budget, size_t elt, void* base, FrontierWs& fw) {
    fw = FrontierWs{};
    if (!budget) return 0;
    fw.budget = budget;
    fw.cap = (size_t)budget + 1;
    fw.words = (u32)(((size_t)g->n + 31) / 32);
    fw.g_words = (int)div_up(fw.words, FR_TILE);
    fw.g_scan_f = (int)div_up((size_t)budget + 1, FR_TILE);
    fw.t_max = (int)div_up(fw.cap, FR_TILE);
    fw.g_scan_t = (int)div_up((size_t)fw.t_max * 256, FR_TILE);
    fw.g_exp = (int)std::min<size_t>(div_up(fw.cap, FR_THREADS), (size_t)g->sm_count * 8);
    fw.g_sum = (int)std::min<size_t>(div_up(fw.cap, FR_THREADS), (size_t)g->sm_count * 8);   // <= the slots of the workspace
    fw.passes = (ceil_log2_u64((u64)g->n) + 7) / 8;
    const size_t nb = (size_t)std::max(fw.g_words, std::max(fw.g_scan_f, fw.g_scan_t)) + 1;
    unsigned char* q = (unsigned char*)base;
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* r = q ? q + off : nullptr; off += fr_align(bytes); return r; };
    fw.sc = (u32*)take(4 * sizeof(u32));
    fw.bits = (u32*)take((size_t)fw.words * sizeof(u32));
    fw.fid = (u32*)take(((size_t)budget + 2) * sizeof(u32));
    fw.fdeg = (u32*)take(((size_t)budget + 2) * sizeof(u32));
    fw.foff = (u32*)take(((size_t)budget + 2) * sizeof(u32));
    fw.bsum = (u32*)take(nb * sizeof(u32));
    fw.table = (u32*)take((size_t)fw.t_max * 256 * sizeof(u32) + sizeof(u32));
    for (int k = 0; k < 2; k++) {
        fw.key[k] = (u32*)take(fw.cap * sizeof(u32));
        fw.val[k] = take(fw.cap * elt);
    }
    return off;
}

template <typename T>
int frontier_launch(rwr_graph* g, const FrontierWs& fw, const IterParams<T>& p, bool emit) {
    cudaStream_t st = g->stream;
    FrDev d{};
    d.ctl = p.ctl; d.sc = fw.sc;
    d.row_ptr = g->row_ptr; d.col = g->col; d.val = g->layout == RWR_LAYOUT_VALUED ? g->val.p : nullptr;
    d.new_of_old = g->new_of_old.p; d.old_of_new = g->old_of_new.p;
    d.n = g->n; d.words = fw.words; d.nnz = (u64)g->nnz; d.budget = fw.budget;
    d.bits = fw.bits; d.fid = fw.fid; d.fdeg = fw.fdeg; d.foff = fw.foff; d.bsum = fw.bsum; d.table = fw.table;
    int launches = 0;
    k_fr_count<<<fw.g_words, FR_THREADS, 0, st>>>(d);
    k_fr_extract<<<fw.g_words, FR_THREADS, 0, st>>>(d);
    k_fr_scan_a<<<fw.g_scan_f, FR_THREADS, 0, st>>>(d, fw.fdeg, fw.sc);
    k_fr_scan_b<<<fw.g_scan_f, FR_THREADS, 0, st>>>(d, fw.fdeg, fw.foff, fw.sc);
    k_fr_expand<T><<<fw.g_exp, FR_THREADS, 0, st>>>(d, p.x, fw.key[0], (T*)fw.val[0]);
    launches += 5;
    int cur = 0;
    for (int pass = 0; pass < fw.passes; pass++) {
        k_fr_hist<<<fw.t_max, FR_THREADS, 0, st>>>(d, fw.key[cur], pass * 8);
        k_fr_scan_a<<<fw.g_scan_t, FR_THREADS, 0, st>>>(d, fw.table, fw.sc + 2);
        k_fr_scan_b<<<fw.g_scan_t, FR_THREADS, 0, st>>>(d, fw.table, fw.table, fw.sc + 2);
        k_fr_scatter<T><<<fw.t_max, FR_THREADS, 0, st>>>(d, fw.key[cur], fw.key[cur ^ 1], (const T*)fw.val[cur], (T*)fw.val[cur ^ 1],
                                                          pass * 8);
        cur ^= 1;
        launches += 4;
    }
    k_fr_sum<T><<<fw.g_sum, FR_THREADS, 0, st>>>(d, fw.key[cur], (const T*)fw.val[cur], p, emit ? 1 : 0);
    launches += 1;
    KERNEL_CHECK();
    g->pool.launches += launches;
    return launches;
}
template int frontier_launch<double>(rwr_graph*, const FrontierWs&, const IterParams<double>&, bool);
template int frontier_launch<float>(rwr_graph*, const FrontierWs&, const IterParams<float>&, bool);
