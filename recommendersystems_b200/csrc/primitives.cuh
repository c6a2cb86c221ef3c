// primitives.cuh -- device-wide exclusive scan (K2) and stable LSD radix sort used by the graph build (K3, K5),
// the synthetic generator (K0), the full ranking (A9) and, through their tile bodies, the sparse prefix of a single-seed run
// (frontier.cu, counts on the device).  Hand-written; no CUB/Thrust.
#pragma once

#include "common.cuh"

namespace prim {

// ======================================================================================= exclusive scan (u32)
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;                        // per thread, blocked
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS; // 2048

__device__ __forceinline__ u32 block_exclusive_scan_256(u32 v, u32* total, u32* smem /*>=9*/) {
    // exclusive scan of one value per thread over a 256-thread block
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) smem[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        u32 w = (lane < 8) ? smem[lane] : 0;
        u32 winc = w;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            u32 t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < 8) smem[lane] = winc - w;
        if (lane == 7) smem[8] = winc;
    }
    __syncthreads();
    u32 res = smem[warp] + inc - v;
    *total = smem[8];
    __syncthreads();
    return res;
}

// The tile bodies below serve the host-sized kernels here and the device-sized ones of the sparse prefix (frontier.cu):
// block b works on tile b of the n items, and the shared arrays belong to the calling kernel.

// sum of the block's tile of in[0, n), in every thread
template <typename InT>
__device__ __forceinline__ u32 scan_tile_total(const InT* __restrict__ in, size_t n, u32* sm /*>=9*/) {
    size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++)
        if (base + k < n) s += (u32)in[base + k];
    u32 total;
    block_exclusive_scan_256(s, &total, sm);
    return total;
}

// exclusive scan of the block's tile of in[0, n) into out, every entry plus the tile's offset off(); returns the tile's sum.
// off() is called after the block scan: k_scan_tile_apply loads the offset there, k_fr_scan_b has computed it before.
template <typename InT, typename Off>
__device__ __forceinline__ u32 scan_tile_apply(const InT* __restrict__ in, u32* __restrict__ out, size_t n, Off off,
                                               u32* sm /*>=9*/) {
    size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_ITEMS;
    u32 v[SCAN_ITEMS];
    u32 s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        v[k] = (base + k < n) ? (u32)in[base + k] : 0;
        s += v[k];
    }
    u32 total;
    u32 ex = block_exclusive_scan_256(s, &total, sm) + off();
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; k++) {
        if (base + k < n) out[base + k] = ex;
        ex += v[k];
    }
    return total;
}

template <typename InT>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_sums(const InT* __restrict__ in, u32* __restrict__ sums, size_t n) {
    __shared__ u32 sm[9];
    u32 total = scan_tile_total<InT>(in, n, sm);
    if (threadIdx.x == 0) sums[blockIdx.x] = total;
}

template <typename InT>
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_apply(const InT* __restrict__ in, u32* __restrict__ out,
                                                                 const u32* __restrict__ tile_off, size_t n) {
    __shared__ u32 sm[9];
    scan_tile_apply<InT>(in, out, n, [&] { return tile_off ? tile_off[blockIdx.x] : 0u; }, sm);
}

// out[i] = sum(in[0..i)), out may alias in when InT is u32; optional total (device pointer) = sum of all, and with
// total_host (which needs total_dev) a copy of it on the host, enqueued before the final synchronisation.
// Temp memory is allocated internally (tile sums, a few hundred KB at most).
template <typename InT>
inline void exclusive_scan(const InT* in, u32* out, size_t n, u32* total_dev, cudaStream_t st, DevPool* pool,
                           u32* total_host = nullptr) {
    if (n == 0) {
        if (total_dev) CUDA_CHECK(cudaMemsetAsync(total_dev, 0, sizeof(u32), st));
        if (total_host) {
            *total_host = 0;
            CUDA_CHECK(cudaStreamSynchronize(st));
        }
        return;
    }
    size_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    DevBuf<u32> sums;
    sums.alloc(tiles + 1);
    k_scan_tile_sums<InT><<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, sums.p, n);
    KERNEL_CHECK();
    if (pool) pool->launches++;
    // scan the tile sums (recursively); sums[tiles] receives the grand total
    if (tiles == 1) {
        if (total_dev) CUDA_CHECK(cudaMemcpyAsync(total_dev, sums.p, sizeof(u32), cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemsetAsync(sums.p, 0, sizeof(u32), st));
    } else {
        exclusive_scan<u32>(sums.p, sums.p, tiles, total_dev ? total_dev : (sums.p + tiles), st, pool);
    }
    k_scan_tile_apply<InT><<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, out, sums.p, n);
    KERNEL_CHECK();
    if (pool) pool->launches++;
    if (total_host) CUDA_CHECK(cudaMemcpyAsync(total_host, total_dev, sizeof(u32), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));   // `sums` is freed on return
}

// The scan for a caller that needs the total on the host: returns it, after the stream has synchronised.  With `csr`,
// out holds n + 1 words and out[n] receives the total as well (CSR offsets).
template <typename InT>
inline u32 scan_total(const InT* in, u32* out, size_t n, bool csr, cudaStream_t st, DevPool* pool) {
    DevBuf<u32> word;
    if (!csr) word.alloc(1);
    u32 total = 0;
    exclusive_scan<InT>(in, out, n, csr ? out + n : word.p, st, pool, &total);
    return total;
}

// ======================================================================================= LSD radix sort
constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 8;
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;   // 2048 keys per CTA
constexpr int RS_WARPS = RS_THREADS / 32;

// digit histogram of the block's tile of keys[0, n) into its column of the digit-major table of `tiles` tiles
template <typename KeyT>
__device__ __forceinline__ void rs_hist_tile(const KeyT* __restrict__ keys, u32* __restrict__ table, size_t n, int shift, u32 tiles,
                                             u32* h /*256*/) {
    h[threadIdx.x] = 0;
    __syncthreads();
    size_t base = (size_t)blockIdx.x * RS_TILE;
#pragma unroll
    for (int k = 0; k < RS_ITEMS; k++) {
        size_t i = base + (size_t)k * RS_THREADS + threadIdx.x;
        if (i < n) atomicAdd(&h[(u32)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    table[(size_t)threadIdx.x * tiles + blockIdx.x] = h[threadIdx.x];   // digit-major
}

// Stable scatter of the block's tile, with the table scanned.  Element order inside a tile is (warp, round, lane): warp w owns
// the contiguous sub-tile [w*32*ITEMS, (w+1)*32*ITEMS), read in rounds of 32 consecutive keys, so ranking by (warp, round,
// lane) preserves the input order.  `tid` is the kernel's threadIdx.x: read in the kernel, it carries the range of the
// launch bounds, which lets the compiler form the warp's first key as tile base | warp offset.
template <typename KeyT, typename ValT, bool HAS_VAL>
__device__ __forceinline__ void rs_scatter_tile(const KeyT* __restrict__ keys_in, KeyT* __restrict__ keys_out,
                                                const ValT* __restrict__ vals_in, ValT* __restrict__ vals_out,
                                                const u32* __restrict__ table, size_t n, int shift, u32 tiles,
                                                u32 (*wh)[256] /*[RS_WARPS]*/, const u32 tid) {
    const int lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < RS_WARPS * 256; i += RS_THREADS) (&wh[0][0])[i] = 0;
    __syncthreads();
    const size_t wbase = (size_t)blockIdx.x * RS_TILE + (size_t)warp * (32 * RS_ITEMS);
    KeyT key[RS_ITEMS];
    u32 rank[RS_ITEMS];
    const u32 lt = (1u << lane) - 1u;
#pragma unroll
    for (int r = 0; r < RS_ITEMS; r++) {
        size_t i = wbase + (size_t)r * 32 + lane;
        bool valid = i < n;
        key[r] = valid ? keys_in[i] : (KeyT)0;
        u32 d = valid ? ((u32)(key[r] >> shift) & 255u) : 256u;   // 256: sentinel shared by the invalid lanes
        u32 peers = __match_any_sync(0xffffffffu, d);
        int leader = __ffs(peers) - 1;
        u32 base = 0;
        if (valid && lane == leader) {
            base = wh[warp][d];
            wh[warp][d] = base + __popc(peers);
        }
        base = __shfl_sync(0xffffffffu, base, leader);
        rank[r] = base + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();
    {   // digit d = tid: exclusive prefix over the warps, seeded with the global offset of (d, tile)
        u32 run = table[(size_t)tid * tiles + blockIdx.x];
#pragma unroll
        for (int w = 0; w < RS_WARPS; w++) {
            u32 t = wh[w][tid];
            wh[w][tid] = run;
            run += t;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < RS_ITEMS; r++) {
        size_t i = wbase + (size_t)r * 32 + lane;
        if (i < n) {
            u32 d = (u32)(key[r] >> shift) & 255u;
            u32 pos = wh[warp][d] + rank[r];
            keys_out[pos] = key[r];
            if (HAS_VAL) vals_out[pos] = vals_in[i];
        }
    }
}

template <typename KeyT>
__global__ void __launch_bounds__(RS_THREADS) k_rs_hist(const KeyT* __restrict__ keys, u32* __restrict__ table, size_t n,
                                                        int shift, u32 tiles) {
    __shared__ u32 h[256];
    rs_hist_tile<KeyT>(keys, table, n, shift, tiles, h);
}

template <typename KeyT, bool HAS_VAL>
__global__ void __launch_bounds__(RS_THREADS) k_rs_scatter(const KeyT* __restrict__ keys_in, KeyT* __restrict__ keys_out,
                                                           const u32* __restrict__ vals_in, u32* __restrict__ vals_out,
                                                           const u32* __restrict__ table, size_t n, int shift, u32 tiles) {
    __shared__ u32 wh[RS_WARPS][256];
    rs_scatter_tile<KeyT, u32, HAS_VAL>(keys_in, keys_out, vals_in, vals_out, table, n, shift, tiles, wh, threadIdx.x);
}

// The buffers of a stable radix sort: two for the keys and, for a sort that carries u32 values, two for the values.
// sort() ping-pongs between each pair; keys() and vals() are the current buffers, which hold the result after a sort.
template <typename KeyT>
struct SortBuffers {
    DevBuf<KeyT> k[2];
    DevBuf<u32> v[2];
    int kc = 0, vc = 0;   // current key / value buffer

    void alloc(size_t n, bool with_vals) {
        k[0].alloc(n); k[1].alloc(n);
        if (with_vals) { v[0].alloc(n); v[1].alloc(n); }
    }
    KeyT* keys() const { return k[kc].p; }
    u32* vals() const { return v[vc].p; }
    // The spare key buffer becomes the current one, for the caller to fill with new keys: the next sort is a stable pass
    // over them that keeps the current order of the values.
    KeyT* rekey() { kc ^= 1; return keys(); }
    void release_spare() { k[kc ^ 1].release(); v[vc ^ 1].release(); }
    void release() { release_spare(); k[kc].release(); v[vc].release(); }
    DevBuf<u32> take_vals() { return std::move(v[vc]); }

    // Sorts the first `n` (< 2^32) current keys ascending on bits [0, end_bit), stable, with their values.
    void sort(size_t n, int end_bit, cudaStream_t st, DevPool* pool) {
        if (n == 0 || end_bit <= 0) return;
        if (n >= (1ULL << 32)) RWR_FAIL(RWR_E_UNSUPPORTED, "radix_sort: more than 2^32-1 elements");
        u32 tiles = (u32)((n + RS_TILE - 1) / RS_TILE);
        DevBuf<u32> table;
        table.alloc((size_t)tiles * 256);
        for (int shift = 0; shift < end_bit; shift += 8) {
            KeyT* ki = k[kc].p;
            KeyT* ko = k[kc ^ 1].p;
            k_rs_hist<KeyT><<<tiles, RS_THREADS, 0, st>>>(ki, table.p, n, shift, tiles);
            KERNEL_CHECK();
            exclusive_scan<u32>(table.p, table.p, (size_t)tiles * 256, nullptr, st, pool);
            if (v[vc].p)
                k_rs_scatter<KeyT, true><<<tiles, RS_THREADS, 0, st>>>(ki, ko, v[vc].p, v[vc ^ 1].p, table.p, n, shift, tiles);
            else
                k_rs_scatter<KeyT, false><<<tiles, RS_THREADS, 0, st>>>(ki, ko, nullptr, nullptr, table.p, n, shift, tiles);
            KERNEL_CHECK();
            if (pool) pool->launches += 2;
            kc ^= 1;
            vc ^= 1;
        }
        CUDA_CHECK(cudaStreamSynchronize(st));
    }
};

}  // namespace prim
