// iterate_dev.cuh -- device-side pieces shared by iterate.cu, stream.cu and frontier.cu: the launch parameters of an
// iteration, PTX helpers (mbarrier, TMA bulk copy, cache-hinted loads) and the fixed-order block and grid reductions.
#pragma once

#include "iterate.h"

constexpr int FIX_THREADS = 256;

template <typename T>
struct IterParams {
    int n;
    const int32_t* ws_src;  // edge stream (stream.cu): source | end-of-row flag in bit 31
    const T* ws_val;        // valued layout only
    const u32* ws_tile;     // [ws_tiles + 1] first row of a tile | continued-row flag in bit 31
    int ws_tiles;
    int tile_links;         // links per tile
    int row_begin, row_end; // rows of W^T this rank owns ([0, n) unless the graph is row-partitioned)
    int parted;             // row-partitioned: the epilogue leaves its partial sums in ctl->red for the allReduce
    int n_peers;            // peers whose copy of x_next the epilogue writes directly (NVLink peer stores)
    void* peer_next[7];
    const T* x;             // gather source, internal labels (k_spmv_ws of a partitioned graph: shifted down by `hub` entries,
                            // the stream stores non-hub sources as label + hub)
    const T* xhub;          // k_spmv_ws: the unshifted gather vector the hub table is loaded from
    int hub_segs;           // > 0: partitioned graph, the hub table is hub_segs segments of hub_seg_len entries, segment s
    int hub_seg_len;        //      starting at label hub_start[s] (the hottest labels of every rank's slice)
    int hub_start[8];
    const T* inv;
    const T* r_prev;        // previous rank (residual)
    T* y;
    T* x_next;
    T omc;                  // (1 - c)
    int seed;               // internal label, -1: uniform restart
    double inv_n;           // 1/N (uniform restart)
    int hub;                // x entries staged in shared memory
    int n_hot;              // labels below: hot, L2-resident (evict-last); above: clustered cold nodes (streamed)
    int debug;              // measurement-only ablations (RWR_DEBUG_MODE, profile hook only)
    int iter;               // iteration of the run this launch computes (0-based): skipped when the frontier kernels did it
    double* head_partial;   // [ws_tiles] sum of the first row of a tile when that row started in an earlier tile
    double* carry;          // [ws_tiles] sum of the open row at the end of a tile (row sums are double in both precisions)
    double* slot_S;         // [blocks of k_finish_ws] restart-mass partials
    double* slot_R;
    IterCtl* ctl;
    // column blocking of x (experimental): k_spmv_ws / k_cutrows_ws write the sums of the virtual rows b * v_rows + (row -
    // row_begin) to yv (passed to them as `y`), k_finish_ws adds the x_blocks partial sums of a row in block order
    T* yv;
    int x_blocks;
    int v_rows;
    // compact slice-aligned blocks (partitioned graph, overlapped exchange): only the non-empty (row, block) pairs are
    // virtual rows; k_finish_ws adds the virtual rows vpair[vrow_ptr[i] .. vrow_ptr[i + 1]) of row i in block order
    int compact;
    const u32* vrow_ptr;    // [v_rows + 1]
    const u32* vpair;       // [v_compact]
    // arrival tags of the peers' slices: k_spmv_ws must not gather from stream block k before arrive[blk_src[k]] >= wait_tag
    const unsigned long long* arrive;   // [n_ranks], written by the peers' copy engines; null: nothing to wait for
    unsigned long long wait_tag;
    int blk_first_tile[8];  // tile holding the first link of stream block k (k = 0: this rank's own rows, never waited for)
    int blk_src[8];         // rank whose slice stream block k gathers from
    // the push warp of k_spmv_ws (overlapped exchange): while the other warps gather, it sends this rank's slice of the
    // vector being gathered from (produced by the previous epilogue) to every peer, peer rank+1 first, then the tag wait_tag
    const unsigned char* push_src;      // null: nothing to push (first iteration of a run)
    unsigned char* push_dst[7];
    unsigned long long* push_flag[7];   // arrive[rank] on those peers
    int push_peers;
    int push_tail;                      // 4-byte words after the 16-byte units
    size_t push_bytes16;
    unsigned* push_done;                // [7] CTAs that have finished a peer
    long long push_delay;               // test knob: cycles the push warp sleeps first (late slices)
    // checked build (-DRWR_CHECKED, librwr_b200_checked.so): bounds of the gather index and of the row-sum store
    int chk_src_end;        // stream sources are < this (n + hub + 8)
    int chk_y_begin, chk_y_end;   // k_spmv_ws / k_cutrows_ws store row sums at [begin, end)
    int chk_pairs;          // compact blocks: vpair entries are < this
};

// The restart vector q of a restart-set run (rwr_run_fixed_restart / rwr_run_threshold_restart), in internal labels: bit i
// of `bits` is set for the m rows with a listed weight; word_base[w] counts the members in the words before w, so the weight
// of member i is q[word_base[i >> 5] + popc(bits[i >> 5] below bit i)] -- q holds the weights in label order.
struct RestartSet {
    const u32* bits;        // [words]
    const u32* word_base;   // [words]
    const double* q;        // [m]
    int m;
    int words;
};

// Checked build: an index outside its array leaves a code in IterCtl.fault (2 gather source, 3 row-sum store, 4 virtual row
// of the epilogue, 5 restart-set bitmap word, 6 restart-set weight) and the access is skipped; the run then fails with
// RWR_E_INVALID instead of corrupting memory.
#ifdef RWR_CHECKED
#define RWR_CHK(cond, ctl, code) ((cond) ? true : ((ctl)->fault = (code), false))
#else
#define RWR_CHK(cond, ctl, code) true
#endif

// ------------------------------------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64* bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

__device__ __forceinline__ void load4_stream(const double* p, u64 pol, double out[4]) {
    out[0] = ld_stream(p, pol); out[1] = ld_stream(p + 1, pol); out[2] = ld_stream(p + 2, pol); out[3] = ld_stream(p + 3, pol);
}
__device__ __forceinline__ void load4_stream(const float* p, u64 pol, float out[4]) {
    out[0] = ld_stream(p, pol); out[1] = ld_stream(p + 1, pol); out[2] = ld_stream(p + 2, pol); out[3] = ld_stream(p + 3, pol);
}

// fixed-order block reduction of two doubles; result valid in thread 0
template <int THREADS>
__device__ __forceinline__ void block_sum2(double& a, double& b, double* scratch /* 2 * THREADS/32 */) {
    a = warp_sum(a);
    b = warp_sum(b);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { scratch[warp] = a; scratch[THREADS / 32 + warp] = b; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sa = 0, sb = 0;
        for (int w = 0; w < THREADS / 32; w++) { sa += scratch[w]; sb += scratch[THREADS / 32 + w]; }
        a = sa; b = sb;
    }
}

// Fixed-order reduction over the blocks of a grid: every block reduces its partials a (and, with TWO, b), stores them in
// slot_a[blockIdx.x] (slot_b) and takes a ticket on ctl->ticket.  Returns true in the last block to arrive, where thread 0
// then holds the sums of all slots, added in block order, in a (and b); that block's caller resets ctl->ticket.
template <int THREADS, bool TWO>
__device__ __forceinline__ bool grid_sum2(double& a, double& b, double* slot_a, double* slot_b, IterCtl* ctl,
                                          double* scratch /* 2 * THREADS/32 */, int* is_last /* shared */) {
    block_sum2<THREADS>(a, b, scratch);
    if (threadIdx.x == 0) {
        slot_a[blockIdx.x] = a;
        if (TWO) slot_b[blockIdx.x] = b;
        __threadfence();
        const unsigned tk = atomicAdd(&ctl->ticket, 1u);
        *is_last = (tk == gridDim.x - 1);
    }
    __syncthreads();
    if (!*is_last) return false;
    __threadfence();
    a = 0.0;
    b = 0.0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += THREADS) {
        a += __ldcg(slot_a + i);
        if (TWO) b += __ldcg(slot_b + i);
    }
    __syncthreads();
    block_sum2<THREADS>(a, b, scratch);
    return true;
}

// ------------------------------------------------------------------------------------------------ shared-space PTX
__device__ __forceinline__ void mbar_wait_a(u32 bar, u32 parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE;\n"
        "bra LAB_WAIT;\n"
        "LAB_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
