// iterate.cu -- the power iteration r <- (1-c) W^T r + S q  (K6, K7) with its convergence test.
//
// Restates Recommenders/RWRBased/Model.cs:
//   :33-50   seeded constructor  (rank[seed] = N, restart = e_seed)        -> k_init
//   :14-31   uniform constructor (rank = 1, restart = 1/N)                  -> k_init (seed == -1)
//   :76-100  deliverRanks  push loop, as a pull over CSR(W^T)               -> stream.cu (k_spmv_ws, k_cutrows_ws, k_finish_ws)
//   :103-108 updateRanks   rank <- next, next <- 0                          -> buffer swap (nothing to zero)
//   :110-115 checkConvergence  sum |rank - next|                            -> fused into the epilogue
//   :52-73   run() / run(double) / run(int)                                 -> rwr_run_threshold / rwr_run_fixed
//   :9       `restart` overwritten by the caller (a weighted node set)      -> rwr_run_fixed_restart / rwr_run_threshold_restart
//                                                                              (k_init_set, k_finish_set_ws)
//
// The iteration kernels live in stream.cu (K7: k_spmv_ws, k_cutrows_ws, k_finish_ws); this file holds the run modes,
// K6 (k_init), the workspaces and the result handle.
#include <algorithm>
#include <cmath>

#include "iterate.h"

#include "iterate_dev.cuh"
#include "primitives.cuh"
#include "stream.h"
#include "frontier.h"
#include "dist.h"


// ------------------------------------------------------------------------------------------------ K6: init
// fr_bits (a run that may go sparse, frontier.cu): the frontier bitmap over the original labels gets the seed (when it
// has out-links) and nothing else, and x1 -- the first x_next, which the frontier kernels write only at the active rows --
// is zeroed.
template <typename T>
__global__ void k_init(int n, int seed, T omc, const T* __restrict__ inv, T* __restrict__ r0, T* __restrict__ x0,
                       T* __restrict__ x1, IterCtl* ctl, double S_uniform, u32* __restrict__ fr_bits, u32 fr_words, int seed_orig) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < 8) { x0[n + j] = (T)0; x1[n + j] = (T)0; }     // x[n] is the always-zero entry the edge stream pads with
    if (j == 0) {
        ctl->resid = 0.0; ctl->done = 0; ctl->iters = 0; ctl->ticket = 0; ctl->fault = 0; ctl->wait_clk = 0;
        ctl->tile_ctr = 0;
        ctl->seed = seed;
        ctl->sparse = fr_bits != nullptr;
        ctl->sparse_iters = 0;
        if (seed < 0) ctl->S = S_uniform;
    }
    if (fr_bits && (u32)j < fr_words)
        fr_bits[j] = ((seed_orig >> 5) == j && inv[seed] != (T)0) ? 1u << (seed_orig & 31) : 0u;
    if (j >= n) return;
    if (fr_bits) x1[j] = (T)0;
    const T r = (seed < 0) ? (T)1 : ((j == seed) ? (T)n : (T)0);           // Model.cs:24 / :44
    const T invj = inv[j];
    const T rw = mul_rn(omc, r);
    r0[j] = r;
    x0[j] = mul_rn(rw, invj);
    if (j == seed) ctl->S = (invj == (T)0) ? (double)r : (double)sub_rn(r, rw);
}

// ---- restart sets: q over a node list, in internal labels (RestartSet, iterate_dev.cuh)
// the bitmap of the listed nodes; lbl[k] = internal label of nodes[k]
__global__ void k_restart_mark(const int32_t* __restrict__ nodes, int m, const int32_t* __restrict__ new_of_old,
                               int32_t* __restrict__ lbl, u32* __restrict__ bits) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const int j = new_of_old[nodes[k]];
    lbl[k] = j;
    atomicOr(&bits[j >> 5], 1u << (j & 31));
}
__global__ void k_restart_popc(const u32* __restrict__ bits, int words, u32* __restrict__ cnt) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w < words) cnt[w] = (u32)__popc(bits[w]);
}
// q in label order: member j is number word_base[j >> 5] + popc(bits below j) (the nodes are distinct)
__global__ void k_restart_place(const int32_t* __restrict__ lbl, const double* __restrict__ weights, int m, const RestartSet rs,
                                double* __restrict__ q) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const int j = lbl[k];
    q[rs.word_base[j >> 5] + __popc(rs.bits[j >> 5] & ((1u << (j & 31)) - 1u))] = weights[k];
}

// K6 of a restart-set run: the initial rank of `init` (RWR_INIT_UNIFORM: 1 everywhere, Model.cs:24; RWR_INIT_NODE: N at the
// internal label `node`, Model.cs:44; RWR_INIT_RESTART: fl(N q_i)) and x0.  S0 is set here for UNIFORM (S_uniform) and NODE;
// k_restart_s0 sums it for RESTART.  No frontier: a restart-set run is dense from its first iteration.
template <typename T>
__global__ void k_init_set(int n, int init, int node, T omc, const T* __restrict__ inv, T* __restrict__ r0, T* __restrict__ x0,
                           T* __restrict__ x1, IterCtl* ctl, double S_uniform, const RestartSet rs) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < 8) { x0[n + j] = (T)0; x1[n + j] = (T)0; }
    if (j == 0) {
        ctl->resid = 0.0; ctl->done = 0; ctl->iters = 0; ctl->ticket = 0; ctl->fault = 0; ctl->wait_clk = 0;
        ctl->tile_ctr = 0;
        ctl->seed = -1;
        ctl->sparse = 0;
        ctl->sparse_iters = 0;
        if (init == RWR_INIT_UNIFORM) ctl->S = S_uniform;
    }
    if (j >= n) return;
    T r = (T)0;
    if (init == RWR_INIT_UNIFORM) {
        r = (T)1;
    } else if (init == RWR_INIT_NODE) {
        r = (j == node) ? (T)n : (T)0;
    } else {
        const u32 word = rs.bits[j >> 5];
        if ((word >> (j & 31)) & 1u)
            r = (T)__dmul_rn((double)n, rs.q[rs.word_base[j >> 5] + __popc(word & ((1u << (j & 31)) - 1u))]);
    }
    const T invj = inv[j];
    const T rw = mul_rn(omc, r);
    r0[j] = r;
    x0[j] = mul_rn(rw, invj);
    if (init == RWR_INIT_NODE && j == node) ctl->S = (invj == (T)0) ? (double)r : (double)sub_rn(r, rw);
}

// S0 of RWR_INIT_RESTART: the restart mass of the listed nodes, in one block and a fixed order (reruns are bit-identical)
template <typename T>
__global__ void __launch_bounds__(FIN_THREADS) k_restart_s0(int n, T omc, const T* __restrict__ inv, const int32_t* __restrict__ lbl,
                                                            const double* __restrict__ weights, int m, IterCtl* ctl) {
    __shared__ double scratch[2 * FIN_THREADS / 32];
    double a = 0.0, b = 0.0;
    for (int k = threadIdx.x; k < m; k += FIN_THREADS) {
        const T r = (T)__dmul_rn((double)n, weights[k]);
        const T rw = mul_rn(omc, r);
        a += (inv[lbl[k]] == (T)0) ? (double)r : (double)sub_rn(r, rw);
    }
    block_sum2<FIN_THREADS>(a, b, scratch);
    if (threadIdx.x == 0) ctl->S = a;
}

// ---- continuing from the rank a result holds (rwr_continue_*, rwr_set_rank)
// K6 of a continuation: x0 = fl(fl((1-c) r) inv) from the held rank r (internal labels) and the zero pad; ctl is reset as
// k_init_set resets it, with S the restart mass kept after the slot's last run (or computed by k_resume_s from a written
// rank).  Threshold mode (r_copy): r also goes to the buffer the residual of the first iteration reads.
template <typename T>
__global__ void k_init_resume(int n, int seed, T omc, const T* __restrict__ inv, const T* __restrict__ r, T* __restrict__ x0,
                              T* __restrict__ x1, T* __restrict__ r_copy, IterCtl* ctl, const double* __restrict__ S) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < 8) { x0[n + j] = (T)0; x1[n + j] = (T)0; }
    if (j == 0) {
        ctl->resid = 0.0; ctl->done = 0; ctl->iters = 0; ctl->ticket = 0; ctl->fault = 0; ctl->wait_clk = 0;
        ctl->tile_ctr = 0;
        ctl->seed = RWR_CHK(seed < n, ctl, 7) ? seed : -1;
        ctl->sparse = 0;
        ctl->sparse_iters = 0;
        ctl->S = *S;
    }
    if (j >= n) return;
    const T rj = r[j];
    x0[j] = mul_rn(mul_rn(omc, rj), inv[j]);
    if (r_copy) r_copy[j] = rj;
}

// S of a caller-written rank r: the restart mass the epilogue sums (k_finish_ws), over the same grid (ws_fin_grid blocks
// of FIN_THREADS), the same rows per thread and the same fixed-order reduction -- writing back the rank an epilogue
// produced gives that epilogue's S bit for bit.
template <typename T>
__global__ void __launch_bounds__(FIN_THREADS) k_resume_s(int n, T omc, const T* __restrict__ inv, const T* __restrict__ r,
                                                          double* __restrict__ slot, IterCtl* ctl, double* __restrict__ S_out) {
    __shared__ double scratch[2 * FIN_THREADS / 32];
    __shared__ int is_last;
    double accS = 0.0, unused = 0.0;
    for (int row = blockIdx.x * FIN_THREADS + threadIdx.x; row < n; row += gridDim.x * FIN_THREADS) {
        const T y = r[row];
        accS += (inv[row] == (T)0) ? (double)y : (double)sub_rn(y, mul_rn(omc, y));
    }
    if (grid_sum2<FIN_THREADS, false>(accS, unused, slot, nullptr, ctl, scratch, &is_last) && threadIdx.x == 0) {
        *S_out = accS;
        ctl->ticket = 0;
    }
}

// `model.rank = v`: v (original labels, double) into the result column r (internal labels), rounded to T
template <typename T>
__global__ void k_set_rank(int n, const double* __restrict__ v, const int32_t* __restrict__ new_of_old, T* __restrict__ r,
                           IterCtl* ctl) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = new_of_old[i];
    if (RWR_CHK((unsigned)j < (unsigned)n, ctl, 7)) r[j] = (T)v[i];
}

__global__ void k_partition(const u32* __restrict__ in_ptr, int n, u32 nnz, int n_chunks, int2* __restrict__ part) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > n_chunks) return;
    u64 d = (u64)k * CHUNK_ITEMS;
    const u64 total = (u64)n + nnz;
    if (d > total) d = total;
    u64 lo = d > nnz ? d - nnz : 0, hi = d < (u64)n ? d : (u64)n;
    while (lo < hi) {
        const u64 mid = (lo + hi) >> 1;
        if ((u64)in_ptr[mid + 1] <= d - mid - 1) lo = mid + 1; else hi = mid;
    }
    part[k] = make_int2((int)lo, (int)(d - lo));
}

__global__ void k_f64_to_f32(const double* __restrict__ in, float* __restrict__ out, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (float)in[i];
}

// row slice: after the allReduce of ctl->red, the sums over all ranks become S and the residual; threshold mode then
// applies the test of Model.cs:114.  A converged run ignores the (stale) sums of its no-op launches.
__global__ void k_after_reduce(IterCtl* ctl, double thr, int use_thr) {
    if (ctl->done) return;
    ctl->S = ctl->red[0];
    ctl->resid = ctl->red[1];
    if (use_thr && ctl->red[1] < thr) ctl->done = 1;
}

template <typename T>
__global__ void k_unpermute(const T* __restrict__ y_int, const int32_t* __restrict__ new_of_old, int n, double* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)y_int[new_of_old[i]];
}

// ------------------------------------------------------------------------------------------------ host side
void iterate_prepare(rwr_graph* g) {
    cudaStream_t st = g->stream;
    const u64 total = (u64)g->n + (u64)g->nnz_in;
    g->n_chunks = (int)std::max<u64>(1, (total + CHUNK_ITEMS - 1) / CHUNK_ITEMS);
    g->part.alloc((size_t)g->n_chunks + 1, &g->pool);
    k_partition<<<div_up((size_t)g->n_chunks + 1, 256), 256, 0, st>>>(g->in_ptr.p, g->n, (u32)g->nnz_in, g->n_chunks, g->part.p);
    KERNEL_CHECK();
    CUDA_CHECK(cudaStreamSynchronize(st));
    stream_prepare(g);
    frontier_prepare(g);
}

void ensure_fp32_arrays(rwr_graph* g) {
    cudaStream_t st = g->stream;
    if (!g->inv32.p) {
        g->inv32.alloc((size_t)g->n + 4, &g->pool);
        if (g->n) k_f64_to_f32<<<div_up(g->n, 256), 256, 0, st>>>(g->inv64.p, g->inv32.p, g->n);
        KERNEL_CHECK();
    }
    if (g->layout == RWR_LAYOUT_VALUED && !g->in_val32.p && g->in_val64.p) {     // (a row slice keeps no whole-graph pull arrays)
        g->in_val32.alloc((size_t)g->nnz_in + IDX_PAD, &g->pool);
        if (g->nnz_in) k_f64_to_f32<<<div_up((size_t)g->nnz_in, 256), 256, 0, st>>>(g->in_val64.p, g->in_val32.p, (size_t)g->nnz_in);
        KERNEL_CHECK();
    }
    if (g->layout == RWR_LAYOUT_VALUED && !g->ws_val32.p && g->ws_val64.n) {
        g->ws_val32.alloc(g->ws_val64.n, &g->pool);
        k_f64_to_f32<<<div_up(g->ws_val64.n, 256), 256, 0, st>>>(g->ws_val64.p, g->ws_val32.p, g->ws_val64.n);
        KERNEL_CHECK();
    }
}

template <typename T> struct Prec;
template <> struct Prec<double> {
    static const double* inv(rwr_graph* g) { return g->inv64.p; }
    static const double* val(rwr_graph* g) { return g->in_val64.p; }
    static const double* wsval(rwr_graph* g) { return g->ws_val64.p; }
    static DevBuf<double>& ybuf(rwr_result* r) { return r->y64; }
    static constexpr int id = RWR_FP64;
};
template <> struct Prec<float> {
    static const float* inv(rwr_graph* g) { return g->inv32.p; }
    static const float* val(rwr_graph* g) { return g->in_val32.p; }
    static const float* wsval(rwr_graph* g) { return g->ws_val32.p; }
    static DevBuf<float>& ybuf(rwr_result* r) { return r->y32; }
    static constexpr int id = RWR_FP32;
};

// One iteration: K7 on this handle's stream, plus the exchange of a row-partitioned graph.
template <typename T>
static void launch_iteration(rwr_graph* g, const IterParams<T>& p, bool resid, double thr, int use_thr, const RestartSet* rs) {
    cudaStream_t st = g->stream;
    const bool parted = dist_n_ranks(g->comm) > 1;
    // on a row slice the convergence test needs the residual of all slices: it runs after the exchange
    ws_launch_iteration<T>(g, p, resid, thr, parted ? 0 : use_thr, rs);
    static const bool skip_exchange = getenv("RWR_DIST_SKIP") != nullptr;      // timing probe only: wrong results
    if (parted && !skip_exchange) {
        // x_next: pushed by the next k_spmv_ws while it gathers (overlapped exchange), or already in every peer's copy when
        // the epilogue stored it there (p.n_peers > 0), else NCCL
        dist_exchange(g, (p.n_peers || g->overlap) ? nullptr : p.x_next, sizeof(T), p.ctl->red);
        k_after_reduce<<<1, 1, 0, st>>>(p.ctl, thr, use_thr);
        KERNEL_CHECK();
    }
}

// The scratch of one run of the iteration kernels.  Nothing in it needs initialising: k_init sets up ctl at the start of
// every run, and every other entry is written earlier in the same iteration than it is read.  k_spmv_ws stores carry[t]
// at the end of every tile t and head[t] at the first row end of a tile whose first row is continued; k_cutrows_ws reads
// carry[m..t) and head[t] only for such a tile t whose continued row ends inside it.  Every block of k_finish_ws stores
// its slot_S / slot_R entry before it takes its ticket, and only the block that takes the last ticket reads them.  (The
// probe ablation RWR_DEBUG_MODE=1 stores no row ends, so its k_cutrows_ws reads head unwritten: its sums mean nothing.)
// The frontier workspace (fr, fw) of a run that may go sparse follows from the push-link budget; the bitmap in it is
// set up by k_init, and the frontier kernels write every other entry before they read it.
struct RunWorkspace {
    Scratch<unsigned char> xa, xb, ya, yv, fr;
    Scratch<double> carry, head, slot_S, slot_R;
    Scratch<IterCtl> ctl;
    FrontierWs fw;
    void* x[2] = {nullptr, nullptr};      // the two gather vectors: scratch, or the peer-mapped buffers of a partitioned graph
    // ya: the second rank vector of threshold mode and the probe's y (a fixed-count run into y_out leaves it unused)
    // fr_budget: push links per sparse iteration (0: the run stays dense)
    template <typename T>
    void alloc(rwr_graph* g, size_t ya_bytes, u64 fr_budget = 0) {
        const size_t vec_bytes = ((size_t)g->n + 8) * sizeof(T);
        if (g->p2p) {
            x[0] = g->px[0]; x[1] = g->px[1];
        } else {
            xa.alloc(&g->scratch, vec_bytes); xb.alloc(&g->scratch, vec_bytes);
            x[0] = xa.p; x[1] = xb.p;
        }
        // column blocking of x (experimental): partial row sums of the virtual rows
        if (g->ws_compact) yv.alloc(&g->scratch, (size_t)g->v_compact * sizeof(T) + 16);
        else if (g->x_blocks > 1) yv.alloc(&g->scratch, (size_t)g->x_blocks * (size_t)g->v_rows * sizeof(T) + 16);
        ya.alloc(&g->scratch, ya_bytes);
        carry.alloc(&g->scratch, (size_t)g->ws_tiles + 1); head.alloc(&g->scratch, (size_t)g->ws_tiles + 1);
        const size_t slots = (size_t)g->sm_count * 8 + 8;
        slot_S.alloc(&g->scratch, slots); slot_R.alloc(&g->scratch, slots);
        ctl.alloc(&g->scratch, 1);
        if (fr_budget) fr.alloc(&g->scratch, frontier_carve(g, fr_budget, sizeof(T), nullptr, fw));
        frontier_carve(g, fr_budget, sizeof(T), fr.p, fw);
    }
};

// rows below this label are hot (their x entries are stored evict-last by the epilogue): the degree-sorted label prefix,
// or -- on a slice of a partitioned graph, whose labels are dealt over the slices -- the hot head of this rank's own rows
static int hot_limit(const rwr_graph* g) {
    const int parts = dist_n_ranks(g->comm);
    if (parts > 1 && (int)g->part_hot.size() == parts) return g->deal_rows[dist_rank(g->comm)] + g->part_hot[dist_rank(g->comm)];
    return g->n_hot;
}

// peers' copies of the buffer `x_next` is (row-partitioned graphs with peer-mapped gather vectors)
template <typename T>
static void set_peers(rwr_graph* g, IterParams<T>& p, const void* x_next) {
    p.parted = dist_n_ranks(g->comm) > 1;
    p.n_peers = 0;
    if (!g->p2p || g->overlap) return;          // overlapped exchange: the copy engines carry the slice, not the epilogue
    const int b = (x_next == g->px[0]) ? 0 : 1, me = dist_rank(g->comm);
    for (int r = 0; r < (int)g->peer_px[b].size(); r++)
        if (r != me) p.peer_next[p.n_peers++] = g->peer_px[b][r];
}

// Block layout of the stream and the tags of the overlapped exchange for the iteration that writes `x_next`.  `first`: the
// gather vector of this iteration comes from k_init (every rank computes all of it), nothing is in flight.
template <typename T>
static void set_exchange(rwr_graph* g, IterParams<T>& p, const void* x_next, bool first, bool live) {
    const int P = dist_n_ranks(g->comm), me = dist_rank(g->comm);
    p.compact = g->ws_compact ? 1 : 0;
    p.vrow_ptr = g->vrow_ptr.p; p.vpair = g->vpair.p;
    for (int k = 0; k < 8; k++) { p.blk_first_tile[k] = g->blk_first_tile[k]; p.blk_src[k] = ((me - k) % P + P) % P; }
    p.arrive = nullptr; p.wait_tag = 0;
    p.push_src = nullptr; p.push_peers = 0; p.push_tail = 0; p.push_bytes16 = 0; p.push_done = g->push_done; p.push_delay = 0;
    if (g->overlap && live) {
        // tag t marks the slices produced by the t-th iteration of this handle's life; all ranks count alike (collective calls)
        const uint64_t tag = ++g->xtag;
        if (!first) {
            // this launch gathers from the vector the previous iteration produced (tag - 1): it pushes this rank's slice of it
            // to the peers and waits for theirs
            DistSync* ds = (DistSync*)g->psync;
            p.arrive = ds->arrive;
            p.wait_tag = tag - 1;
            const int b = ((const void*)p.x == g->px[0]) ? 0 : 1;
            const size_t off = (size_t)g->row_begin * sizeof(T), len = (size_t)(g->row_end - g->row_begin) * sizeof(T);
            p.push_src = (const unsigned char*)g->px[b] + off;
            p.push_bytes16 = len & ~(size_t)15;
            p.push_tail = (int)((len % 16) / 4);
            p.push_peers = P - 1;
            for (int j = 1; j < P; j++) {
                const int peer = (me + j) % P;
                p.push_dst[j - 1] = (unsigned char*)g->peer_px[b][peer] + off;
                p.push_flag[j - 1] = &((DistSync*)g->peer_psync[peer])->arrive[me];
            }
            static const long long delay_us = getenv("RWR_DIST_PUSH_DELAY") ? atoll(getenv("RWR_DIST_PUSH_DELAY")) : 0;
            p.push_delay = delay_us * 1900;
        }
    }
}

// The launch parameters every iteration of a run shares: graph, seed (internal label of seed_orig, -1: uniform restart),
// hub, hot limit and workspace.  The vectors (x, x_next, r_prev, y) and the exchange are set per launch.
template <typename T>
static IterParams<T> iter_params(rwr_graph* g, const RunWorkspace& ws, int seed_orig, double c) {
    int seed_int = -1;
    if (seed_orig >= 0) {
        CUDA_CHECK(cudaMemcpyAsync(&seed_int, g->new_of_old.p + seed_orig, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
        CUDA_CHECK(cudaStreamSynchronize(g->stream));
    }
    IterParams<T> p{};
    p.n = g->n; p.inv = Prec<T>::inv(g);
    p.ws_src = g->ws_src.p; p.ws_val = Prec<T>::wsval(g); p.ws_tile = g->ws_tile.p; p.ws_tiles = g->ws_tiles; p.tile_links = g->ws_tile_links;
    p.row_begin = g->row_begin; p.row_end = g->row_end;
    p.omc = (T)(1.0 - c);                                      // Model.cs:84 `(1 - dampingFactor)`
    p.seed = seed_int; p.inv_n = g->n ? 1.0 / (double)g->n : 0.0; p.hub = ws_hub_entries(g, Prec<T>::id); p.n_hot = hot_limit(g);
    p.head_partial = ws.head.p; p.carry = ws.carry.p;
    p.slot_S = ws.slot_S.p; p.slot_R = ws.slot_R.p; p.ctl = ws.ctl.p;
    p.yv = reinterpret_cast<T*>(ws.yv.p); p.x_blocks = g->x_blocks; p.v_rows = g->v_rows;
    return p;
}

// The restart set of one rwr_run_*_restart call on the device, built by restart_prepare
struct RestartDev {
    Scratch<u32> bits, word_base;
    Scratch<int32_t> nodes, lbl;
    Scratch<double> w, q;
    RestartSet rs{};
    int init = RWR_INIT_RESTART;
    int init_node = -1;       // internal label (RWR_INIT_NODE)
};

// Runs one seed (or the restart set `set`, seed_orig -1).  mode 0: fixed n_iter; mode 1: threshold.  Final rank lands in
// y_out (internal labels).  The run starts from the constructor state (k_init, k_init_set) or, with held_S, from the rank
// y_out holds and the restart mass *held_S (device; k_init_resume): such a run is dense from its first iteration.  cont
// (a continuation of a result): launch kernel by kernel, neither using nor replacing the cached iteration graph.
template <typename T>
static void run_one(rwr_graph* g, RunWorkspace& ws, int seed_orig, double c, int mode, int n_iter, double thr, int max_iter,
                    T* y_out, int* iters_out, double* resid_out, float* iter_ms, cudaEvent_t ev0, cudaEvent_t ev1,
                    const RestartDev* set = nullptr, const double* held_S = nullptr, bool cont = false) {
    cudaStream_t st = g->stream;
    const int n = g->n;
    IterParams<T> p = iter_params<T>(g, ws, seed_orig, c);
    T* xa = reinterpret_cast<T*>(ws.x[0]);
    T* xb = reinterpret_cast<T*>(ws.x[1]);
    T* ya = reinterpret_cast<T*>(ws.ya.p);

    // uniform constructor: S0 = sum over nodes of (dangling ? 1 : 1 - fl((1-c)*1))
    const double omc_d = (double)p.omc;
    const double S_uniform = (double)g->n_dangling + (double)(n - g->n_dangling) * (1.0 - omc_d);
    // r0 goes to y_out in fixed mode (also the answer for n_iter == 0); threshold mode ping-pongs ya <-> y_out
    T* r_cur = (mode == 0) ? y_out : ya;
    // single-seed fixed-count run: the first iterations may be pushed from the frontier (frontier.cu)
    const bool fr_on = mode == 0 && ws.fw.budget > 0 && seed_orig >= 0 && !set && !held_S;
    if (held_S) {
        k_init_resume<T><<<div_up(std::max(n, 1), 256), 256, 0, st>>>(n, p.seed, p.omc, p.inv, y_out, xa, xb,
                                                                       mode == 0 ? nullptr : ya, ws.ctl.p, held_S);
        KERNEL_CHECK();
        g->pool.launches += 1;
    } else if (set) {
        k_init_set<T><<<div_up(std::max(n, 1), 256), 256, 0, st>>>(n, set->init, set->init_node, p.omc, p.inv, r_cur, xa, xb,
                                                                   ws.ctl.p, S_uniform, set->rs);
        KERNEL_CHECK();
        g->pool.launches += 1;
        if (set->init == RWR_INIT_RESTART) {
            k_restart_s0<T><<<1, FIN_THREADS, 0, st>>>(n, p.omc, p.inv, set->lbl.p, set->w.p, set->rs.m, ws.ctl.p);
            KERNEL_CHECK();
            g->pool.launches += 1;
        }
    } else {
        k_init<T><<<div_up(std::max(n, 1), 256), 256, 0, st>>>(n, p.seed, p.omc, p.inv, r_cur, xa, xb, ws.ctl.p, S_uniform,
                                                                fr_on ? ws.fw.bits : nullptr, ws.fw.words, seed_orig);
        KERNEL_CHECK();
        g->pool.launches += 1;
    }
    const RestartSet* rs = set ? &set->rs : nullptr;

    CUDA_CHECK(cudaEventRecord(ev0, st));
    T* x_cur = xa;
    T* x_nxt = xb;
    int launched = 0;
    if (mode == 0) {
        const int fr_iters = fr_on ? std::min(FR_ITERS, n_iter) : 0;
        auto launch_all = [&]() {
            for (int it = 0; it < n_iter; it++) {
                p.x = x_cur; p.x_next = x_nxt; p.r_prev = nullptr; p.y = y_out; p.iter = it;
                if (it < fr_iters) frontier_launch<T>(g, ws.fw, p, it + 1 < fr_iters);
                set_peers<T>(g, p, x_nxt);
                set_exchange<T>(g, p, x_nxt, it == 0, true);
                launch_iteration<T>(g, p, /*resid=*/false, 0.0, 0, rs);
                std::swap(x_cur, x_nxt);
            }
        };
        static const bool no_graph = getenv("RWR_NO_GRAPH") != nullptr;
        rwr_graph::IterGraph& ig = g->iter_graph[Prec<T>::id];
        const u64 fr_budget = fr_on ? ws.fw.budget : 0;
        const void* key[9] = {xa, xb, y_out, ws.ctl.p, ws.head.p, ws.carry.p, ws.slot_S.p, ws.slot_R.p, fr_on ? ws.fr.p : nullptr};
        // a restart-set run launches kernel by kernel: the graphs are keyed for seeded and uniform runs only
        const bool graphable = n_iter >= 2 && dist_n_ranks(g->comm) == 1 && !no_graph && g->x_blocks == 1 && !set && !cont;
        const bool same = ig.n_iter == n_iter && ig.hub == p.hub && ig.c == c && ig.fr_budget == fr_budget &&
                          memcmp(ig.ptr, key, sizeof(key)) == 0;
        if (graphable && same && (ig.exec || ig.seen)) {
            // second and later runs with this key: replay the graph of the whole loop (captured now if this is the second
            // run); nothing in it depends on the seed
            if (!ig.exec) {
                const int64_t counted = g->pool.launches;
                cudaGraph_t graph = nullptr;
                CUDA_CHECK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
                try {
                    launch_all();
                } catch (...) {
                    cudaStreamEndCapture(st, &graph);
                    if (graph) cudaGraphDestroy(graph);
                    throw;
                }
                CUDA_CHECK(cudaStreamEndCapture(st, &graph));
                const cudaError_t err = cudaGraphInstantiate(&ig.exec, graph, 0);
                cudaGraphDestroy(graph);
                if (err != cudaSuccess) { ig.exec = nullptr; CUDA_CHECK(err); }
                ig.launches = g->pool.launches - counted;
                g->pool.launches = counted;
            }
            CUDA_CHECK(cudaGraphLaunch(ig.exec, st));
            g->pool.launches += ig.launches;
        } else {
            // first run with this key (or no graph at all): launch kernel by kernel.  Capturing and instantiating costs more
            // than one run saves, and the reference asks each graph for a single recommendation (Experiment.cs:109).
            if (graphable) {
                if (ig.exec) { cudaGraphExecDestroy(ig.exec); ig.exec = nullptr; }
                ig.seen = true; ig.n_iter = n_iter; ig.hub = p.hub; ig.c = c; ig.fr_budget = fr_budget;
                memcpy(ig.ptr, key, sizeof(key));
            }
            launch_all();
        }
        launched = n_iter;
        *iters_out = n_iter;
        *resid_out = NAN;
    } else {
        // Model.cs:57-66.  Launch in batches; converged launches are no-ops, the flag is read between batches.
        IterCtl h{};
        const int BATCH = 8;
        bool done = false;
        while (!done) {
            for (int b = 0; b < BATCH; b++) {
                if (max_iter > 0 && launched >= max_iter) break;
                T* target = (r_cur == ya) ? y_out : ya;
                p.x = x_cur; p.x_next = x_nxt; p.r_prev = r_cur; p.y = target;
                set_peers<T>(g, p, x_nxt);
                set_exchange<T>(g, p, x_nxt, launched == 0, true);
                launch_iteration<T>(g, p, /*resid=*/true, thr, 1, rs);
                std::swap(x_cur, x_nxt);
                r_cur = target;
                launched++;
            }
            CUDA_CHECK(cudaMemcpyAsync(&h, ws.ctl.p, sizeof(h), cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaStreamSynchronize(st));
            done = h.done || (max_iter > 0 && launched >= max_iter);
        }
        *iters_out = h.iters;
        *resid_out = h.resid;
        // the rank of iteration h.iters sits in ya when h.iters is even (r0 was in ya), else in y_out
        if ((h.iters & 1) == 0 && n) CUDA_CHECK(cudaMemcpyAsync(y_out, ya, (size_t)n * sizeof(T), cudaMemcpyDeviceToDevice, st));
    }
    if (launched > 0) {
        // (overlapped exchange: the pushes are part of the k_spmv_ws launches, nothing is in flight once they have run)
        dist_allgather_rows(g, y_out, sizeof(T));                     // row-partitioned: every rank gets the whole rank vector
    }
    CUDA_CHECK(cudaEventRecord(ev1, st));
    if (!iter_ms) return;                          // the caller keeps enqueueing and reads the events after its own sync
    CUDA_CHECK(cudaEventSynchronize(ev1));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, ev0, ev1));
    *iter_ms += ms;
}

// a k_spmv_ws that gave up waiting for a peer's slice leaves a mark: the results of that run are void
static void check_exchange_fault(rwr_graph* g, const IterCtl* ctl) {
#ifndef RWR_CHECKED
    if (!g->overlap) return;
#endif
    IterCtl h{};
    CUDA_CHECK(cudaMemcpyAsync(&h, ctl, sizeof(h), cudaMemcpyDeviceToHost, g->stream));
    CUDA_CHECK(cudaStreamSynchronize(g->stream));
    if (getenv("RWR_XCHG_TRACE"))
        fprintf(stderr, "[rwr xchg r%d] %d iterations, warps waited %.3f ms in total for slices (%.4f ms per warp and iteration)\n",
                dist_rank(g->comm), h.iters, (double)h.wait_clk / 1.9e6,
                h.iters ? (double)h.wait_clk / 1.9e6 / (148.0 * 16.0) / h.iters : 0.0);
    if (h.fault > 1) RWR_FAIL(RWR_E_INVALID, "checked build: index out of bounds in the iteration kernels (code %d)", h.fault);
    if (h.fault) RWR_FAIL(RWR_E_NCCL, "row-partitioned exchange: a peer's slice of x did not arrive in time (rank out of step or down)");
}

// probe RWR_FRONTIER_TRACE: how many iterations of the run just finished the frontier kernels did (host sync per seed)
static void trace_frontier(rwr_graph* g, const RunWorkspace& ws, int seed_orig, const RestartDev* set) {
    IterCtl h{};
    CUDA_CHECK(cudaMemcpyAsync(&h, ws.ctl.p, sizeof(h), cudaMemcpyDeviceToHost, g->stream));
    CUDA_CHECK(cudaStreamSynchronize(g->stream));
    if (set)
        fprintf(stderr, "[rwr frontier] restart set of %d nodes: %d of %d iterations sparse (budget %llu links)\n", set->rs.m,
                h.sparse_iters, h.iters, (unsigned long long)ws.fw.budget);
    else
        fprintf(stderr, "[rwr frontier] seed %d: %d of %d iterations sparse (budget %llu links)\n", seed_orig, h.sparse_iters, h.iters,
                (unsigned long long)ws.fw.budget);
}

// Runs every slot of `res` from the constructor state (seeds), or -- cont -- continues every slot from the rank it holds:
// n_iter more iterations (mode 0) or a threshold run (mode 1).  A fixed-count continuation of a slot whose rank nobody
// wrote runs from the constructor state for the total count when the slot holds that state or stopped inside the sparse
// prefix (frontier.cu): the frontier kernels and the dense ones agree to the FP64 bar only, and a run of a + b iterations
// must keep the bits of run(a + b).
template <typename T>
static void run_all(rwr_graph* g, rwr_result* res, const int32_t* seeds, int n_seeds, double c, int mode, int n_iter,
                    double thr, int max_iter, int32_t* iters_out, const RestartDev* set, bool cont = false) {
    cudaStream_t st = g->stream;
    const size_t n = (size_t)g->n;
    if (Prec<T>::id == RWR_FP32) ensure_fp32_arrays(g);
    const size_t ld = (n + 3) & ~(size_t)3;
    res->ld = ld;
    if (Prec<T>::ybuf(res).n != std::max<size_t>(1, ld * (size_t)n_seeds))      // a re-run keeps its rank buffers
        Prec<T>::ybuf(res).alloc(std::max<size_t>(1, ld * (size_t)n_seeds), nullptr);
    if (res->s_keep.n != (size_t)std::max(1, n_seeds)) {
        res->s_keep.alloc((size_t)std::max(1, n_seeds), nullptr);
        res->sparse_keep.alloc((size_t)std::max(1, n_seeds), nullptr);
    }
    std::vector<int32_t> sparse((size_t)n_seeds, 0);
    if (cont && n_seeds) {
        CUDA_CHECK(cudaMemcpyAsync(sparse.data(), res->sparse_keep.p, sizeof(int32_t) * (size_t)n_seeds, cudaMemcpyDeviceToHost, st));
        CUDA_CHECK(cudaStreamSynchronize(st));
    }
    RunWorkspace ws;
    ws.alloc<T>(g, (n + 8) * sizeof(T), (mode == 0 && !set) ? frontier_budget(g) : 0);
    DevEvent ev0, ev1, evA, evB;
    const int64_t launches0 = g->pool.launches;
    CUDA_CHECK(cudaEventRecord(evA, st));
    res->iterate_ms = 0.f;
    for (int s = 0; s < n_seeds; s++) {
        int it = 0;
        double rs = NAN;
        const int done = cont ? res->iters[s] : 0;
        const bool replay = cont && mode == 0 && !set && !res->written[s] &&
                            (done == 0 || (done < FR_ITERS && sparse[s] == done));
        const double* held_S = (cont && !replay) ? res->s_keep.p + s : nullptr;
        run_one<T>(g, ws, seeds[s], c, mode, replay ? done + n_iter : n_iter, thr, max_iter,
                   Prec<T>::ybuf(res).p + (size_t)s * ld, &it, &rs, &res->iterate_ms, ev0, ev1, set, held_S, cont);
        if (replay) it -= done;                    // the iterations of this call
        res->iters[s] = done + it;
        res->residual = rs;
        if (iters_out) iters_out[s] = it;
        CUDA_CHECK(cudaMemcpyAsync(res->s_keep.p + s, &ws.ctl.p->S, sizeof(double), cudaMemcpyDeviceToDevice, st));
        CUDA_CHECK(cudaMemcpyAsync(res->sparse_keep.p + s, &ws.ctl.p->sparse_iters, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        if (getenv("RWR_FRONTIER_TRACE")) trace_frontier(g, ws, seeds[s], set);
    }
    CUDA_CHECK(cudaEventRecord(evB, st));
    CUDA_CHECK(cudaEventSynchronize(evB));
    CUDA_CHECK(cudaEventElapsedTime(&res->total_ms, evA, evB));
    res->launches = g->pool.launches - launches0;
    if (n_seeds) check_exchange_fault(g, ws.ctl.p);       // (no seed: nothing ran, and nothing has set up ctl)
}

template <typename T>
static void profile_impl(rwr_graph* g, int seed_orig, double c, int reps, float* spmv_ms, float* fixup_ms) {
    cudaStream_t st = g->stream;
    const size_t n = (size_t)g->n;
    if (Prec<T>::id == RWR_FP32) ensure_fp32_arrays(g);
    RunWorkspace ws;
    ws.alloc<T>(g, (n + 8) * sizeof(T));
    IterParams<T> p = iter_params<T>(g, ws, seed_orig, c);
    T* xa = reinterpret_cast<T*>(ws.x[0]);
    T* xb = reinterpret_cast<T*>(ws.x[1]);
    T* ya = reinterpret_cast<T*>(ws.ya.p);
    p.r_prev = nullptr; p.y = ya;
    { const char* dm = getenv("RWR_DEBUG_MODE"); p.debug = dm ? atoi(dm) : 0; }
    k_init<T><<<div_up(std::max((int)n, 1), 256), 256, 0, st>>>((int)n, p.seed, p.omc, p.inv, ya, xa, xb, ws.ctl.p, 0.0,
                                                                    nullptr, 0u, -1);
    KERNEL_CHECK();
    std::vector<DevEvent> ev(3 * (size_t)reps);
    T* x_cur = xa;
    T* x_nxt = xb;
    for (int it = 0; it < 3 + reps; it++) {
        p.x = x_cur; p.x_next = x_nxt;
        set_peers<T>(g, p, x_nxt);
        set_exchange<T>(g, p, x_nxt, true, false);       // kernel timing only: no pushes, nothing to wait for
        const int r = it - 3;
        if (r >= 0) CUDA_CHECK(cudaEventRecord(ev[3 * r], st));
        ws_launch_spmv_only<T>(g, p);
        if (r >= 0) CUDA_CHECK(cudaEventRecord(ev[3 * r + 1], st));
        ws_launch_finish_only<T>(g, p, false, 0.0, 0);
        KERNEL_CHECK();
        if (r >= 0) CUDA_CHECK(cudaEventRecord(ev[3 * r + 2], st));
        std::swap(x_cur, x_nxt);
    }
    CUDA_CHECK(cudaStreamSynchronize(st));
    double a = 0, b = 0;
    for (int r = 0; r < reps; r++) {
        float m1 = 0, m2 = 0;
        CUDA_CHECK(cudaEventElapsedTime(&m1, ev[3 * r], ev[3 * r + 1]));
        CUDA_CHECK(cudaEventElapsedTime(&m2, ev[3 * r + 1], ev[3 * r + 2]));
        a += m1; b += m2;
    }
    *spmv_ms = (float)(a / reps);
    *fixup_ms = (float)(b / reps);
    g->pool.launches += 1 + 2 * (3 + reps);
}

// One fixed-iteration run of one seed into a caller-provided rank vector (internal labels); used by the fused
// request path (rwr_recommend) so that no result object and no cudaMalloc / cudaFree sit on that path.
template <typename T>
void iterate_single_into(rwr_graph* g, int seed_orig, double c, int n_iter, T* y_out, float* iter_ms, int64_t* launches,
                         cudaEvent_t ext0, cudaEvent_t ext1) {
    if (Prec<T>::id == RWR_FP32) ensure_fp32_arrays(g);
    RunWorkspace ws;
    ws.alloc<T>(g, 16, frontier_budget(g));
    const int64_t l0 = g->pool.launches;
    int it = 0;
    double rs = 0;
#ifdef RWR_CHECKED
    const bool must_check = true;
#else
    const bool must_check = g->overlap;
#endif
    if (ext0 && ext1 && !must_check) {
        // no host synchronisation: the workspace goes back to the scratch pool while the kernels are still queued, which is
        // safe because every later user of those blocks enqueues on the same stream
        run_one<T>(g, ws, seed_orig, c, 0, n_iter, 0.0, 0, y_out, &it, &rs, nullptr, ext0, ext1);
    } else {
        DevEvent ev0, ev1;
        run_one<T>(g, ws, seed_orig, c, 0, n_iter, 0.0, 0, y_out, &it, &rs, iter_ms, ev0, ev1);
        check_exchange_fault(g, ws.ctl.p);
        if (ext0 && ext1) {                       // the caller reads its own events: bracket the (finished) run for it
            CUDA_CHECK(cudaEventRecord(ext0, g->stream));
            CUDA_CHECK(cudaEventRecord(ext1, g->stream));
        }
    }
    *launches += g->pool.launches - l0;
}
template void iterate_single_into<double>(rwr_graph*, int, double, int, double*, float*, int64_t*, cudaEvent_t, cudaEvent_t);
template void iterate_single_into<float>(rwr_graph*, int, double, int, float*, float*, int64_t*, cudaEvent_t, cudaEvent_t);

// The arguments of rwr_run_*_restart: q = weights at nodes (original labels), the initial rank `init`
struct RestartArgs {
    const int32_t* nodes;
    const double* weights;
    int32_t m;
    int32_t init;
    int32_t init_node;
};

// the argument rules of the restart-set entry points (host only, before anything touches the device)
static void restart_validate(const rwr_graph* g, const RestartArgs& a) {
    if (!a.nodes || !a.weights) RWR_FAIL(RWR_E_INVALID, "restart set: NULL node list or weights");
    if (a.m < 1) RWR_FAIL(RWR_E_INVALID, "restart set: %d nodes (at least one is needed)", a.m);
    if (a.init != RWR_INIT_UNIFORM && a.init != RWR_INIT_NODE && a.init != RWR_INIT_RESTART)
        RWR_FAIL(RWR_E_INVALID, "restart set: unknown init %d", a.init);
    if (a.init == RWR_INIT_NODE && (a.init_node < 0 || a.init_node >= g->n))
        RWR_FAIL(RWR_E_BADSEED, "restart set: init_node %d outside [0, %d)", a.init_node, g->n);
    for (int32_t k = 0; k < a.m; k++) {
        if (a.nodes[k] < 0 || a.nodes[k] >= g->n) RWR_FAIL(RWR_E_BADSEED, "restart set: node %d outside [0, %d)", a.nodes[k], g->n);
        if (!std::isfinite(a.weights[k]) || a.weights[k] < 0.0)
            RWR_FAIL(RWR_E_INVALID, "restart set: weight %g of node %d is negative or not finite", a.weights[k], a.nodes[k]);
    }
    std::vector<int32_t> sorted(a.nodes, a.nodes + a.m);
    std::sort(sorted.begin(), sorted.end());
    const auto dup = std::adjacent_find(sorted.begin(), sorted.end());
    if (dup != sorted.end()) RWR_FAIL(RWR_E_INVALID, "restart set: node %d is listed twice", *dup);
    if (dist_n_ranks(g->comm) > 1 || g->part_build) RWR_FAIL(RWR_E_UNSUPPORTED, "restart sets do not run on row-partitioned graphs");
}

// uploads the node list and the weights once and builds the bitmap, the word counts and q in internal labels
static void restart_prepare(rwr_graph* g, const RestartArgs& a, RestartDev& d) {
    cudaStream_t st = g->stream;
    const int m = a.m, words = (g->n + 31) / 32;
    d.nodes.alloc(&g->scratch, m); d.lbl.alloc(&g->scratch, m); d.w.alloc(&g->scratch, m); d.q.alloc(&g->scratch, m);
    d.bits.alloc(&g->scratch, words); d.word_base.alloc(&g->scratch, (size_t)words + 1);
    CUDA_CHECK(cudaMemcpyAsync(d.nodes.p, a.nodes, (size_t)m * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    CUDA_CHECK(cudaMemcpyAsync(d.w.p, a.weights, (size_t)m * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_CHECK(cudaMemsetAsync(d.bits.p, 0, (size_t)words * sizeof(u32), st));
    k_restart_mark<<<div_up(m, 256), 256, 0, st>>>(d.nodes.p, m, g->new_of_old.p, d.lbl.p, d.bits.p);
    KERNEL_CHECK();
    k_restart_popc<<<div_up(words, 256), 256, 0, st>>>(d.bits.p, words, d.word_base.p);
    KERNEL_CHECK();
    prim::exclusive_scan<u32>(d.word_base.p, d.word_base.p, words, d.word_base.p + words, st, &g->pool);
    d.rs.bits = d.bits.p; d.rs.word_base = d.word_base.p; d.rs.q = d.q.p; d.rs.m = m; d.rs.words = words;
    k_restart_place<<<div_up(m, 256), 256, 0, st>>>(d.lbl.p, d.w.p, m, d.rs, d.q.p);
    KERNEL_CHECK();
    g->pool.launches += 3;
    d.init = a.init;
    d.init_node = -1;
    if (a.init == RWR_INIT_NODE)
        CUDA_CHECK(cudaMemcpyAsync(&d.init_node, g->new_of_old.p + a.init_node, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
}

static int run_entry(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, int mode, int32_t n_iter, double thr,
                     int32_t max_iter, int32_t precision, int32_t* iters_out, rwr_result** out, rwr_result* reuse = nullptr,
                     const RestartArgs* restart = nullptr) {
    rwr_result* res = nullptr;
    try {
        if (!out && !reuse) RWR_FAIL(RWR_E_INVALID, "out is NULL");
        if (out) *out = nullptr;
        if (!g) RWR_FAIL(RWR_E_INVALID, "graph is NULL");
        if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run (KeyNotFoundException at Model.cs:79)");
        if (n_seeds < 0 || (n_seeds && !seeds)) RWR_FAIL(RWR_E_INVALID, "bad seed list");
        if (mode == 0 && n_iter < 0) n_iter = 0;                     // `for (n = 0; n < nIterations; ..)` runs zero times
        if (precision != RWR_FP64 && precision != RWR_FP32) RWR_FAIL(RWR_E_INVALID, "unknown precision %d", precision);
        if (!(c == c)) RWR_FAIL(RWR_E_INVALID, "c is NaN");
        for (int s = 0; s < n_seeds; s++)
            if (seeds[s] < -1 || seeds[s] >= g->n) RWR_FAIL(RWR_E_BADSEED, "seed %d outside [0, %d)", seeds[s], g->n);
        if (restart) restart_validate(g, *restart);
        if (reuse && !reuse->restart_nodes.empty())
            RWR_FAIL(RWR_E_INVALID, "a restart-set result cannot be re-run with seeds: call rwr_run_*_restart again");
        CUDA_CHECK(cudaSetDevice(g->device));
        if (mode == 1 && !(thr > 0.0)) thr = (1.0 / 1.7976931348623157e308) * (double)g->n;   // Model.cs:53
        AllocStream alloc_on(g->stream);
        res = reuse ? reuse : new rwr_result();
        res->y64.plain = true;                    // rank buffers may be freed after the graph (and its stream) are gone
        res->y32.plain = true;
        res->s_keep.plain = true;
        res->sparse_keep.plain = true;
        res->g = g;
        res->device = g->device;
        res->n_seeds = n_seeds;
        res->precision = precision;
        res->c = c;
        res->seeds.assign(seeds, seeds + n_seeds);
        res->iters.assign(n_seeds, 0);
        res->written.assign(n_seeds, 0);
        RestartDev set;
        if (restart) {
            restart_prepare(g, *restart, set);
            res->restart_nodes.assign(restart->nodes, restart->nodes + restart->m);
            res->restart_weights.assign(restart->weights, restart->weights + restart->m);
        }
        const RestartDev* sp = restart ? &set : nullptr;
        if (precision == RWR_FP64) run_all<double>(g, res, seeds, n_seeds, c, mode, n_iter, thr, max_iter, iters_out, sp);
        else run_all<float>(g, res, seeds, n_seeds, c, mode, n_iter, thr, max_iter, iters_out, sp);
        if (out) *out = res;
        return RWR_OK;
    } catch (const RwrError& e) {
        if (!reuse) delete res;
        return e.code;
    } catch (...) {
        if (!reuse) delete res;
        rwr_set_error("unexpected exception");
        return RWR_E_INVALID;
    }
}

// the result rules of the continuation entry points (rwr_continue_*, rwr_set_rank)
static void resume_validate(const rwr_result* r) {
    if (!r || !r->g) RWR_FAIL(RWR_E_INVALID, "NULL result");
    if (dist_n_ranks(r->g->comm) > 1 || r->g->part_build)
        RWR_FAIL(RWR_E_UNSUPPORTED, "a result of a row-partitioned graph cannot be continued or written");
}

// Model.run(int) / run(double) on a Model that has run: every slot continues from the rank r holds (run_all, cont)
static int continue_entry(rwr_result* r, int mode, int32_t n_iter, double thr, int32_t max_iter, int32_t* iters_out) {
    RWR_API_BEGIN
    resume_validate(r);
    if (mode == 1 && !iters_out) RWR_FAIL(RWR_E_INVALID, "iters_out is NULL");
    if (mode == 0 && n_iter <= 0) return RWR_OK;
    rwr_graph* g = r->g;
    CUDA_CHECK(cudaSetDevice(g->device));
    if (mode == 1 && !(thr > 0.0)) thr = (1.0 / 1.7976931348623157e308) * (double)g->n;   // Model.cs:53
    AllocStream alloc_on(g->stream);
    RestartDev set;
    if (!r->restart_nodes.empty()) {
        const RestartArgs a{r->restart_nodes.data(), r->restart_weights.data(), (int32_t)r->restart_nodes.size(), RWR_INIT_RESTART, -1};
        restart_prepare(g, a, set);
    }
    const RestartDev* sp = r->restart_nodes.empty() ? nullptr : &set;
    if (r->precision == RWR_FP64) run_all<double>(g, r, r->seeds.data(), r->n_seeds, r->c, mode, n_iter, thr, max_iter, iters_out, sp, true);
    else run_all<float>(g, r, r->seeds.data(), r->n_seeds, r->c, mode, n_iter, thr, max_iter, iters_out, sp, true);
    return RWR_OK;
    RWR_API_END
}

template <typename T>
static void set_rank_impl(rwr_graph* g, rwr_result* r, int slot, const double* v) {
    cudaStream_t st = g->stream;
    const int n = g->n;
    if (Prec<T>::id == RWR_FP32) ensure_fp32_arrays(g);
    Scratch<double> vd, slots;
    Scratch<IterCtl> ctl;
    vd.alloc(&g->scratch, (size_t)n);
    slots.alloc(&g->scratch, (size_t)ws_fin_grid(g));
    ctl.alloc(&g->scratch, 1);
    T* col = Prec<T>::ybuf(r).p + (size_t)slot * r->ld;
    CUDA_CHECK(cudaMemsetAsync(ctl.p, 0, sizeof(IterCtl), st));
    if (n) CUDA_CHECK(cudaMemcpyAsync(vd.p, v, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, st));
    k_set_rank<T><<<div_up(std::max(n, 1), 256), 256, 0, st>>>(n, vd.p, g->new_of_old.p, col, ctl.p);
    KERNEL_CHECK();
    k_resume_s<T><<<ws_fin_grid(g), FIN_THREADS, 0, st>>>(n, (T)(1.0 - r->c), Prec<T>::inv(g), col, slots.p, ctl.p, r->s_keep.p + slot);
    KERNEL_CHECK();
    g->pool.launches += 2;
    check_exchange_fault(g, ctl.p);
}

extern "C" {

int rwr_continue_fixed(rwr_result* r, int32_t n_iter) {
    return continue_entry(r, 0, n_iter, 0.0, 0, nullptr);
}

int rwr_continue_threshold(rwr_result* r, double thr, int32_t max_iter, int32_t* iters_out) {
    return continue_entry(r, 1, 0, thr, max_iter, iters_out);
}

int rwr_set_rank(rwr_result* r, int32_t seed_slot, const double* v) {
    RWR_API_BEGIN
    resume_validate(r);
    if (!v) RWR_FAIL(RWR_E_INVALID, "v is NULL");
    if (seed_slot < 0 || seed_slot >= r->n_seeds) RWR_FAIL(RWR_E_INVALID, "seed slot %d outside [0, %d)", seed_slot, r->n_seeds);
    rwr_graph* g = r->g;
    CUDA_CHECK(cudaSetDevice(g->device));
    AllocStream alloc_on(g->stream);
    if (r->precision == RWR_FP64) set_rank_impl<double>(g, r, seed_slot, v);
    else set_rank_impl<float>(g, r, seed_slot, v);
    r->written[seed_slot] = 1;
    r->iters[seed_slot] = 0;
    return RWR_OK;
    RWR_API_END
}

int rwr_run_fixed(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, int32_t n_iter, int32_t precision,
                  rwr_result** out) {
    return run_entry(g, seeds, n_seeds, c, 0, n_iter, 0.0, 0, precision, nullptr, out);
}

int rwr_run_threshold(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, double thr, int32_t max_iter,
                      int32_t precision, int32_t* iters_out, rwr_result** out) {
    return run_entry(g, seeds, n_seeds, c, 1, 0, thr, max_iter, precision, iters_out, out);
}

// `model.restart = q; model.run(n)` with q = weights at nodes: a Model whose restart vector the caller overwrote
int rwr_run_fixed_restart(rwr_graph* g, const int32_t* nodes, const double* weights, int32_t n_restart, int32_t init,
                          int32_t init_node, double c, int32_t n_iter, int32_t precision, rwr_result** out) {
    const int32_t none = -1;
    const RestartArgs a{nodes, weights, n_restart, init, init_node};
    return run_entry(g, &none, 1, c, 0, n_iter, 0.0, 0, precision, nullptr, out, nullptr, &a);
}

int rwr_run_threshold_restart(rwr_graph* g, const int32_t* nodes, const double* weights, int32_t n_restart, int32_t init,
                              int32_t init_node, double c, double thr, int32_t max_iter, int32_t precision, int32_t* iters_out,
                              rwr_result** out) {
    const int32_t none = -1;
    const RestartArgs a{nodes, weights, n_restart, init, init_node};
    return run_entry(g, &none, 1, c, 1, 0, thr, max_iter, precision, iters_out, out, nullptr, &a);
}

// `new Model(graph, c, seed).run(n)` again on a live Model object: same graph, seed count and precision, the rank
// buffers are reused (no device allocation on the call).
int rwr_rerun_fixed(rwr_result* r, const int32_t* seeds, double c, int32_t n_iter) {
    if (!r || !r->g) { rwr_set_error("NULL result"); return RWR_E_INVALID; }
    return run_entry(r->g, seeds, r->n_seeds, c, 0, n_iter, 0.0, 0, r->precision, nullptr, nullptr, r);
}

int rwr_result_get_info(rwr_result* r, rwr_run_info* info) {
    RWR_API_BEGIN
    if (!r || !info) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    memset(info, 0, sizeof(*info));
    info->n_seeds = r->n_seeds;
    info->n_nodes = r->g->n;
    info->precision = r->precision;
    info->iterations = r->n_seeds ? r->iters[r->n_seeds - 1] : 0;
    info->residual = r->residual;
    info->iterate_ms = r->iterate_ms;
    info->total_ms = r->total_ms;
    info->kernel_launches = r->launches;
    return RWR_OK;
    RWR_API_END
}

int rwr_scores(rwr_result* r, int32_t seed_slot, double* out_n) {
    RWR_API_BEGIN
    if (!r || !out_n) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (seed_slot < 0 || seed_slot >= r->n_seeds) RWR_FAIL(RWR_E_INVALID, "seed slot %d outside [0, %d)", seed_slot, r->n_seeds);
    rwr_graph* g = r->g;
    CUDA_CHECK(cudaSetDevice(g->device));
    const int n = g->n;
    if (n == 0) return RWR_OK;
    Scratch<double> tmp;
    tmp.alloc(&g->scratch, n);
    if (r->precision == RWR_FP64)
        k_unpermute<double><<<div_up(n, 256), 256, 0, g->stream>>>(r->y64.p + (size_t)seed_slot * r->ld, g->new_of_old.p, n, tmp.p);
    else
        k_unpermute<float><<<div_up(n, 256), 256, 0, g->stream>>>(r->y32.p + (size_t)seed_slot * r->ld, g->new_of_old.p, n, tmp.p);
    KERNEL_CHECK();
    CUDA_CHECK(cudaMemcpyAsync(out_n, tmp.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, g->stream));
    CUDA_CHECK(cudaStreamSynchronize(g->stream));
    return RWR_OK;
    RWR_API_END
}

// Times the two kernels of one iteration separately (CUDA events on the handle's stream), `reps` iterations after
// 3 warm-up iterations.  bench.py uses it for the roofline of the dominant kernel.
int rwr_profile_iteration(rwr_graph* g, int32_t seed, double c, int32_t precision, int32_t reps, float* spmv_ms,
                          float* fixup_ms) {
    RWR_API_BEGIN
    if (!g || !spmv_ms || !fixup_ms) RWR_FAIL(RWR_E_INVALID, "NULL argument");
    if (!g->built) RWR_FAIL(RWR_E_NOT_BUILT, "buildGraph() has not run");
    if (seed < 0 || seed >= g->n) RWR_FAIL(RWR_E_BADSEED, "seed %d outside [0, %d)", seed, g->n);
    if (reps < 1) reps = 1;
    CUDA_CHECK(cudaSetDevice(g->device));
    if (precision == RWR_FP32) profile_impl<float>(g, seed, c, reps, spmv_ms, fixup_ms);
    else profile_impl<double>(g, seed, c, reps, spmv_ms, fixup_ms);
    return RWR_OK;
    RWR_API_END
}

#ifdef RWR_PROFILE_CLOCKS
int rwr_debug_clocks(unsigned long long* out16, int reset) {
    if (out16) cudaMemcpyFromSymbol(out16, g_clk, sizeof(unsigned long long) * 16);
    if (reset) { unsigned long long z[16] = {0}; cudaMemcpyToSymbol(g_clk, z, sizeof(z)); }
    return 0;
}
#endif

void rwr_result_destroy(rwr_result* r) {
    if (!r) return;
    cudaSetDevice(r->device);       // never dereferences r->g: the graph may already be gone
    delete r;
}

}  // extern "C"
