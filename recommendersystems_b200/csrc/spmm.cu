// spmm.cu -- K8: batched power iteration  Y[N,B] = (1-c) W^T R[N,B] + S[B] o Q  for B seed columns at once.
//
// Same restatement of Model.cs:76-108 as stream.cu, with one rank vector per seed laid out row-major: a gathered
// source row is 64 contiguous bytes (B = 8 FP64 / 16 FP32 columns), so one matrix pass serves B seeds and every
// gathered sector is fully used.  Four lanes (a quad) own one destination row at a time, 16 bytes of the row each.
//   k_spmm        8 groups x 128 threads per CTA, merge-path tiles over the pull CSR (k_partition, iterate.cu: equal
//                 rows + links per tile); tile indices (and values) staged in
//                 shared memory; rows < 32 nnz: one quad, sources in storage order; 32..255: one warp; >= 256: the group
//   k_spmm_fixup  rows cut by a tile boundary, the B seed entries (+S_j), fixed-order reduction of the restart masses
#include <algorithm>
#include <cmath>

#include "iterate.h"

constexpr int MM_GROUPS = 8;
constexpr int MM_THREADS = MM_GROUPS * GROUP_THREADS;     // 1024
constexpr int MM_QUADS = GROUP_THREADS / 4;               // 32 rows in flight per group
constexpr int MM_LONG = 32, MM_HUGE = 256;
static_assert(CHUNK_ITEMS / MM_LONG + 1 <= 32 && CHUNK_ITEMS / MM_HUGE + 2 <= 8, "capacity of the per-group row lists");
constexpr int MM_MAXB = 16;

template <typename T> struct Vec;
template <> struct Vec<double> { typedef double2 type; static constexpr int CW = 2; static constexpr int B = 8; };
template <> struct Vec<float> { typedef float4 type; static constexpr int CW = 4; static constexpr int B = 16; };

struct MMCtl {
    double S[MM_MAXB];
    double seed_sum[MM_MAXB];
    int seed_flag[MM_MAXB];
    unsigned ticket;
    int fault;             // checked build (-DRWR_CHECKED): a gather source outside [0, n)
    unsigned poison;       // bit j: the S_j this iteration used was NaN / Inf -> every entry of column j is NaN (k_spmm_poison)
};

template <typename T>
struct MMParams {
    const u32* in_ptr;
    const int32_t* in_src;
    const T* in_val;
    const int2* part;
    int n_chunks, n;
    int n_keep;            // source rows below stay in L2 (evict-last); the rest is streamed (evict-first)
    const T* x;            // [n, B]
    const T* inv;          // [n]
    T* y;                  // [n, B] or null
    T* x_next;             // [n, B]
    T omc;
    int seeds[MM_MAXB];    // internal labels, -2: inactive column
    double* head;          // [n_chunks, B]
    double* carry;         // [n_chunks, B]
    double* slot_S;        // [grid + fix_grid, B]
    MMCtl* ctl;
};

__device__ __forceinline__ void mm_group_sync(int group) {
    asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "r"(GROUP_THREADS) : "memory");
}

// 16-byte gather of piece `piece` of source row `src` (read-only path, keep in L2)
__device__ __forceinline__ void ld_piece(const double* x, int src, int piece, u64 pol, double (&v)[2]) {
    const double* p = x + (size_t)src * 8 + piece * 2;
    asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v[0]), "=d"(v[1]) : "l"(p), "l"(pol));
}
__device__ __forceinline__ void ld_piece(const float* x, int src, int piece, u64 pol, float (&v)[4]) {
    const float* p = x + (size_t)src * 16 + piece * 4;
    asm volatile("ld.global.nc.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "l"(p), "l"(pol));
}
__device__ __forceinline__ void st_piece(double* dst, const double (&v)[2], u64 pol) {
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(dst), "d"(v[0]), "d"(v[1]), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_piece(float* dst, const float (&v)[4], u64 pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(dst), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]), "l"(pol)
                 : "memory");
}

// sum over edges q0, q0 + step, ... < q1 of the tile (positions relative to the tile base) for this lane's piece.
// Loads are issued four at a time; additions follow the edge order.
template <typename T, bool VALUED>
__device__ __forceinline__ void accumulate(const MMParams<T>& p, const int* idx_s, const T* val_s, u32 q0, u32 q1, u32 step,
                                           int piece, u64 pol_keep, u64 pol_stream, double (&acc)[Vec<T>::CW]) {
    constexpr int CW = Vec<T>::CW;
    for (u32 q = q0; q < q1; q += 4 * step) {
        T v[4][CW];
        T w[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const u32 qq = (q + k * step < q1) ? q + k * step : q;        // clamped: always a valid slot
            int src = idx_s[qq];
#ifdef RWR_CHECKED
            if (src < 0 || src >= p.n) { p.ctl->fault = 2; src = 0; }
#endif
            ld_piece(p.x, src, piece, src < p.n_keep ? pol_keep : pol_stream, v[k]);
            if (VALUED) w[k] = val_s[qq];
        }
        if (sizeof(T) == 4) {
            // FP32 mode: the four products of a round are added in float (three additions of non-negative terms, <= 2 ulp of
            // float) and enter the double accumulator as one value -- a quarter of the F2F.F64.F32 conversions and FP64
            // additions, which share the narrow FP64 pipe (1e-6 L1 is the bar of this mode; the FP64 mode is untouched)
#pragma unroll
            for (int c = 0; c < CW; c++) {
                T part = (T)0;
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    T t = v[k][c];
                    if (VALUED) t = mul_rn(t, w[k]);
                    part = add_rn(part, (q + k * step < q1) ? t : (T)0);
                }
                acc[c] = __dadd_rn(acc[c], (double)part);
            }
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const bool on = q + k * step < q1;
#pragma unroll
                for (int c = 0; c < CW; c++) {
                    T t = v[k][c];
                    if (VALUED) t = mul_rn(t, w[k]);
                    acc[c] = __dadd_rn(acc[c], on ? (double)t : 0.0);
                }
            }
        }
    }
}

template <typename T, bool WRITE_Y>
__device__ __forceinline__ void mm_finalize(const MMParams<T>& p, const int* seeds_s, int row, int piece, u64 pol_keep,
                                            u64 pol_stream, const double (&sum)[Vec<T>::CW], double (&accS)[Vec<T>::CW]) {
    constexpr int CW = Vec<T>::CW, B = Vec<T>::B;
    const T invr = p.inv[row];
    T yv[CW], xv[CW];
#pragma unroll
    for (int c = 0; c < CW; c++) {
        const int col = piece * CW + c;
        const T y = (T)sum[c];
        const T rw = mul_rn(p.omc, y);
        yv[c] = y;
        xv[c] = mul_rn(rw, invr);
        const int sd = seeds_s[col];
        if (row == sd) {                              // the seed entry waits for +S_j in the fix-up kernel
            p.ctl->seed_sum[col] = sum[c];
            p.ctl->seed_flag[col] = 1;
        } else if (sd >= 0) {
            accS[c] += (invr == (T)0) ? (double)y : (double)sub_rn(y, rw);
        }
    }
    if (WRITE_Y) st_piece(p.y + (size_t)row * B + piece * CW, yv, pol_stream);
    st_piece(p.x_next + (size_t)row * B + piece * CW, xv, row < p.n_keep ? pol_keep : pol_stream);
}

template <typename T>
__device__ __forceinline__ void mm_emit_partial(double* dst, int chunk, int piece, const double (&sum)[Vec<T>::CW]) {
    constexpr int CW = Vec<T>::CW, B = Vec<T>::B;
#pragma unroll
    for (int c = 0; c < CW; c++) dst[(size_t)chunk * B + piece * CW + c] = sum[c];
}

// reduce `acc` over the quads of a warp (lanes with the same piece): xor 4, 8, 16 -- fixed tree, result in every lane
template <int CW>
__device__ __forceinline__ void quad_reduce(double (&acc)[CW]) {
#pragma unroll
    for (int o = 4; o < 32; o <<= 1)
#pragma unroll
        for (int c = 0; c < CW; c++) acc[c] = __dadd_rn(acc[c], __shfl_xor_sync(0xffffffffu, acc[c], o));
}

template <typename T, bool VALUED, bool WRITE_Y>
__global__ void __launch_bounds__(MM_THREADS, 1) k_spmm(const MMParams<T> p) {
    constexpr int CW = Vec<T>::CW, B = Vec<T>::B;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // per group: idx[CHUNK_SPAN] | val[CHUNK_SPAN] (valued) | lists | warp partials
    constexpr int GROUP_BYTES = CHUNK_SPAN * 4 + (VALUED ? CHUNK_SPAN * (int)sizeof(T) : 0) + 1024 + 4 * 16 * 8;
    const int group = threadIdx.x / GROUP_THREADS, gtid = threadIdx.x % GROUP_THREADS;
    const int lane = threadIdx.x & 31, gwarp = gtid >> 5;
    const int quad = gtid >> 2, piece = gtid & 3;
    unsigned char* gbase = smem_raw + 4096 + (size_t)group * GROUP_BYTES;
    int* idx_s = reinterpret_cast<int*>(gbase);
    T* val_s = reinterpret_cast<T*>(gbase + CHUNK_SPAN * 4);
    int* lists = reinterpret_cast<int*>(gbase + CHUNK_SPAN * 4 + (VALUED ? CHUNK_SPAN * (int)sizeof(T) : 0));
    int* l_r = lists; int* l_s = lists + 32; int* l_e = lists + 64; int* l_rs = lists + 96;     // long rows (cap 32)
    int* h_r = lists + 128; int* h_s = lists + 136; int* h_e = lists + 144; int* h_rs = lists + 152;   // huge rows (cap 8)
    int* l_cnt = lists + 160; int* h_cnt = lists + 161;
    double* wpart = reinterpret_cast<double*>(lists + 256);                 // [4 warps][16 columns]
    double* scratch = reinterpret_cast<double*>(smem_raw);                  // block reduce: [32 warps][16 columns] doubles
    __shared__ int seeds_s[MM_MAXB];
    if (threadIdx.x < MM_MAXB) seeds_s[threadIdx.x] = p.seeds[threadIdx.x];
    __syncthreads();

    if (gtid == 0) { *l_cnt = 0; *h_cnt = 0; }
    const u64 pol_stream = policy_evict_first(), pol_keep = policy_evict_last();
    double accS[CW];
#pragma unroll
    for (int c = 0; c < CW; c++) accS[c] = 0.0;
    const int stride = gridDim.x * MM_GROUPS;
    int chunk = blockIdx.x * MM_GROUPS + group;
    int2 c0 = make_int2(0, 0), c1 = make_int2(0, 0);
    int4 iv[CHUNK_ROUNDS];
    T wv[CHUNK_ROUNDS][4];
    auto load_tile_regs = [&](int ch) {
        c0 = p.part[ch];
        c1 = p.part[ch + 1];
        const u32 nnz1 = (u32)c1.y, base = (u32)c0.y & ~3u;
#pragma unroll
        for (int j = 0; j < CHUNK_ROUNDS; j++) {
            const u32 pos = base + (u32)(j * GROUP_THREADS + gtid) * 4u;
            iv[j] = make_int4(0, 0, 0, 0);
            if (pos < nnz1) {
                iv[j] = ld_stream_int4(reinterpret_cast<const int4*>(p.in_src + pos), pol_stream);
                if (VALUED) {
#pragma unroll
                    for (int k = 0; k < 4; k++) wv[j][k] = ld_stream(p.in_val + pos + k, pol_stream);
                }
            }
        }
    };
    if (chunk < p.n_chunks) load_tile_regs(chunk);
    mm_group_sync(group);

    for (; chunk < p.n_chunks; chunk += stride) {
        const u32 nnz0 = (u32)c0.y, nnz1 = (u32)c1.y, base = nnz0 & ~3u;
        const int row0 = c0.x, row1 = c1.x;
        // ---- stage this tile's indices (and values) in shared memory, then prefetch the next tile into registers
#pragma unroll
        for (int j = 0; j < CHUNK_ROUNDS; j++) {
            const u32 rel = (u32)(j * GROUP_THREADS + gtid) * 4u;
            if (base + rel < nnz1) {
                *reinterpret_cast<int4*>(idx_s + rel) = iv[j];
                if (VALUED) {
#pragma unroll
                    for (int k = 0; k < 4; k++) val_s[rel + k] = wv[j][k];
                }
            }
        }
        const int next = chunk + stride;
        if (next < p.n_chunks) load_tile_regs(next);
        mm_group_sync(group);

        // ---- pass A: one quad per row, sources in storage order (rows < 32 nnz); longer rows go to the lists
        for (int r = row0 + quad; r <= row1 && r < p.n; r += MM_QUADS) {
            const bool complete = r < row1;
            const u32 rs = p.in_ptr[r];
            const u32 s = rs > nnz0 ? rs : nnz0;
            u32 e = complete ? p.in_ptr[r + 1] : nnz1;
            if (e < s) e = s;
            const u32 len = e - s;
            if (len >= (u32)MM_LONG) {
                if (piece == 0) {
                    if (len >= (u32)MM_HUGE) {
                        const int slot = atomicAdd(h_cnt, 1);
                        h_r[slot] = r; h_s[slot] = (int)(s - base); h_e[slot] = (int)(e - base); h_rs[slot] = (int)rs;
                    } else {
                        const int slot = atomicAdd(l_cnt, 1);
                        l_r[slot] = r; l_s[slot] = (int)(s - base); l_e[slot] = (int)(e - base); l_rs[slot] = (int)rs;
                    }
                }
                continue;
            }
            double acc[CW];
#pragma unroll
            for (int c = 0; c < CW; c++) acc[c] = 0.0;
            accumulate<T, VALUED>(p, idx_s, val_s, s - base, e - base, 1, piece, pol_keep, pol_stream, acc);
            if (!complete) mm_emit_partial<T>(p.carry, chunk, piece, acc);
            else if (rs < nnz0) mm_emit_partial<T>(p.head, chunk, piece, acc);
            else mm_finalize<T, WRITE_Y>(p, seeds_s, r, piece, pol_keep, pol_stream, acc, accS);
        }
        mm_group_sync(group);
        // ---- pass B: rows of 32..255 nnz, one warp each: 8 quads stride over the edges, fixed shuffle tree.  The lists
        // fill in atomicAdd order, which depends on the timing of the warps; passes B and C visit them in an order of their
        // own, so that every thread adds the same rows to its restart-mass partials (accS) in the same order on every run.
        // Pass B: longest first (ties by row), dealt to the 4 warps in snake order (0 1 2 3 3 2 1 0 ...) -- balanced
        const int n_long = *l_cnt;
        int my_rank = lane;                                 // rank of list entry `lane` (the keys are distinct)
        if (n_long > 1) {
            const int my_key = lane < n_long ? ((1023 - (l_e[lane] - l_s[lane])) << 10) | (l_r[lane] - row0) : 0x7fffffff;
            my_rank = 0;
#pragma unroll
            for (int j = 0; j < 32; j++) my_rank += __shfl_sync(0xffffffffu, my_key, j) < my_key;
        }
        for (int k = 0;; k++) {
            const int q = 4 * k + ((k & 1) ? 3 - gwarp : gwarp);
            if (q >= n_long) break;
            const int li = __ffs(__ballot_sync(0xffffffffu, my_rank == q)) - 1;
            const int r = l_r[li];
            const u32 s = (u32)l_s[li], e = (u32)l_e[li], rs = (u32)l_rs[li];
            double acc[CW];
#pragma unroll
            for (int c = 0; c < CW; c++) acc[c] = 0.0;
            accumulate<T, VALUED>(p, idx_s, val_s, s + (lane >> 2), e, 8, piece, pol_keep, pol_stream, acc);
            quad_reduce<CW>(acc);
            if (lane < 4) {
                if (r >= row1) mm_emit_partial<T>(p.carry, chunk, piece, acc);
                else if (rs < nnz0) mm_emit_partial<T>(p.head, chunk, piece, acc);
                else mm_finalize<T, WRITE_Y>(p, seeds_s, r, piece, pol_keep, pol_stream, acc, accS);
            }
        }
        // ---- pass C: rows of >= 256 nnz (at most 3 per tile), in row order: the whole group
        const int n_huge = *h_cnt;
        for (int q = 0, prev = -1; q < n_huge; q++) {
            int hi = 0;                                     // the entry with the q-th smallest row
            for (int j = 1; j < n_huge; j++)
                if (h_r[j] > prev && (h_r[hi] <= prev || h_r[j] < h_r[hi])) hi = j;
            const int r = h_r[hi];
            prev = r;
            const u32 s = (u32)h_s[hi], e = (u32)h_e[hi], rs = (u32)h_rs[hi];
            double acc[CW];
#pragma unroll
            for (int c = 0; c < CW; c++) acc[c] = 0.0;
            accumulate<T, VALUED>(p, idx_s, val_s, s + quad, e, MM_QUADS, piece, pol_keep, pol_stream, acc);
            quad_reduce<CW>(acc);
            if (lane < 4) {
#pragma unroll
                for (int c = 0; c < CW; c++) wpart[gwarp * 16 + piece * CW + c] = acc[c];
            }
            mm_group_sync(group);
            if (gtid < 4) {
                double tot[CW];
#pragma unroll
                for (int c = 0; c < CW; c++) {
                    tot[c] = 0.0;
                    for (int w = 0; w < GROUP_THREADS / 32; w++) tot[c] = __dadd_rn(tot[c], wpart[w * 16 + piece * CW + c]);
                }
                if (r >= row1) mm_emit_partial<T>(p.carry, chunk, piece, tot);
                else if (rs < nnz0) mm_emit_partial<T>(p.head, chunk, piece, tot);
                else mm_finalize<T, WRITE_Y>(p, seeds_s, r, piece, pol_keep, pol_stream, tot, accS);
            }
            mm_group_sync(group);
        }
        mm_group_sync(group);                       // indices and lists are free again
        if (gtid == 0) { *l_cnt = 0; *h_cnt = 0; }
    }

    // ---- restart-mass partials: per column, fixed order (quads of a warp, then the 32 warps)
    quad_reduce<CW>(accS);
    __syncthreads();
    if (lane < 4) {
#pragma unroll
        for (int c = 0; c < CW; c++) scratch[(threadIdx.x >> 5) * 16 + piece * CW + c] = accS[c];
    }
    __syncthreads();
    if (threadIdx.x < B) {
        double tot = 0.0;
        for (int w = 0; w < MM_THREADS / 32; w++) tot += scratch[w * 16 + threadIdx.x];
        p.slot_S[(size_t)blockIdx.x * B + threadIdx.x] = tot;
    }
}

// One thread per (chunk, column): rows cut by a tile boundary; then the seed entries; then the final reduction.
template <typename T, bool WRITE_Y>
__global__ void __launch_bounds__(256) k_spmm_fixup(const MMParams<T> p, int main_grid) {
    constexpr int B = Vec<T>::B;
    __shared__ double sm[256];
    __shared__ int is_last;
    MMCtl* ctl = p.ctl;
    const int tid = blockIdx.x * 256 + threadIdx.x;
    const int k = tid / B, col = tid % B;
    double accS = 0.0;
    auto finalize_scalar = [&](int row, double total) {
        const T invr = p.inv[row];
        const T y = (T)total;
        const T rw = mul_rn(p.omc, y);
        if (WRITE_Y) p.y[(size_t)row * B + col] = y;
        p.x_next[(size_t)row * B + col] = mul_rn(rw, invr);
        if (p.seeds[col] >= 0) accS += (invr == (T)0) ? (double)y : (double)sub_rn(y, rw);
    };
    if (k < p.n_chunks) {
        const int2 c0 = p.part[k], c1 = p.part[k + 1];
        if (c0.x < c1.x && p.in_ptr[c0.x] < (u32)c0.y) {
            const int row = c0.x;
            int m0 = k - 1;
            while (m0 > 0 && p.part[m0].x == row) m0--;
            double total = 0.0;
            for (int m = m0; m < k; m++) total = __dadd_rn(total, p.carry[(size_t)m * B + col]);
            total = __dadd_rn(total, p.head[(size_t)k * B + col]);
            if (row == p.seeds[col]) total = __dadd_rn(total, ctl->S[col]);
            finalize_scalar(row, total);
        }
    }
    if (k == 0 && ctl->seed_flag[col]) {                       // seed entry of column `col` finished inside one tile
        finalize_scalar(p.seeds[col], __dadd_rn(ctl->seed_sum[col], ctl->S[col]));
        ctl->seed_flag[col] = 0;
    }
    // per-column block reduction in thread order
    sm[threadIdx.x] = accS;
    __syncthreads();
    if (threadIdx.x < B) {
        double tot = 0.0;
        for (int i = threadIdx.x; i < 256; i += B) tot += sm[i];
        p.slot_S[(size_t)(main_grid + blockIdx.x) * B + threadIdx.x] = tot;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned t = atomicAdd(&ctl->ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        const int total = main_grid + (int)gridDim.x;
        // 256 threads: column = threadIdx.x % B, 256 / B strided partial sums, then a fixed-order combine
        double a = 0.0;
        for (int i = threadIdx.x / B; i < total; i += 256 / B) a += __ldcg(p.slot_S + (size_t)i * B + (threadIdx.x % B));
        sm[threadIdx.x] = a;
        __syncthreads();
        if (threadIdx.x == 0) ctl->poison = 0;
        __syncthreads();
        if (threadIdx.x < B) {
            double tot = 0.0;
            for (int i = threadIdx.x; i < 256; i += B) tot += sm[i];
            // the S_j this iteration ran with: `S * 0` is NaN iff some rank of the previous vector was NaN / Inf (see k_spmm_poison)
            if (p.seeds[threadIdx.x] >= 0 && !((ctl->S[threadIdx.x] * 0.0) == 0.0)) atomicOr(&ctl->poison, 1u << threadIdx.x);
            ctl->S[threadIdx.x] = tot;
            if (threadIdx.x == 0) ctl->ticket = 0;
        }
    }
}

// Model.cs:92-93 / :96-97 add `x * restart[r]` to EVERY node r.  With a one-hot restart vector that is `x * 0`: nothing, unless a
// rank x of the previous vector is NaN or Inf (a row whose weights sum to 0, Graph.cs:81) -- then every entry of the next
// vector is NaN in the reference.  k_spmm_fixup marks such columns; this kernel (a no-op otherwise: one word read per block)
// overwrites them.
template <typename T, bool WRITE_Y>
__global__ void __launch_bounds__(256) k_spmm_poison(const MMParams<T> p) {
    constexpr int B = Vec<T>::B;
    const unsigned mask = p.ctl->poison;
    if (mask == 0) return;
    const T nan = (T)__longlong_as_double(0x7ff8000000000000LL);
    const size_t total = (size_t)p.n * B;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (size_t)gridDim.x * 256) {
        if ((mask >> (unsigned)(i % B)) & 1u) {
            p.x_next[i] = nan;
            if (WRITE_Y) p.y[i] = nan;
        }
    }
}

template <typename T>
__global__ void k_spmm_init(int n, MMParams<T> p, T* __restrict__ r0 /* may be null */, T* __restrict__ x0) {
    constexpr int B = Vec<T>::B;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) {
        for (int c = 0; c < MM_MAXB; c++) { p.ctl->seed_sum[c] = 0.0; p.ctl->seed_flag[c] = 0; p.ctl->S[c] = 0.0; }
        p.ctl->ticket = 0;
        p.ctl->fault = 0;
        p.ctl->poison = 0;
    }
    if (i >= (size_t)n * B) return;
    const int row = (int)(i / B), col = (int)(i % B);
    const T r = (row == p.seeds[col]) ? (T)n : (T)0;              // Model.cs:44
    const T invr = p.inv[row];
    const T rw = mul_rn(p.omc, r);
    if (r0) r0[i] = r;
    x0[i] = mul_rn(rw, invr);
}
template <typename T>
__global__ void k_spmm_init_S(int n, MMParams<T> p) {           // after k_spmm_init: S_j of the constructor state
    constexpr int B = Vec<T>::B;
    const int col = threadIdx.x;
    if (col < B && p.seeds[col] >= 0) {
        const T r = (T)n, invr = p.inv[p.seeds[col]], rw = mul_rn(p.omc, r);
        p.ctl->S[col] = (invr == (T)0) ? (double)r : (double)sub_rn(r, rw);
    }
}

// ------------------------------------------------------------------------------------------------ host side
template <typename T> struct PrecMM;
template <> struct PrecMM<double> {
    static const double* inv(rwr_graph* g) { return g->inv64.p; }
    static const double* val(rwr_graph* g) { return g->in_val64.p; }
};
template <> struct PrecMM<float> {
    static const float* inv(rwr_graph* g) { return g->inv32.p; }
    static const float* val(rwr_graph* g) { return g->in_val32.p; }
};

void ensure_fp32_arrays(rwr_graph* g);    // iterate.cu

template <typename T>
struct SpmmWorkspace {
    Scratch<T> xa, xb;
    Scratch<double> head, carry, slot_S;
    Scratch<MMCtl> ctl;
    int main_grid = 0, fix_grid = 0;
    size_t smem = 0;
};

template <typename T>
static size_t spmm_smem_bytes(bool valued) {
    const size_t group = CHUNK_SPAN * 4 + (valued ? CHUNK_SPAN * sizeof(T) : 0) + 1024 + 4 * 16 * 8;
    return 4096 + MM_GROUPS * group;
}

// Runs n_iter iterations for up to B seeds (internal labels in seeds_int, -2 pads); the ranks of the last iteration
// land row-major in y_out[n, B].  n_iter == 0: the constructor state.
template <typename T>
void spmm_run_tile(rwr_graph* g, const int* seeds_int, int n_active, double c, int n_iter, T* y_out, int64_t* launches) {
    constexpr int B = Vec<T>::B;
    cudaStream_t st = g->stream;
    const size_t n = (size_t)g->n;
    const bool valued = g->layout == RWR_LAYOUT_VALUED;
    SpmmWorkspace<T> ws;
    ws.xa.alloc(&g->scratch, n * B + 16); ws.xb.alloc(&g->scratch, n * B + 16);
    ws.head.alloc(&g->scratch, (size_t)g->n_chunks * B); ws.carry.alloc(&g->scratch, (size_t)g->n_chunks * B);
    ws.main_grid = std::max(1, std::min(g->sm_count, (g->n_chunks + MM_GROUPS - 1) / MM_GROUPS));
    ws.fix_grid = (int)div_up((size_t)g->n_chunks * B, 256);
    ws.slot_S.alloc(&g->scratch, (size_t)(ws.main_grid + ws.fix_grid) * B);
    ws.ctl.alloc(&g->scratch, 1);
    CUDA_CHECK(cudaMemsetAsync(ws.head.p, 0, (size_t)g->n_chunks * B * sizeof(double), st));
    CUDA_CHECK(cudaMemsetAsync(ws.carry.p, 0, (size_t)g->n_chunks * B * sizeof(double), st));
    CUDA_CHECK(cudaMemsetAsync(ws.slot_S.p, 0, (size_t)(ws.main_grid + ws.fix_grid) * B * sizeof(double), st));
    ws.smem = spmm_smem_bytes<T>(valued);

    MMParams<T> p;
    p.in_ptr = g->in_ptr.p; p.in_src = g->in_src.p; p.in_val = PrecMM<T>::val(g); p.part = g->part.p;
    p.n_chunks = g->n_chunks; p.n = g->n; p.inv = PrecMM<T>::inv(g);
    // rows of x and x_next that may stay L2-resident: ~40 MB each of the 126 MB L2
    p.n_keep = std::min<int>(g->n_hot, (int)((40u << 20) / (B * sizeof(T))));
    p.omc = (T)(1.0 - c);
    for (int j = 0; j < MM_MAXB; j++) p.seeds[j] = (j < n_active) ? seeds_int[j] : -2;
    p.head = ws.head.p; p.carry = ws.carry.p; p.slot_S = ws.slot_S.p; p.ctl = ws.ctl.p;
    p.x = nullptr; p.x_next = nullptr; p.y = nullptr;
    const size_t total = n * B;
    k_spmm_init<T><<<div_up(std::max<size_t>(total, 1), 256), 256, 0, st>>>(g->n, p, y_out, ws.xa.p);
    k_spmm_init_S<T><<<1, 32, 0, st>>>(g->n, p);
    KERNEL_CHECK();
    *launches += 2;
    T* x_cur = ws.xa.p;
    T* x_nxt = ws.xb.p;
    for (int it = 0; it < n_iter; it++) {
        p.x = x_cur; p.x_next = x_nxt; p.y = y_out;
        const bool last = it == n_iter - 1;
#define MM_LAUNCH(V, W)                                                                                         \
    do {                                                                                                        \
        auto kern = k_spmm<T, V, W>;                                                                            \
        CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ws.smem));      \
        kern<<<ws.main_grid, MM_THREADS, ws.smem, st>>>(p);                                                     \
        k_spmm_fixup<T, W><<<ws.fix_grid, 256, 0, st>>>(p, ws.main_grid);                                       \
        k_spmm_poison<T, W><<<std::max(1, g->sm_count), 256, 0, st>>>(p);                                       \
    } while (0)
        if (valued) { if (last) MM_LAUNCH(true, true); else MM_LAUNCH(true, false); }
        else { if (last) MM_LAUNCH(false, true); else MM_LAUNCH(false, false); }
#undef MM_LAUNCH
        KERNEL_CHECK();
        *launches += 3;
        std::swap(x_cur, x_nxt);
    }
    CUDA_CHECK(cudaStreamSynchronize(st));      // the workspace goes back to the handle's scratch pool on return
#ifdef RWR_CHECKED
    MMCtl h{};
    CUDA_CHECK(cudaMemcpy(&h, ws.ctl.p, sizeof(h), cudaMemcpyDeviceToHost));
    if (h.fault) RWR_FAIL(RWR_E_INVALID, "checked build: k_spmm index out of bounds (code %d)", h.fault);
#endif
}

template void spmm_run_tile<double>(rwr_graph*, const int*, int, double, int, double*, int64_t*);
template void spmm_run_tile<float>(rwr_graph*, const int*, int, double, int, float*, int64_t*);

int spmm_tile_width(int precision) { return precision == RWR_FP32 ? Vec<float>::B : Vec<double>::B; }
