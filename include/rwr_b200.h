/* rwr_b200.h -- C ABI of librwr_b200.so: the B200-native Random-Walk-with-Restart scoring path.
 *
 * Drop-in boundary for the reference's `Recommenders.RWRBased` library (C#, no FFI of its own).  Each entry
 * point names the reference member it replaces; paths are relative to the reference repository root.
 * The C# side keeps `Graph` / `Model` / `Recommender` signatures and forwards through P/Invoke
 * (recommendersystems_b200/csharp/RwrNative.cs, INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; the caller owns every input and output buffer, the library copies
 *     to/from the device and never retains host pointers;
 *   - every function returns RWR_OK (0) or a negative rwr_status; rwr_last_error() gives the message of the
 *     last failing call on the calling thread;
 *   - handles are opaque; functions are re-entrant across distinct handles (one CUDA stream and workspace
 *     per graph handle); concurrent calls on the SAME handle are not supported (neither is the reference's
 *     Model);
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with RWR_E_CUDA.
 *   - enum integer values are ABI: NodeType 0..3, EdgeType 0..7 (Recommenders/RWRBased/Recommender.cs:4-5).
 */
#ifndef RWR_B200_H
#define RWR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RWR_ABI_VERSION 2

typedef enum rwr_status {
    RWR_OK = 0,
    RWR_E_INVALID = -1,       /* bad argument (null pointer, negative size, unknown option)                    */
    RWR_E_BADSEED = -2,       /* KeyNotFoundException at Recommender.cs:21 (seed has no `edges` entry) or a     */
                              /* seed index outside [0, N)                                                      */
    RWR_E_ALREADY_BUILT = -3, /* ArgumentException from Dictionary.Add when buildGraph() runs twice, Graph.cs:86 */
    RWR_E_BADINDEX = -4,      /* IndexOutOfRangeException at Model.cs:87 (link target outside [0, N))           */
    RWR_E_NOT_BUILT = -5,     /* KeyNotFoundException at Model.cs:79 (`graph.graph[i]` before buildGraph())      */
    RWR_E_CUDA = -6,          /* CUDA runtime error / no device / extension not usable                          */
    RWR_E_NCCL = -7,
    RWR_E_OOM = -8,
    RWR_E_UNSUPPORTED = -9
} rwr_status;

/* Recommender.cs:4 */
enum { RWR_NODE_UNDEFINED = 0, RWR_NODE_USER = 1, RWR_NODE_ITEM = 2, RWR_NODE_ETC = 3 };
/* Recommender.cs:5 */
enum { RWR_EDGE_UNDEFINED = 0, RWR_EDGE_LIKE = 1, RWR_EDGE_FRIENDSHIP = 2, RWR_EDGE_FOLLOW = 3, RWR_EDGE_MENTION = 4,
       RWR_EDGE_AUTHORSHIP = 5, RWR_EDGE_PURCHASE = 6, RWR_EDGE_ETC = 7 };

enum { RWR_FP64 = 0, RWR_FP32 = 1 };

/* matrix layout of the pull CSR (W^T) used by the iteration kernels */
enum { RWR_LAYOUT_AUTO = 0,    /* index-only when every row of W has one repeated weight, else valued          */
       RWR_LAYOUT_VALUED = 1,  /* 4 B source index + one value per link                                         */
       RWR_LAYOUT_INDEX = 2 }; /* 4 B source index only; the row's common weight is folded into x (bit-equal)   */

typedef struct rwr_graph rwr_graph;     /* ~ Recommenders.RWRBased.Graph (+ the Recommender bound to it) */
typedef struct rwr_result rwr_result;   /* ~ Recommenders.RWRBased.Model after run(): one rank vector per seed */

typedef struct rwr_opts {
    int32_t device;        /* CUDA ordinal; -1 = current device                                                 */
    int32_t layout;        /* RWR_LAYOUT_*                                                                      */
    int32_t relabel;       /* 0 = auto (on): internal relabel by descending out-degree; 1 = off                 */
    int32_t hub_entries;   /* x entries staged in shared memory per CTA; -1 = auto (sized to leave L1 room), 0 = none */
    int32_t batch_width;   /* seed columns per SpMM tile; 0 = auto                                              */
    int32_t kernel;        /* reserved, must be 0 (the warp-streamed edge-stream kernels are the only SpMV path)          */
    uint64_t stream;       /* cudaStream_t to run on (0 = the handle creates its own non-blocking stream)       */
    int32_t hot_min_degree;/* nodes with fewer explicit links are clustered by first neighbour; 0 = auto (8), 1 = off */
    int32_t undefined_type_mask; /* bit t set: links of EdgeType t count as UNDEFINED at buildGraph() -- they stay in  */
                           /* `edges` but leave the matrix, as the methodology switches of Experiment.cs:84-101 do   */
                           /* by retyping FRIENDSHIP links (mask 1 << RWR_EDGE_FRIENDSHIP); LIKE links masked here   */
                           /* still exclude their targets from the recommendation (Recommender.cs:20-24)             */
    int32_t zero_weight_type_mask; /* bit t set: links of EdgeType t stay in the matrix with weight 0.0 -- what               */
                           /* DataLoader.addMentionCount2 produces for MENTION links when the member has no FRIENDSHIP link  */
                           /* (`nFriendhips * Math.Log(..) / ..`, DataLoader.cs:423-434; Methodology 15) -- and only for a   */
                           /* source that holds an explicit link of another type: a member without an `allLinks` entry gets  */
                           /* no mention links (DataLoader.cs:403-405) and stays a dangling row, not a row of NaN weights     */
    int32_t x_blocks;      /* column blocking of the gather vector for graphs whose x is far beyond L2: 0 = auto, 1 = off,    */
                           /* 2..64 = that many blocks (DESIGN.md, K10)                                                       */
    int32_t empty_seed_ok; /* 1: a seed without raw links is accepted by the recommendation calls -- an `edges` entry that   */
                           /* exists but is empty (Recommender.cs:21 only throws for a MISSING key; the flattened input      */
                           /* cannot tell the two apart, the managed shim checks ContainsKey itself and sets this)           */
    int32_t reserved;      /* must be 0                                                                                       */
} rwr_opts;

/* Deterministic synthetic generator (this repository's spec; replaces TweetRecommender/DataLoader.cs:256-436
 * and SQLiteAdapter.cs).  Integer-only, counter-based; CPU (oracle) and GPU produce identical links.        */
typedef struct rwr_synth_spec {
    uint64_t seed;
    int32_t n_users, n_items, n_third;  /* node order: USER [0,U), ITEM [U,U+T), ETC [U+T,U+T+X) (DataLoader order) */
    int32_t authorship_per_mille;       /* share of items that get an AUTHORSHIP relation                       */
    int64_t n_like, n_friend, n_follow, n_mention;   /* relations drawn (before (src,type,dst) dedup)           */
    int32_t undefined_per_mille;        /* share of FRIENDSHIP relations retyped UNDEFINED (Experiment.cs:84-101) */
    int32_t scramble;                   /* 1: pseudo-random relabel so ids carry no locality                    */
    int32_t p1_byte;                    /* per-bit probability of a 1, in 1/256 (61: R-MAT a+b = 0.76)          */
    int32_t reserved;
} rwr_synth_spec;

typedef struct rwr_graph_info {
    int32_t n_nodes;
    int32_t built;
    int64_t n_links_raw;     /* all links handed in (incl. UNDEFINED); row-partitioned handle: those this rank holds */
    int64_t nnz;             /* explicit links == nnz(W) (of the whole graph, also on a row-partitioned handle)   */
    int32_t n_dangling;      /* rows of W without explicit links (Graph.cs:53, :86 `null`)                      */
    int32_t layout;          /* RWR_LAYOUT_VALUED or RWR_LAYOUT_INDEX actually used                             */
    int32_t relabelled;
    int32_t n_hot;           /* internal labels [0, n_hot) are the degree-sorted hot nodes                      */
    int32_t hub_entries_fp64, hub_entries_fp32;
    int32_t n_chunks;        /* merge-path work items of the batched (SpMM) kernel                              */
    int32_t max_in_degree, max_out_degree;
    float build_ms;          /* rwr_graph_build device time (CUDA events)                                       */
    float synth_ms;          /* rwr_synth_create device time                                                    */
    int64_t device_bytes;    /* device memory held by the handle                                                */
    int32_t row_begin, row_end;  /* rows of W^T (internal labels) this rank iterates on: [0, N) unless partitioned   */
    int32_t n_ranks;         /* 1 unless the graph was created with rwr_*_create_partitioned                    */
    int32_t x_blocks;        /* column blocks of the gather vector the edge stream was built with (1 = none)       */
} rwr_graph_info;

typedef struct rwr_run_info {
    int32_t n_seeds;
    int32_t n_nodes;
    int32_t precision;
    int32_t iterations;      /* deliverRanks() calls of the last (or only) seed since its constructor state or the
                              * rank last written into it (rwr_set_rank)                                         */
    double residual;         /* last L1 residual (threshold mode), else NaN                                     */
    float iterate_ms;        /* device time of the power-iteration loop only (CUDA events on the stream)        */
    float total_ms;          /* init + iterations (+ top-k for rwr_recommend)                                   */
    int64_t kernel_launches; /* kernels launched by the call                                                    */
} rwr_run_info;

/* ---- library ---- */
int rwr_abi_version(void);
int rwr_device_count(void);                 /* number of CUDA devices, 0 if none/driver missing                  */
const char* rwr_last_error(void);           /* thread-local, never NULL                                          */

/* ---- graph: `new Graph(nodes, edges)` Graph.cs:45 ----
 * Links are passed flattened, `for i in 0..N-1: foreach l in edges[i]`, i.e. grouped by source with each
 * source's insertion order kept (any source order is accepted; a stable sort by source is applied when the
 * input is not already source-ascending).  A source without links == a missing `edges` key.               */
int rwr_graph_create(int32_t n_nodes, const int64_t* node_id, const int32_t* node_type, int64_t n_links,
                     const int32_t* src, const int32_t* dst, const int32_t* etype, const double* w,
                     const rwr_opts* opts, rwr_graph** out);
/* generator on the device (K0); the graph is in the same "created, not built" state as after rwr_graph_create */
int rwr_synth_create(const rwr_synth_spec* spec, const rwr_opts* opts, rwr_graph** out);
/* `Graph.buildGraph()` Graph.cs:51-88: out-degree count, exclusive scan, stable CSR scatter, sequential row
 * sums, IEEE division; then the pull layout (transpose) used by the iteration.                             */
int rwr_graph_build(rwr_graph* g);
int rwr_graph_get_info(rwr_graph* g, rwr_graph_info* info);     /* `Graph.size()` Graph.cs:91 and more       */
/* raw links back on the host, in the canonical (source, insertion) order (`Graph.nodes`, `Graph.edges`)    */
int rwr_graph_export_links(rwr_graph* g, int64_t* node_id, int32_t* node_type, int32_t* src, int32_t* dst,
                           int32_t* etype, double* w);
/* `Graph.graph` (Graph.cs:43): row_ptr[N+1], col[nnz], val[nnz]; null rows have equal row_ptr entries.
 * Not available on a row-partitioned handle (RWR_E_UNSUPPORTED: every rank holds the rows of its own sources only;
 * rwr_graph_export_links returns those links, rwr_graph_get_degrees sums over the ranks and is a collective call). */
int rwr_graph_get_csr(rwr_graph* g, int64_t* row_ptr, int32_t* col, double* val);
/* `graph[i][k].type` (Graph.cs:73-74 copies the whole ForwardLink): the EdgeType of every explicit link, CSR order     */
int rwr_graph_get_csr_types(rwr_graph* g, int32_t* etype /*[nnz]*/);
int rwr_graph_get_degrees(rwr_graph* g, int32_t* out_degree /*N explicit links*/, int32_t* raw_degree /*N, may be NULL*/);
/* On a handle created with rwr_*_create_partitioned this is a collective call (every rank destroys its handle; the
 * peer-mapped gather vectors are unmapped by all ranks before any rank frees them), made before rwr_comm_destroy.   */
void rwr_graph_destroy(rwr_graph* g);

/* ---- model: `new Model(graph, c, seed)` + `run(int)` Model.cs:33-50, :68-73 ----
 * One rank vector per seed.  seed == -1 selects the uniform-restart constructor (Model.cs:14-31).
 * `c` is the double the reference computes with: pass (double)0.15f for `Recommendation(.., 0.15f, ..)`.    */
int rwr_run_fixed(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, int32_t n_iter,
                  int32_t precision, rwr_result** out);
/* `Model.run(double threshold)` Model.cs:57-66; thr <= 0 selects `Model.run()` (Model.cs:52-55:
 * thr = (1/double.MaxValue) * N).  max_iter <= 0: unbounded like the reference (may never return when no
 * bitwise fixed point exists); iters_out[n_seeds] receives the number of deliverRanks() calls.            */
int rwr_run_threshold(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, double thr,
                      int32_t max_iter, int32_t precision, int32_t* iters_out, rwr_result** out);
/* ---- restart set: `Model.restart` (Model.cs:9) overwritten with a weighted node set, then run(int) / run(double) ----
 * q = weights[k] at nodes[k] (original labels, distinct), 0 elsewhere; q is not normalised (Model.cs:92-93, :96-97 add
 * `rank_restart * restart[r]` to every node r).  Personalized PageRank with a preference vector: a group of users, a
 * session of items.  The initial rank:
 *   RWR_INIT_UNIFORM  1 everywhere        (`new Model(graph, c)`, Model.cs:24, then restart overwritten)
 *   RWR_INIT_NODE     N at init_node      (`new Model(graph, c, init_node)`, Model.cs:44, then restart overwritten)
 *   RWR_INIT_RESTART  fl(N * q_i)         (for a one-hot q the same as RWR_INIT_NODE)
 * init_node is read for RWR_INIT_NODE only.  The result holds one rank vector (seed slot 0); rwr_topk / rwr_rank_all
 * exclude the union of the LIKE targets of the raw links of every listed node (Recommender.cs:20-24 for each of them;
 * a listed node without links adds nothing).  RWR_E_INVALID: a NULL pointer, n_restart < 1, a node listed twice, a
 * negative or non-finite weight, an unknown init; RWR_E_BADSEED: a node or init_node outside [0, N);
 * RWR_E_UNSUPPORTED: a row-partitioned handle.  rwr_rerun_fixed does not take a restart-set result (RWR_E_INVALID).  */
enum { RWR_INIT_UNIFORM = 0, RWR_INIT_NODE = 1, RWR_INIT_RESTART = 2 };
int rwr_run_fixed_restart(rwr_graph* g, const int32_t* nodes, const double* weights, int32_t n_restart, int32_t init,
                          int32_t init_node, double c, int32_t n_iter, int32_t precision, rwr_result** out);
int rwr_run_threshold_restart(rwr_graph* g, const int32_t* nodes, const double* weights, int32_t n_restart, int32_t init,
                              int32_t init_node, double c, double thr, int32_t max_iter, int32_t precision,
                              int32_t* iters_out, rwr_result** out);
/* the same Model re-run from the constructor state with other seeds (same count): rank buffers are reused, no
 * device allocation happens on the call.  The graph handle must still be alive.                             */
int rwr_rerun_fixed(rwr_result* r, const int32_t* seeds, double c, int32_t n_iter);
/* ---- a Model that has run, run again: `run(5); run(5)` is ten iterations (Model.cs:68-73), `run(double)` iterates
 * from whatever `rank` holds (Model.cs:57-66), and a caller-written `rank` (Model.cs:7) is a warm start.  A result keeps
 * per seed slot its rank, the restart mass the next iteration adds, and -- for a restart-set result -- its nodes and
 * weights; every seed slot continues from its own rank, on the device, with the precision, layout and options of the
 * run that made the result.  rwr_scores, rwr_topk and rwr_rank_all work on a continued or written result unchanged
 * (a restart-set result keeps its union LIKE exclusion); rwr_rerun_fixed still starts from the constructor state.
 * RWR_E_INVALID: a NULL r / v / iters_out, a slot outside [0, n_seeds); RWR_E_UNSUPPORTED: a result of a
 * row-partitioned handle (continuing there would be a collective call).
 * Model.run(int) on a Model that has already run: n_iter more deliverRanks() from the ranks r holds, for every slot.
 * Bit-identical to one run of the total count (same precision, layout, options).  n_iter <= 0: nothing happens. */
int rwr_continue_fixed(rwr_result* r, int32_t n_iter);
/* Model.run(double) / run() (thr <= 0) from the ranks r holds; iters_out[n_seeds] = deliverRanks() calls of THIS call;
 * max_iter <= 0: unbounded, as in rwr_run_threshold. */
int rwr_continue_threshold(rwr_result* r, double thr, int32_t max_iter, int32_t* iters_out);
/* `model.rank = v` (Model.cs:7): overwrite slot `seed_slot` with v[N] (original labels; rounded to float in FP32).
 * The next continuation starts from v, with S recomputed from it.  Any double is accepted, as the reference accepts
 * any: NaN / Inf entries poison every node one iteration later, as they do today. */
int rwr_set_rank(rwr_result* r, int32_t seed_slot, const double* v);
int rwr_result_get_info(rwr_result* r, rwr_run_info* info);
/* `Model.rank` (Model.cs:7) of one seed, widened to double in FP32 mode                                    */
int rwr_scores(rwr_result* r, int32_t seed_slot, double* out_n);
/* `Recommender.Recommendation(idx, c, nIter, topN)` Recommender.cs:42-51 on the ranks held by `r`:
 * out_ids/out_scores are [n_seeds * k], out_counts[n_seeds] (fewer than k when fewer candidates).
 * Fails with RWR_E_BADSEED when a seed has no raw links (KeyNotFoundException, Recommender.cs:21).          */
int rwr_topk(rwr_result* r, int32_t k, int64_t* out_ids, double* out_scores, int32_t* out_counts);
/* `Recommender.Recommendation(idx, c, nIter)` Recommender.cs:14-40: the full ranking of one seed,
 * (score desc, id desc); writes min(count, cap) pairs and the candidate count.                             */
int rwr_rank_all(rwr_result* r, int32_t seed_slot, int64_t* ids, double* scores, int64_t cap, int64_t* count);
void rwr_result_destroy(rwr_result* r);

/* ---- fused request path: n_seeds x `Recommendation(seed, c, nIter, k)` in seed tiles (SpMM) ----
 * Ranks are not kept; only the k best (id, score) per seed come back.                                      */
int rwr_recommend(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, int32_t n_iter,
                  int32_t precision, int32_t k, int64_t* out_ids, double* out_scores, int32_t* out_counts,
                  rwr_run_info* info /* may be NULL */);

/* ---- measurement probe: average device time of one iteration's kernels (CUDA events on the handle's stream, `reps`
 * iterations after 3 warm-up iterations): spmv_ms = k_spmv_ws, fixup_ms = k_cutrows_ws + k_finish_ws.  Used by
 * bench.py for the roofline of the dominant kernel.                                                                  */
int rwr_profile_iteration(rwr_graph* g, int32_t seed, double c, int32_t precision, int32_t reps, float* spmv_ms,
                          float* fixup_ms);
/* ---- parity probe: the rank vectors the batched request path (rwr_recommend with n_seeds >= 2, rwr_evaluate_users)
 * computes -- seeds in SpMM tiles of 8 (FP64) / 16 (FP32) consecutive seeds, n_iter iterations from the seeded
 * constructor state -- written to out[n_seeds * N] in original labels, widened to double.  For tests.  Validation as in
 * rwr_recommend (seed -1: RWR_E_INVALID, outside [0, N): RWR_E_BADSEED, row-partitioned handle: RWR_E_UNSUPPORTED); a seed
 * without raw links is accepted: that rule belongs to the recommendation, not to the iteration.                      */
int rwr_probe_tile_ranks(rwr_graph* g, const int32_t* seeds, int32_t n_seeds, double c, int32_t n_iter,
                         int32_t precision, double* out);

/* ---- evaluation (next row N1): Experiment.cs:121-128 on a ranking held on the host ---- */
int rwr_evaluate(const int64_t* ranked_ids, int64_t n, const int64_t* test_ids, int64_t n_test, int32_t* hits,
                 double* avg_precision);

/* ---- N3: `Methodology` -> feature set (TweetRecommender/DataLoader.cs:142-219, Experiment.cs:7-16, :84-101) as link-type
 * masks.  A graph that carries every relation (what Methodology.ALL loads) becomes methodology m's graph by leaving the
 * link types of *undefined_type_mask out of the matrix (types DataLoader would not have loaded, plus FRIENDSHIP where it
 * is only "temporarily included" and retyped UNDEFINED at Experiment.cs:84-101) and by zeroing the weight of the types in
 * *zero_weight_type_mask (MENTION for methodology 15, whose mention weights are `0 * ln(cnt) / ..`: no friendship was
 * loaded).  *feature_mask: bit f = Feature f (FRIENDSHIP, FOLLOWSHIP_ON_THIRDPARTY, AUTHORSHIP, MENTIONCOUNT) is in the
 * list graphConfiguration(List<Feature>, fold) receives.  Pass the two masks in rwr_opts.  Node count and third-party
 * nodes stay those of the full graph (the reference would not have created ETC nodes without followship: its scores are
 * the same up to the common factor N'/N, Model.cs:44).  Returns RWR_E_INVALID outside 0..15.                            */
int rwr_methodology_masks(int32_t methodology, int32_t* feature_mask, int32_t* undefined_type_mask,
                          int32_t* zero_weight_type_mask);

/* ---- N2: k-fold hold-out on the device: DataLoader.splitLikeHistory (DataLoader.cs:122-140) and the LIKE links that
 * never enter the graph for the test fold (:287-298), for any number of test users at once.  Call between create and
 * rwr_graph_build.  For each (distinct) user u: likes(u) = targets of u's raw LIKE links that are ITEM nodes, ordered by
 * node id (`likesList.Sort()`); unit = |likes| / n_folds; test fold = positions [unit*fold, fold < n_folds-1 ?
 * unit*(fold+1) : |likes|).  The links u->t and t->u of type LIKE with t in the test fold leave `edges`.  A held-out tweet
 * that no LIKE link reaches any more is no node of the reference's graph (DataLoader creates tweet nodes while it walks
 * somebody's likes, :291-303; addAuthorship skips tweets that are no nodes, :355-356): its remaining links leave `edges`
 * too and its node type becomes RWR_NODE_UNDEFINED -- no candidate, never a hit; node indices do not shift.  The test sets
 * stay in the handle (rwr_evaluate_users) and are returned: test_ptr[n_users+1], test_ids[min(total, cap)] (node ids,
 * ascending per user), *n_test = total.  Output pointers may be NULL.  The reference holds out the ego user (index 0)
 * only; BASELINE config 5 holds out 100k users of one graph (n_folds = 10, fold = 9: the newest tenth).                */
int rwr_graph_hold_out(rwr_graph* g, const int32_t* users, int32_t n_users, int32_t n_folds, int32_t fold,
                       int64_t* test_ptr, int64_t* test_ids, int64_t cap, int64_t* n_test);

/* ---- N1: Experiment.cs:121-128 for many users without materialising the rankings: `Recommendation(u, c, n_iter)` in
 * seed tiles; the position of every test item in the (score desc, id desc) order of Recommender.cs:34-38 is counted on
 * the device (1 + number of candidates that rank before it), then hits[u] = nHits, avg_precision[u] = (nHits == 0) ? 0 :
 * sumPrecision / nHits with sumPrecision accumulated in ranking order (Experiment.cs:124-127, :136), hits_at_k[u] = test
 * items among the first k.  A test id that is no candidate (unknown id, not an ITEM, or one of u's LIKE targets) is no
 * hit.  test_ptr / test_ids NULL: the sets stored by rwr_graph_hold_out, `users` NULL: its user list.                  */
int rwr_evaluate_users(rwr_graph* g, const int32_t* users, int32_t n_users, const int64_t* test_ptr, const int64_t* test_ids,
                       double c, int32_t n_iter, int32_t precision, int32_t k, int32_t* hits, double* avg_precision,
                       int32_t* hits_at_k, int32_t* n_test_of_user, rwr_run_info* info /* may be NULL */);

/* ---- row-partitioned single graph (no reference analogue): slices of W^T + NCCL allGather per iteration ----
 * One process per GPU.  Rank 0 calls rwr_comm_unique_id and hands the 128 bytes to the other ranks by any means
 * (the tests use torch.distributed); every rank then calls rwr_comm_create (opts->device picks the GPU) and one of
 * the *_create_partitioned functions with the SAME input, then rwr_graph_build.  From there rwr_run_fixed /
 * rwr_run_threshold / rwr_scores / rwr_topk / rwr_rank_all / rwr_recommend (k <= 16) are collective calls: every
 * rank makes them with the same arguments and every rank receives the full result.  The communicator must outlive
 * the graphs created on it.  NCCL (libnccl.so.2) is bound at run time; RWR_NCCL_LIB overrides the path.          */
typedef struct rwr_comm rwr_comm;
int rwr_comm_unique_id(void* id128 /* 128 bytes */);
int rwr_comm_create(int32_t rank, int32_t n_ranks, const void* id128, const rwr_opts* opts, rwr_comm** out);
void rwr_comm_destroy(rwr_comm* c);
/* every rank generates the same graph and keeps the rows of W^T it owns (balanced by link count)           */
int rwr_synth_create_partitioned(const rwr_synth_spec* spec, const rwr_opts* opts, rwr_comm* comm, rwr_graph** out);
int rwr_graph_create_partitioned(int32_t n_nodes, const int64_t* node_id, const int32_t* node_type, int64_t n_links,
                                 const int32_t* src, const int32_t* dst, const int32_t* etype, const double* w,
                                 const rwr_opts* opts, rwr_comm* comm, rwr_graph** out);

#ifdef __cplusplus
}
#endif
#endif /* RWR_B200_H */
