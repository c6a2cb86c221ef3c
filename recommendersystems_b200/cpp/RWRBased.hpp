// RWRBased.hpp -- C++ host side of the drop-in: the public surface of the reference's `Recommenders.RWRBased`
// (Recommenders/RWRBased/Graph.cs, Model.cs, Recommender.cs) over the C ABI of librwr_b200.so (include/rwr_b200.h).
//
// The reference is compiled code (C#) and this image has no C# toolchain, so next to the P/Invoke shim shipped as source
// (../csharp/) the same surface exists in C++: same type and member names, same argument meaning, the .NET exceptions the
// reference's callers can see as C++ exception types of the same name.  A caller written against the reference
// (TweetRecommender/Experiment.cs:104-109) reads the same here:
//
//     Graph graph(nodes, edges);                 // Dictionary<int, Node>, Dictionary<int, List<ForwardLink>>
//     graph.buildGraph();
//     Recommender recommender(graph);
//     auto recommendation = recommender.Recommendation(0, 0.15f, nIterations);      // List<KeyValuePair<long, double>>
//
// (or, spelt the way oracle/cs2cpp.py respells C# class references: `Graph* graph = new Graph(nodes, edges); graph->buildGraph();
// Recommender* recommender = new Recommender(graph);` -- tests/cpp/experiment_caller.cpp is ONE such caller, compiled against this
// header and against the reference's own sources; the two programs must print the same lists.)
//
// Header only; link with -lrwr_b200.  Nothing is computed here: flattening `edges` in `for i in 0..N-1: foreach l in edges[i]`
// order (rwr_graph_create's input contract), widening `float dampingFactor` to double exactly as Recommender.cs:16 does, and
// mapping status codes to exceptions.  There is no CPU fallback: without a CUDA device every call throws RwrException(RWR_E_CUDA).
#pragma once

#include <cstdint>
#include <cstring>
#include <limits>
#include <map>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../../include/rwr_b200.h"

namespace Recommenders {
namespace RWRBased {

enum class NodeType : int { UNDEFINED, USER, ITEM, ETC };                                               // Recommender.cs:4
enum class EdgeType : int { UNDEFINED, LIKE, FRIENDSHIP, FOLLOW, MENTION, AUTHORSHIP, PURCHASE, ETC };   // Recommender.cs:5

struct Node {                                                                                            // Graph.cs:4-17
    long long id = 0;
    NodeType type = NodeType::UNDEFINED;
    Node() {}
    Node(long long id) : id(id) {}
    Node(long long id, NodeType type) : id(id), type(type) {}
};

struct ForwardLink {                                                                                     // Graph.cs:19-35
    int targetNode = 0;
    EdgeType type = EdgeType::UNDEFINED;
    double weight = 0;
    ForwardLink() {}
    ForwardLink(int targetNode, double weight) : targetNode(targetNode), weight(weight) {}
    ForwardLink(int targetNode, EdgeType type, double weight) : targetNode(targetNode), type(type), weight(weight) {}
};

// what the reference's callers can catch
struct KeyNotFoundException : std::runtime_error { using std::runtime_error::runtime_error; };        // Recommender.cs:21, Model.cs:79
struct ArgumentException : std::runtime_error { using std::runtime_error::runtime_error; };           // Graph.cs:86 (buildGraph twice)
struct IndexOutOfRangeException : std::runtime_error { using std::runtime_error::runtime_error; };    // Model.cs:87
struct NotSupportedException : std::runtime_error { using std::runtime_error::runtime_error; };       // Model.run(double), see Model
struct RwrException : std::runtime_error {                                                            // everything else (CUDA, NCCL, ...)
    int code;
    RwrException(int code, const std::string& what) : std::runtime_error(what), code(code) {}
};

// the containers of the reference's signatures, with the members its callers use (DataLoader.cs:60-77, Experiment.cs:123):
// std::map / std::vector underneath, so any standard algorithm works on them as well
template <typename K, typename V>
struct Dictionary : std::map<K, V> {
    void Add(const K& k, const V& v) {
        if (!this->emplace(k, v).second) throw ArgumentException("An item with the same key has already been added");
    }
    bool ContainsKey(const K& k) const { return this->find(k) != this->end(); }
    int Count() const { return (int)this->size(); }
    V& operator[](const K& k) {                      // the indexer's getter: KeyNotFoundException, never an insertion
        auto it = this->find(k);
        if (it == this->end()) throw KeyNotFoundException("The given key was not present in the dictionary");
        return it->second;
    }
};
template <typename T>
struct List : std::vector<T> {
    using std::vector<T>::vector;
    void Add(const T& x) { this->push_back(x); }
    int Count() const { return (int)this->size(); }
};
template <typename K, typename V>
struct KeyValuePair {
    K Key;
    V Value;
    KeyValuePair() : Key(), Value() {}
    KeyValuePair(const K& k, const V& v) : Key(k), Value(v) {}
};

inline void check(int rc) {
    if (rc == RWR_OK) return;
    const std::string msg = rwr_last_error();
    switch (rc) {
        case RWR_E_BADSEED:
        case RWR_E_NOT_BUILT: throw KeyNotFoundException(msg);
        case RWR_E_ALREADY_BUILT: throw ArgumentException(msg);
        case RWR_E_BADINDEX: throw IndexOutOfRangeException(msg);
        default: throw RwrException(rc, msg);
    }
}

class Graph {                                                                                            // Graph.cs:37-94
public:
    // Graph information: the caller's dictionaries, kept by reference and read at buildGraph() like the reference does
    Dictionary<int, Node>& nodes;
    Dictionary<int, List<ForwardLink>>& edges;

    Graph(Dictionary<int, Node>& nodes, Dictionary<int, List<ForwardLink>>& edges, int device = -1)
        : nodes(nodes), edges(edges), device_(device) {}
    Graph(const Graph&) = delete;
    Graph& operator=(const Graph&) = delete;
    ~Graph() { rwr_graph_destroy(h_); }

    void buildGraph() {                                                                                  // Graph.cs:51-88
        if (h_) {                                   // graph.Add(i, ..) on an existing key
            check(rwr_graph_build(h_));
            return;
        }
        const int n = (int)nodes.size();
        std::vector<int64_t> id((size_t)n);
        std::vector<int32_t> type((size_t)n), src, dst, et;
        std::vector<double> w;
        for (int i = 0; i < n; i++) {               // keys are the dense indices 0..N-1 (DataLoader.cs:41, :54)
            auto it = nodes.find(i);
            if (it == nodes.end()) throw KeyNotFoundException("nodes has no entry for index " + std::to_string(i));
            id[(size_t)i] = it->second.id;
            type[(size_t)i] = (int32_t)it->second.type;
            auto e = edges.find(i);                 // `if (edges.ContainsKey(i))`, Graph.cs:55
            if (e == edges.end()) continue;
            for (const ForwardLink& l : e->second) {
                src.push_back(i); dst.push_back(l.targetNode); et.push_back((int32_t)l.type); w.push_back(l.weight);
            }
        }
        rwr_opts o{};
        o.device = device_;
        o.hub_entries = -1;
        o.empty_seed_ok = 1;                        // an `edges` entry that exists but is empty is served; Recommender checks the key itself
        check(rwr_graph_create(n, id.data(), type.data(), (int64_t)src.size(), src.data(), dst.data(), et.data(), w.data(), &o, &h_));
        check(rwr_graph_build(h_));
    }

    int size() { return (int)nodes.size(); }                                                            // Graph.cs:91

    // `graph[i]` (Graph.cs:43): the adjusted forward links of node i; empty for a null (dangling) row
    List<ForwardLink> graph(int i) {
        load_csr();
        List<ForwardLink> row;
        for (int64_t k = row_ptr_[(size_t)i]; k < row_ptr_[(size_t)i + 1]; k++)
            row.Add(ForwardLink(col_[(size_t)k], (EdgeType)etype_[(size_t)k], val_[(size_t)k]));
        return row;
    }

    rwr_graph* handle() {
        if (!h_) throw KeyNotFoundException("buildGraph() has not run (graph.graph[i], Model.cs:79)");
        return h_;
    }

private:
    void load_csr() {
        if (!row_ptr_.empty()) return;
        rwr_graph_info info{};
        check(rwr_graph_get_info(handle(), &info));
        row_ptr_.assign((size_t)info.n_nodes + 1, 0);
        col_.assign((size_t)info.nnz, 0); val_.assign((size_t)info.nnz, 0.0); etype_.assign((size_t)info.nnz, 0);
        check(rwr_graph_get_csr(h_, row_ptr_.data(), col_.data(), val_.data()));
        check(rwr_graph_get_csr_types(h_, etype_.data()));
    }
    rwr_graph* h_ = nullptr;
    int device_;
    std::vector<int64_t> row_ptr_;
    std::vector<int32_t> col_, etype_;
    std::vector<double> val_;
};

class Model {                                                                                            // Model.cs:5-116
public:
    Graph* graph;
    // Model.cs:7.  A caller may overwrite it: the next run starts from the written vector (a warm start).  Detected by
    // comparison with the vector the last run delivered, as a changed `restart` is.
    std::vector<double> rank;
    // Model.cs:9: e_seed, or 1/N everywhere.  A caller may overwrite it: a vector that differs from the constructor's runs
    // as a restart set (its nonzeros, rwr_run_*_restart).  A run after `restart` changed starts from the constructor state:
    // run(int) for the run(int) iterations so far (threshold iterations are not replayed), and run(double) throws
    // NotSupportedException once run(int) has run.
    std::vector<double> restart;
    int nNodes;
    double dampingFactor;
    int nIterations = 0;            // deliverRanks() calls so far

    Model(Graph& graph, double dampingFactor) : graph(&graph), nNodes(graph.size()), dampingFactor(dampingFactor), seed_(-1) {
        rank.assign((size_t)nNodes, 1.0);                                                                // Model.cs:24
        restart.assign((size_t)nNodes, 1.0 / nNodes);                                                    // Model.cs:25
        delivered_ = rank;
    }
    Model(Graph& graph, double dampingFactor, int targetNode)
        : graph(&graph), nNodes(graph.size()), dampingFactor(dampingFactor), seed_(targetNode) {
        rank.assign((size_t)nNodes, 0.0);                                                                // Model.cs:44
        restart.assign((size_t)nNodes, 0.0);                                                             // Model.cs:45-48
        if (targetNode >= 0 && targetNode < nNodes) {
            rank[(size_t)targetNode] = nNodes;
            restart[(size_t)targetNode] = 1.0;
        }
        delivered_ = rank;
    }
    // a C# class variable is a reference: `new Model(graph, c, seed)` with `Graph* graph` reads the same here
    Model(Graph* graph, double dampingFactor) : Model(*graph, dampingFactor) {}
    Model(Graph* graph, double dampingFactor, int targetNode) : Model(*graph, dampingFactor, targetNode) {}
    // the Model owns the result its runs continue from: moved, never copied
    Model(const Model&) = delete;
    Model& operator=(const Model&) = delete;
    Model(Model&& o) noexcept { *this = std::move(o); }
    Model& operator=(Model&& o) noexcept {
        if (this != &o) {
            rwr_result_destroy(res_);
            graph = o.graph; rank = std::move(o.rank); restart = std::move(o.restart); nNodes = o.nNodes;
            dampingFactor = o.dampingFactor; nIterations = o.nIterations; seed_ = o.seed_; total_ = o.total_;
            res_ = o.res_; ran_restart_ = std::move(o.ran_restart_); delivered_ = std::move(o.delivered_);
            o.res_ = nullptr;
        }
        return *this;
    }
    ~Model() { rwr_result_destroy(res_); }

    void run() { run_threshold(0.0); }                                    // Model.cs:52-55: (1 / double.MaxValue) * N, chosen by the library
    void run(double threshold) { run_threshold(threshold); }              // Model.cs:57-66
    void run(int nIterations) {                                           // Model.cs:68-73; successive calls accumulate, as in the reference
        const int n = nIterations > 0 ? nIterations : 0;
        total_ += n;
        if (!res_ && !written()) {
            fresh(total_);
        } else if (live()) {
            write_rank();
            check(rwr_continue_fixed(res_, n));
            fetch();
        } else {
            fresh(total_);
            this->nIterations = total_;
            return;
        }
        this->nIterations += n;
    }

private:
    void run_threshold(double thr) {
        int32_t iters = 0;
        if (live()) {
            write_rank();
            check(rwr_continue_threshold(res_, thr, 0, &iters));
            fetch();
            nIterations += iters;
            return;
        }
        if (total_) throw NotSupportedException("run(double) after run(int) / a changed `restart`: a run from the constructor state "
                                                "would not start from `rank`");
        rwr_result* r = nullptr;
        std::vector<int32_t> nodes;
        std::vector<double> weights;
        if (restart_set(nodes, weights))
            check(rwr_run_threshold_restart(graph->handle(), nodes.data(), weights.data(), (int32_t)nodes.size(), init_kind(), seed_,
                                            dampingFactor, thr, 0, RWR_FP64, &iters, &r));
        else
            check(rwr_run_threshold(graph->handle(), &seed_, 1, dampingFactor, thr, 0, RWR_FP64, &iters, &r));
        own(r);
        nIterations = iters;
    }
    // a run of n_iter iterations from the constructor state becomes the live result
    void fresh(int n_iter) {
        rwr_result* r = nullptr;
        std::vector<int32_t> nodes;
        std::vector<double> weights;
        if (restart_set(nodes, weights))
            check(rwr_run_fixed_restart(graph->handle(), nodes.data(), weights.data(), (int32_t)nodes.size(), init_kind(), seed_,
                                        dampingFactor, n_iter, RWR_FP64, &r));
        else
            check(rwr_run_fixed(graph->handle(), &seed_, 1, dampingFactor, n_iter, RWR_FP64, &r));
        own(r);
    }
    void own(rwr_result* r) {
        rwr_result_destroy(res_);
        res_ = r;
        ran_restart_ = restart;
        fetch();
    }
    // the live result can be continued: `restart` has not changed since it ran (a written rank is written into it first;
    // one written before the first run gets a result of the constructor state to be written into)
    bool live() {
        if (!res_) {
            if (!written()) return false;
            const std::vector<double> w = rank;
            fresh(0);
            rank = w;
            return true;
        }
        return same_bits(restart, ran_restart_);
    }
    bool written() const { return !same_bits(rank, delivered_); }
    void write_rank() {
        if ((int)rank.size() != nNodes) throw ArgumentException("rank must hold one value per node");
        if (written()) check(rwr_set_rank(res_, 0, rank.data()));
    }
    static bool same_bits(const std::vector<double>& a, const std::vector<double>& b) {
        return a.size() == b.size() && (a.empty() || std::memcmp(a.data(), b.data(), a.size() * sizeof(double)) == 0);
    }
    // the nonzeros of `restart` when it differs from the constructor's vector; false: unchanged
    bool restart_set(std::vector<int32_t>& nodes, std::vector<double>& weights) const {
        if ((int)restart.size() != nNodes) throw ArgumentException("restart must hold one weight per node");
        bool same = true;
        for (int i = 0; i < nNodes && same; i++)
            same = restart[(size_t)i] == (seed_ < 0 ? 1.0 / nNodes : (i == seed_ ? 1.0 : 0.0));
        if (same) return false;
        for (int i = 0; i < nNodes; i++)
            if (restart[(size_t)i] != 0.0) { nodes.push_back(i); weights.push_back(restart[(size_t)i]); }
        return true;
    }
    int32_t init_kind() const { return seed_ < 0 ? RWR_INIT_UNIFORM : RWR_INIT_NODE; }
    void fetch() {
        rank.resize((size_t)nNodes);
        check(rwr_scores(res_, 0, rank.data()));
        delivered_ = rank;
    }
    int32_t seed_ = -1;
    int total_ = 0;                 // run(int) iterations so far: the count a run after `restart` changed replays
    rwr_result* res_ = nullptr;
    std::vector<double> ran_restart_;   // `restart` as it was when res_ ran
    std::vector<double> delivered_;     // `rank` as the last run delivered it
};

class Recommender {                                                                                      // Recommender.cs:7-52
public:
    Recommender(Graph& graph) : graph(graph) {}
    Recommender(Graph* graph) : graph(*graph) {}

    List<KeyValuePair<long long, double>> Recommendation(int idxTargetUser, float dampingFactor, int nIteration) {
        require_entry(idxTargetUser);
        rwr_result* r = nullptr;
        const int32_t seed = idxTargetUser;
        check(rwr_run_fixed(graph.handle(), &seed, 1, (double)dampingFactor, nIteration, RWR_FP64, &r));     // float -> double, :16
        const size_t cap = (size_t)graph.size();
        std::vector<int64_t> ids(cap ? cap : 1);
        std::vector<double> scores(cap ? cap : 1);
        int64_t count = 0;
        const int rc = rwr_rank_all(r, 0, ids.data(), scores.data(), (int64_t)cap, &count);
        rwr_result_destroy(r);
        check(rc);
        List<KeyValuePair<long long, double>> recommendation;
        recommendation.reserve((size_t)count);
        for (int64_t i = 0; i < count; i++) recommendation.Add(KeyValuePair<long long, double>((long long)ids[(size_t)i], scores[(size_t)i]));
        return recommendation;
    }

    List<KeyValuePair<long long, double>> Recommendation(int idxTargetUser, float dampingFactor, int nIteration, int topN) {
        if (topN <= 0 || topN > 16) {               // `Count == topN` never fires for topN <= 0 (Recommender.cs:47): the whole list
            auto recommendation = Recommendation(idxTargetUser, dampingFactor, nIteration);
            if (topN > 0 && (size_t)topN < recommendation.size()) recommendation.resize((size_t)topN);
            return recommendation;
        }
        require_entry(idxTargetUser);
        const int32_t seed = idxTargetUser;
        int64_t ids[16];
        double scores[16];
        int32_t count = 0;
        check(rwr_recommend(graph.handle(), &seed, 1, (double)dampingFactor, nIteration, RWR_FP64, topN, ids, scores, &count, nullptr));
        List<KeyValuePair<long long, double>> topNRecommendation;
        for (int i = 0; i < count; i++) topNRecommendation.Add(KeyValuePair<long long, double>((long long)ids[i], scores[i]));
        return topNRecommendation;
    }

    // Not in the reference: the ranking for a weighted node set (a group of users, a session of items) from a Model whose
    // `restart` is `weights` at `nodes`, initial rank fl(N * weight).  Candidates: the ITEM nodes none of the listed nodes
    // has liked (Recommender.cs:20-24 for each), (score desc, id desc); topN > 0 keeps the first topN.
    List<KeyValuePair<long long, double>> RecommendationForSet(const std::vector<int>& nodes, const std::vector<double>& weights,
                                                               float dampingFactor, int nIteration, int topN = 0) {
        if (nodes.size() != weights.size()) throw ArgumentException("one weight per node");
        const std::vector<int32_t> n32(nodes.begin(), nodes.end());
        rwr_result* r = nullptr;
        check(rwr_run_fixed_restart(graph.handle(), n32.data(), weights.data(), (int32_t)n32.size(), RWR_INIT_RESTART, 0,
                                    (double)dampingFactor, nIteration, RWR_FP64, &r));
        const size_t cap = topN > 0 ? (size_t)topN : (size_t)graph.size();
        std::vector<int64_t> ids(cap ? cap : 1);
        std::vector<double> scores(cap ? cap : 1);
        int64_t count = 0;
        const int rc = rwr_rank_all(r, 0, ids.data(), scores.data(), (int64_t)cap, &count);
        rwr_result_destroy(r);
        check(rc);
        if ((size_t)count > cap) count = (int64_t)cap;
        List<KeyValuePair<long long, double>> recommendation;
        for (int64_t i = 0; i < count; i++) recommendation.Add(KeyValuePair<long long, double>((long long)ids[(size_t)i], scores[(size_t)i]));
        return recommendation;
    }

private:
    void require_entry(int idx) {                   // `graph.edges[idxTargetUser]`, Recommender.cs:21
        if (graph.edges.find(idx) == graph.edges.end())
            throw KeyNotFoundException("edges has no entry for node " + std::to_string(idx) + " (Recommender.cs:21)");
    }
    Graph& graph;
};

}  // namespace RWRBased
}  // namespace Recommenders
