// Recommender.cs -- drop-in for Recommenders/RWRBased/Recommender.cs: the two Recommendation overloads consumed by
// TweetRecommender/Experiment.cs:109 and :121-128.  `float dampingFactor` is widened to double HERE, exactly as the
// managed code does at Recommender.cs:16 (0.15f -> 0.15000000596046448).  Source only; see INTEGRATION.md.
using System;
using System.Collections.Generic;
using Recommenders.RWRBased.Native;

namespace Recommenders.RWRBased {
    public enum NodeType { UNDEFINED, USER, ITEM, ETC }
    public enum EdgeType { UNDEFINED, LIKE, FRIENDSHIP, FOLLOW, MENTION, AUTHORSHIP, PURCHASE, ETC }

    public class Recommender {
        readonly Graph graph;
        public Recommender(Graph graph) { this.graph = graph; }

        // Full ranking: every ITEM node the user has not liked, (score desc, id desc).
        public List<KeyValuePair<long, double>> Recommendation(int idxTargetUser, float dampingFactor, int nIteration) {
            double c = dampingFactor;
            graph.RequireBuilt();
            graph.RequireEdgesEntry(idxTargetUser);
            ResultHandle res;
            RwrNative.Check(RwrNative.rwr_run_fixed(graph.handle, new[] { idxTargetUser }, 1, c, nIteration, RwrNative.FP64, out res));
            using (res) {
                int n = graph.size();
                var ids = new long[n]; var scores = new double[n];
                long count;
                RwrNative.Check(RwrNative.rwr_rank_all(res, 0, ids, scores, n, out count));
                var list = new List<KeyValuePair<long, double>>((int)count);
                for (long i = 0; i < count; i++) list.Add(new KeyValuePair<long, double>(ids[i], scores[i]));
                return list;
            }
        }

        // First topN of the ranking; the fused request path returns only the k best pairs from the device.
        public List<KeyValuePair<long, double>> Recommendation(int idxTargetUser, float dampingFactor, int nIteration, int topN) {
            if (topN <= 0 || topN > 16) {
                var all = Recommendation(idxTargetUser, dampingFactor, nIteration);
                return (topN > 0 && topN < all.Count) ? all.GetRange(0, topN) : all;
            }
            double c = dampingFactor;
            graph.RequireBuilt();
            graph.RequireEdgesEntry(idxTargetUser);
            var ids = new long[topN]; var scores = new double[topN]; var counts = new int[1];
            RwrRunInfo info;
            RwrNative.Check(RwrNative.rwr_recommend(graph.handle, new[] { idxTargetUser }, 1, c, nIteration, RwrNative.FP64, topN, ids,
                                                    scores, counts, out info));
            var list = new List<KeyValuePair<long, double>>(counts[0]);
            for (int i = 0; i < counts[0]; i++) list.Add(new KeyValuePair<long, double>(ids[i], scores[i]));
            return list;
        }

        // Not in the reference: the ranking for a weighted node set -- a group of users, a session of items -- from a Model whose
        // `restart` is `weights` at `nodes` (personalized PageRank with a preference vector), initial rank fl(N * weight).  The
        // candidates are the ITEM nodes none of the listed nodes has liked (Recommender.cs:20-24 for each), (score desc, id desc);
        // topN > 0 keeps the first topN.
        public List<KeyValuePair<long, double>> RecommendationForSet(int[] nodes, double[] weights, float dampingFactor, int nIteration,
                                                                     int topN = 0) {
            double c = dampingFactor;
            graph.RequireBuilt();
            if (nodes == null || weights == null || nodes.Length != weights.Length) throw new ArgumentException("one weight per node");
            ResultHandle res;
            RwrNative.Check(RwrNative.rwr_run_fixed_restart(graph.handle, nodes, weights, nodes.Length, RwrNative.INIT_RESTART, 0, c,
                                                            nIteration, RwrNative.FP64, out res));
            using (res) {
                int n = graph.size();
                long cap = topN > 0 ? topN : n;
                var ids = new long[cap]; var scores = new double[cap];
                long count;
                RwrNative.Check(RwrNative.rwr_rank_all(res, 0, ids, scores, cap, out count));
                long m = Math.Min(count, cap);
                var list = new List<KeyValuePair<long, double>>((int)m);
                for (long i = 0; i < m; i++) list.Add(new KeyValuePair<long, double>(ids[i], scores[i]));
                return list;
            }
        }

        // Not in the reference: n seeds at once through the SpMM tiles (Experiment-style evaluation of many users).
        public List<KeyValuePair<long, double>>[] RecommendationBatch(int[] users, float dampingFactor, int nIteration, int topN) {
            double c = dampingFactor;
            graph.RequireBuilt();
            foreach (int u in users) graph.RequireEdgesEntry(u);
            var ids = new long[users.Length * topN]; var scores = new double[users.Length * topN]; var counts = new int[users.Length];
            RwrRunInfo info;
            RwrNative.Check(RwrNative.rwr_recommend(graph.handle, users, users.Length, c, nIteration, RwrNative.FP64, topN, ids, scores,
                                                    counts, out info));
            var outp = new List<KeyValuePair<long, double>>[users.Length];
            for (int u = 0; u < users.Length; u++) {
                outp[u] = new List<KeyValuePair<long, double>>(counts[u]);
                for (int i = 0; i < counts[u]; i++) outp[u].Add(new KeyValuePair<long, double>(ids[u * topN + i], scores[u * topN + i]));
            }
            return outp;
        }
    }
}
