// Model.cs -- drop-in for Recommenders/RWRBased/Model.cs: constructors, run() / run(double) / run(int), the public
// fields rank / nextRank / restart and the three step methods.  deliverRanks / updateRanks / checkConvergence run on
// the device inside the run* calls; called one by one (nobody in the reference does) they are served by re-running the
// device loop from the constructor state, which costs O(step) per call but keeps the surface.  A caller who overwrites
// `restart` (Model.cs:9 is a public field) gets a walk that restarts over that weighted node set: every run path passes its
// nonzeros to rwr_run_*_restart, with the constructor's initial rank.  Source only.
using System;
using System.Collections.Generic;
using Recommenders.RWRBased.Native;

namespace Recommenders.RWRBased {
    public class Model : IDisposable {
        public Graph graph;
        public int nNodes;
        public double dampingFactor;
        public int nIterations;                 // deliverRanks() calls performed so far
        public double[] nextRank;               // Model.cs:8: zero except between deliverRanks() and updateRanks()
        public double[] restart;                // Model.cs:9: e_seed, or 1/N everywhere (uniform constructor); writable
        readonly int seed;                      // -1: uniform restart (Model.cs:14-31)
        ResultHandle result;
        double[] rankCache;

        public Model(Graph graph, double dampingFactor) : this(graph, dampingFactor, -1) { }
        public Model(Graph graph, double dampingFactor, int targetNode) {
            this.graph = graph; this.nNodes = graph.size(); this.dampingFactor = dampingFactor; this.seed = targetNode;
            nextRank = new double[nNodes];
            restart = new double[nNodes];
            for (int i = 0; i < nNodes; i++) restart[i] = seed < 0 ? 1.0 / nNodes : (i == seed ? 1.0 : 0.0);   // Model.cs:25, :45-48
        }

        public void run() { runThreshold(0.0); }                    // thr <= 0 selects (1/double.MaxValue) * N, Model.cs:53
        public void run(double threshold) { runThreshold(threshold); }
        public void run(int nIterations) {                          // Model.cs:68-73; successive calls accumulate
            runFixed(this.nIterations + Math.Max(nIterations, 0));
        }
        // the nonzeros of `restart` when the caller changed it from the constructor's vector; false: unchanged
        bool restartSet(out int[] nodes, out double[] weights) {
            nodes = null; weights = null;
            if (restart == null || restart.Length != nNodes) throw new ArgumentException("restart must hold one weight per node");
            bool same = true;
            for (int i = 0; i < nNodes && same; i++) same = restart[i] == (seed < 0 ? 1.0 / nNodes : (i == seed ? 1.0 : 0.0));
            if (same) return false;
            var n = new List<int>(); var w = new List<double>();
            for (int i = 0; i < nNodes; i++) if (restart[i] != 0.0) { n.Add(i); w.Add(restart[i]); }
            nodes = n.ToArray(); weights = w.ToArray();
            return true;
        }
        int initKind { get { return seed < 0 ? RwrNative.INIT_UNIFORM : RwrNative.INIT_NODE; } }

        void runFixedInto(int total, out ResultHandle res) {
            int[] nodes; double[] weights;
            if (restartSet(out nodes, out weights))
                RwrNative.Check(RwrNative.rwr_run_fixed_restart(graph.handle, nodes, weights, nodes.Length, initKind, seed, dampingFactor,
                                                                total, RwrNative.FP64, out res));
            else
                RwrNative.Check(RwrNative.rwr_run_fixed(graph.handle, new[] { seed }, 1, dampingFactor, total, RwrNative.FP64, out res));
        }
        void runFixed(int total) {
            graph.RequireBuilt();
            Release();
            runFixedInto(total, out result);
            nIterations = total;
        }
        void runThreshold(double thr) {
            graph.RequireBuilt();
            if (nIterations != 0) throw new NotSupportedException("run(threshold) after run(int) / deliverRanks() on the same Model");
            Release();
            var iters = new int[1];
            int[] nodes; double[] weights;
            if (restartSet(out nodes, out weights))
                RwrNative.Check(RwrNative.rwr_run_threshold_restart(graph.handle, nodes, weights, nodes.Length, initKind, seed, dampingFactor,
                                                                    thr, 0, RwrNative.FP64, iters, out result));
            else
                RwrNative.Check(RwrNative.rwr_run_threshold(graph.handle, new[] { seed }, 1, dampingFactor, thr, 0, RwrNative.FP64, iters, out result));
            nIterations = iters[0];
        }

        // Model.cs:76-100: nextRank <- one more iteration from `rank`
        public void deliverRanks() {
            graph.RequireBuilt();
            ResultHandle next;
            runFixedInto(nIterations + 1, out next);
            using (next) RwrNative.Check(RwrNative.rwr_scores(next, 0, nextRank));
        }
        // Model.cs:103-108: rank <- nextRank, nextRank <- 0
        public void updateRanks() {
            rankCache = (double[])nextRank.Clone();
            Array.Clear(nextRank, 0, nNodes);
            nIterations += 1;
            if (result != null) { result.Dispose(); result = null; }
        }
        // Model.cs:110-115: sequential sum of |rank - nextRank|, strict `<`
        public bool checkConvergence(double threshold) {
            double diff = 0;
            double[] r = rank;
            for (int i = 0; i < nNodes; i++) diff += Math.Abs(r[i] - nextRank[i]);
            return diff < threshold;
        }

        public double[] rank {
            get {
                if (rankCache != null) return rankCache;
                var r = new double[nNodes];
                if (result == null) {               // constructor state, Model.cs:24 / :44
                    for (int i = 0; i < nNodes; i++) r[i] = seed < 0 ? 1.0 : (i == seed ? nNodes : 0.0);
                    return rankCache = r;
                }
                RwrNative.Check(RwrNative.rwr_scores(result, 0, r));
                return rankCache = r;
            }
        }

        void Release() { rankCache = null; if (result != null) { result.Dispose(); result = null; } }
        public void Dispose() { Release(); }
    }
}
