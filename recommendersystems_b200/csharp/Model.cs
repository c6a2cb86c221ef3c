// Model.cs -- drop-in for Recommenders/RWRBased/Model.cs: constructors, run() / run(double) / run(int), the public
// fields rank / nextRank / restart and the three step methods.  The Model keeps its result on the device: run(int) and
// run(double) continue from the rank it holds (rwr_continue_fixed / rwr_continue_threshold; `run(5); run(5)` is `run(10)`
// bit for bit), a caller-written `rank` is written into it first (rwr_set_rank: a warm start), and a deliverRanks() /
// updateRanks() pair is one continued iteration.  A caller who overwrites `restart` (Model.cs:9 is a public field) gets a
// walk that restarts over that weighted node set: a run passes its nonzeros to rwr_run_*_restart; a run after `restart`
// changed starts from the constructor state: run(int) for the run(int) and updateRanks() iterations so far (threshold
// iterations are not replayed), and run(double) throws NotSupportedException once either has run.  Source only.
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
        ResultHandle result;                    // the live result the runs continue from
        double[] rankCache;                     // `rank` as the result holds it (a caller may write into it)
        double[] delivered;                     // a copy of rankCache as read: a difference is a caller-written rank
        double[] ranRestart;                    // `restart` as it was when `result` ran
        double[] beforeDeliver;                 // deliverRanks() advanced `result`: the rank before it
        int total;                              // run(int) and updateRanks() iterations so far: the count a run after `restart` changed replays

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
            graph.RequireBuilt();
            Settle();
            int n = Math.Max(nIterations, 0);
            total += n;
            if (result == null && !Written()) { Fresh(total); this.nIterations = total; return; }
            if (!Live()) { Fresh(total); this.nIterations = total; return; }
            WriteRank();
            RwrNative.Check(RwrNative.rwr_continue_fixed(result, n));
            rankCache = null;
            this.nIterations += n;
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

        void runFixedInto(int nIter, out ResultHandle res) {
            int[] nodes; double[] weights;
            if (restartSet(out nodes, out weights))
                RwrNative.Check(RwrNative.rwr_run_fixed_restart(graph.handle, nodes, weights, nodes.Length, initKind, seed, dampingFactor,
                                                                nIter, RwrNative.FP64, out res));
            else
                RwrNative.Check(RwrNative.rwr_run_fixed(graph.handle, new[] { seed }, 1, dampingFactor, nIter, RwrNative.FP64, out res));
        }
        // a run of nIter iterations from the constructor state becomes the live result
        void Fresh(int nIter) {
            Release();
            runFixedInto(nIter, out result);
            ranRestart = (double[])restart.Clone();
        }
        // the live result can be continued: `restart` has not changed since it ran.  A rank written before the first run gets
        // a result of the constructor state to be written into.
        bool Live() {
            if (result == null) {
                if (!Written()) return false;
                double[] w = rankCache;
                Fresh(0);
                rankCache = w;
                return true;
            }
            if (restart == null || restart.Length != nNodes) return false;      // the run from the constructor state throws
            for (int i = 0; i < nNodes; i++) if (restart[i] != ranRestart[i]) return false;
            return true;
        }
        bool Written() {
            if (rankCache == null) return false;
            if (delivered == null) return true;
            for (int i = 0; i < nNodes; i++)
                if (BitConverter.DoubleToInt64Bits(rankCache[i]) != BitConverter.DoubleToInt64Bits(delivered[i])) return true;
            return false;
        }
        void WriteRank() { if (Written()) RwrNative.Check(RwrNative.rwr_set_rank(result, 0, rankCache)); }
        void runThreshold(double thr) {
            graph.RequireBuilt();
            Settle();
            var iters = new int[1];
            if (Live()) {
                WriteRank();
                RwrNative.Check(RwrNative.rwr_continue_threshold(result, thr, 0, iters));
                rankCache = null;
                nIterations += iters[0];
                return;
            }
            if (total != 0)
                throw new NotSupportedException("run(double) after run(int) / updateRanks() and a changed `restart`: a run from the " +
                                                "constructor state would not start from `rank`");
            Release();
            int[] nodes; double[] weights;
            if (restartSet(out nodes, out weights))
                RwrNative.Check(RwrNative.rwr_run_threshold_restart(graph.handle, nodes, weights, nodes.Length, initKind, seed, dampingFactor,
                                                                    thr, 0, RwrNative.FP64, iters, out result));
            else
                RwrNative.Check(RwrNative.rwr_run_threshold(graph.handle, new[] { seed }, 1, dampingFactor, thr, 0, RwrNative.FP64, iters, out result));
            ranRestart = (double[])restart.Clone();
            nIterations = iters[0];
        }
        // a deliverRanks() without its updateRanks(): `rank` is still the rank before it, put it back
        void Settle() {
            if (beforeDeliver == null) return;
            RwrNative.Check(RwrNative.rwr_set_rank(result, 0, beforeDeliver));
            rankCache = beforeDeliver; delivered = (double[])beforeDeliver.Clone(); beforeDeliver = null;
            Array.Clear(nextRank, 0, nNodes);
        }

        // Model.cs:76-100: nextRank <- one more iteration from `rank`; `rank` is unchanged.  A second call before
        // updateRanks() changes nothing.
        public void deliverRanks() {
            graph.RequireBuilt();
            if (beforeDeliver != null) return;
            if (result == null && !Written()) Fresh(0);
            if (!Live()) {                          // `restart` changed: from the constructor state, O(step) per call
                ResultHandle next;
                runFixedInto(total + 1, out next);
                using (next) RwrNative.Check(RwrNative.rwr_scores(next, 0, nextRank));
                return;
            }
            WriteRank();
            double[] before = (double[])rank.Clone();
            RwrNative.Check(RwrNative.rwr_continue_fixed(result, 1));
            RwrNative.Check(RwrNative.rwr_scores(result, 0, nextRank));
            beforeDeliver = before;
        }
        // Model.cs:103-108: rank <- nextRank, nextRank <- 0
        public void updateRanks() {
            total += 1;
            if (beforeDeliver != null) {
                rankCache = (double[])nextRank.Clone(); delivered = (double[])nextRank.Clone(); beforeDeliver = null;
            } else if (Live()) {
                WriteRank();
                RwrNative.Check(RwrNative.rwr_continue_fixed(result, 1));
                rankCache = null;
            } else {
                Fresh(total);
                nIterations = total - 1;
            }
            Array.Clear(nextRank, 0, nNodes);
            nIterations += 1;
        }
        // Model.cs:110-115: sequential sum of |rank - nextRank|, strict `<`
        public bool checkConvergence(double threshold) {
            double diff = 0;
            double[] r = rank;
            for (int i = 0; i < nNodes; i++) diff += Math.Abs(r[i] - nextRank[i]);
            return diff < threshold;
        }

        // Model.cs:7.  The array is the Model's: a caller may write into it, or assign a new one, and the next run starts from
        // what it holds (a warm start).
        public double[] rank {
            get {
                if (beforeDeliver != null) return beforeDeliver;
                if (rankCache != null) return rankCache;
                var r = new double[nNodes];
                if (result == null) {               // constructor state, Model.cs:24 / :44
                    for (int i = 0; i < nNodes; i++) r[i] = seed < 0 ? 1.0 : (i == seed ? nNodes : 0.0);
                } else {
                    RwrNative.Check(RwrNative.rwr_scores(result, 0, r));
                }
                delivered = (double[])r.Clone();
                return rankCache = r;
            }
            set {
                if (value == null || value.Length != nNodes) throw new ArgumentException("rank must hold one value per node");
                Settle();                           // a pending deliverRanks(): the result goes back to the rank before it
                if (rankCache == null) { var unused = rank; }      // `delivered`: what the result holds
                rankCache = value;
            }
        }

        void Release() { rankCache = null; delivered = null; beforeDeliver = null; if (result != null) { result.Dispose(); result = null; } }
        public void Dispose() { Release(); }
    }
}
