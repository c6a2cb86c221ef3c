// RwrNative.cs -- P/Invoke bindings of librwr_b200.so (include/rwr_b200.h), one [DllImport] per exported symbol.
// Shipped as source for the maintainers of Recommenders.dll; not compiled in this repository (no C# toolchain here).
// Replaces nothing by itself: Graph.cs / Model.cs / Recommender.cs in this directory forward to it.
using System;
using System.Collections.Generic;
using System.Runtime.InteropServices;

namespace Recommenders.RWRBased.Native {
    public enum RwrStatus {
        OK = 0, E_INVALID = -1, E_BADSEED = -2, E_ALREADY_BUILT = -3, E_BADINDEX = -4, E_NOT_BUILT = -5,
        E_CUDA = -6, E_NCCL = -7, E_OOM = -8, E_UNSUPPORTED = -9
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct RwrOpts {
        public int device, layout, relabel, hub_entries, batch_width, kernel;
        public ulong stream;
        public int hot_min_degree, undefined_type_mask, zero_weight_type_mask, x_blocks, empty_seed_ok, reserved;
        // empty_seed_ok: the managed Graph checks `edges.ContainsKey(seed)` itself (KeyNotFoundException, Recommender.cs:21),
        // so a key that exists with an empty list is served like the reference serves it
        public static RwrOpts Default() { return new RwrOpts { device = -1, hub_entries = -1, empty_seed_ok = 1 }; }
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct RwrSynthSpec {
        public ulong seed;
        public int n_users, n_items, n_third, authorship_per_mille;
        public long n_like, n_friend, n_follow, n_mention;
        public int undefined_per_mille, scramble, p1_byte, reserved;
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct RwrGraphInfo {
        public int n_nodes, built;
        public long n_links_raw, nnz;
        public int n_dangling, layout, relabelled, n_hot, hub_entries_fp64, hub_entries_fp32, n_chunks, max_in_degree, max_out_degree;
        public float build_ms, synth_ms;
        public long device_bytes;
        public int row_begin, row_end, n_ranks, x_blocks;
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct RwrRunInfo {
        public int n_seeds, n_nodes, precision, iterations;
        public double residual;
        public float iterate_ms, total_ms;
        public long kernel_launches;
    }

    public sealed class GraphHandle : SafeHandle {
        public GraphHandle() : base(IntPtr.Zero, true) { }
        public override bool IsInvalid { get { return handle == IntPtr.Zero; } }
        protected override bool ReleaseHandle() { RwrNative.rwr_graph_destroy(handle); return true; }
    }
    public sealed class ResultHandle : SafeHandle {
        public ResultHandle() : base(IntPtr.Zero, true) { }
        public override bool IsInvalid { get { return handle == IntPtr.Zero; } }
        protected override bool ReleaseHandle() { RwrNative.rwr_result_destroy(handle); return true; }
    }

    public static class RwrNative {
        const string Lib = "rwr_b200";          // librwr_b200.so on Linux (mono / .NET probe the lib prefix)
        public const int FP64 = 0, FP32 = 1;

        [DllImport(Lib)] public static extern int rwr_abi_version();
        [DllImport(Lib)] public static extern int rwr_device_count();
        [DllImport(Lib)] static extern IntPtr rwr_last_error();

        [DllImport(Lib)] public static extern int rwr_graph_create(int nNodes, long[] nodeId, int[] nodeType, long nLinks,
            int[] src, int[] dst, int[] etype, double[] w, ref RwrOpts opts, out GraphHandle graph);
        [DllImport(Lib)] public static extern int rwr_synth_create(ref RwrSynthSpec spec, ref RwrOpts opts, out GraphHandle graph);
        [DllImport(Lib)] public static extern int rwr_graph_build(GraphHandle g);
        [DllImport(Lib)] public static extern int rwr_graph_get_info(GraphHandle g, out RwrGraphInfo info);
        [DllImport(Lib)] public static extern int rwr_graph_export_links(GraphHandle g, long[] nodeId, int[] nodeType, int[] src,
            int[] dst, int[] etype, double[] w);
        [DllImport(Lib)] public static extern int rwr_graph_get_csr(GraphHandle g, long[] rowPtr, int[] col, double[] val);
        [DllImport(Lib)] public static extern int rwr_graph_get_csr_types(GraphHandle g, int[] etype);
        [DllImport(Lib)] public static extern int rwr_graph_get_degrees(GraphHandle g, int[] outDegree, int[] rawDegree);
        [DllImport(Lib)] public static extern void rwr_graph_destroy(IntPtr g);

        [DllImport(Lib)] public static extern int rwr_run_fixed(GraphHandle g, int[] seeds, int nSeeds, double c, int nIter,
            int precision, out ResultHandle result);
        [DllImport(Lib)] public static extern int rwr_run_threshold(GraphHandle g, int[] seeds, int nSeeds, double c, double thr,
            int maxIter, int precision, int[] itersOut, out ResultHandle result);
        // a restart set: Model.restart overwritten with weights at nodes (RWR_INIT_*: the initial rank)
        public const int INIT_UNIFORM = 0, INIT_NODE = 1, INIT_RESTART = 2;
        [DllImport(Lib)] public static extern int rwr_run_fixed_restart(GraphHandle g, int[] nodes, double[] weights, int nRestart, int init,
            int initNode, double c, int nIter, int precision, out ResultHandle result);
        [DllImport(Lib)] public static extern int rwr_run_threshold_restart(GraphHandle g, int[] nodes, double[] weights, int nRestart,
            int init, int initNode, double c, double thr, int maxIter, int precision, int[] itersOut, out ResultHandle result);
        [DllImport(Lib)] public static extern int rwr_rerun_fixed(ResultHandle r, int[] seeds, double c, int nIter);
        [DllImport(Lib)] public static extern int rwr_continue_fixed(ResultHandle r, int nIter);
        [DllImport(Lib)] public static extern int rwr_continue_threshold(ResultHandle r, double thr, int maxIter, int[] itersOut);
        [DllImport(Lib)] public static extern int rwr_set_rank(ResultHandle r, int seedSlot, double[] v);
        [DllImport(Lib)] public static extern int rwr_result_get_info(ResultHandle r, out RwrRunInfo info);
        [DllImport(Lib)] public static extern int rwr_scores(ResultHandle r, int seedSlot, double[] outN);
        [DllImport(Lib)] public static extern int rwr_topk(ResultHandle r, int k, long[] outIds, double[] outScores, int[] outCounts);
        [DllImport(Lib)] public static extern int rwr_rank_all(ResultHandle r, int seedSlot, long[] ids, double[] scores, long cap,
            out long count);
        [DllImport(Lib)] public static extern void rwr_result_destroy(IntPtr r);

        [DllImport(Lib)] public static extern int rwr_recommend(GraphHandle g, int[] seeds, int nSeeds, double c, int nIter,
            int precision, int k, long[] outIds, double[] outScores, int[] outCounts, out RwrRunInfo info);
        [DllImport(Lib)] public static extern int rwr_evaluate(long[] rankedIds, long n, long[] testIds, long nTest, out int hits,
            out double avgPrecision);
        // callers of the hot path: Methodology masks (DataLoader.cs:142-219), k-fold hold-out (DataLoader.cs:122-140),
        // hits / average precision of many users (Experiment.cs:121-128)
        [DllImport(Lib)] public static extern int rwr_methodology_masks(int methodology, out int featureMask, out int undefinedTypeMask,
            out int zeroWeightTypeMask);
        [DllImport(Lib)] public static extern int rwr_graph_hold_out(GraphHandle g, int[] users, int nUsers, int nFolds, int fold,
            long[] testPtr, long[] testIds, long cap, out long nTest);
        [DllImport(Lib)] public static extern int rwr_evaluate_users(GraphHandle g, int[] users, int nUsers, long[] testPtr, long[] testIds,
            double c, int nIter, int precision, int k, int[] hits, double[] avgPrecision, int[] hitsAtK, int[] nTestOfUser,
            out RwrRunInfo info);
        [DllImport(Lib)] public static extern int rwr_profile_iteration(GraphHandle g, int seed, double c, int precision, int reps,
            out float spmvMs, out float fixupMs);
        // parity probe (tests): the ranks of the batched request path, out[nSeeds * N] in original labels
        [DllImport(Lib)] public static extern int rwr_probe_tile_ranks(GraphHandle g, int[] seeds, int nSeeds, double c, int nIter,
            int precision, double[] output);

        // row-partitioned mode: one process per GPU; the 128-byte id goes from rank 0 to the other ranks by any channel
        [DllImport(Lib)] public static extern int rwr_comm_unique_id(byte[] id128);
        [DllImport(Lib)] public static extern int rwr_comm_create(int rank, int nRanks, byte[] id128, ref RwrOpts opts, out IntPtr comm);
        [DllImport(Lib)] public static extern void rwr_comm_destroy(IntPtr comm);
        [DllImport(Lib)] public static extern int rwr_synth_create_partitioned(ref RwrSynthSpec spec, ref RwrOpts opts, IntPtr comm,
            out GraphHandle graph);
        [DllImport(Lib)] public static extern int rwr_graph_create_partitioned(int nNodes, long[] nodeId, int[] nodeType, long nLinks,
            int[] src, int[] dst, int[] etype, double[] w, ref RwrOpts opts, IntPtr comm, out GraphHandle graph);

        public static string LastError() { return Marshal.PtrToStringAnsi(rwr_last_error()) ?? ""; }

        // Status codes -> the exception types the managed implementation throws at the cited lines.
        public static void Check(int rc) {
            if (rc == 0) return;
            string msg = LastError();
            switch ((RwrStatus)rc) {
                case RwrStatus.E_BADSEED:                                      // Recommender.cs:21
                case RwrStatus.E_NOT_BUILT: throw new KeyNotFoundException(msg);   // Model.cs:79
                case RwrStatus.E_ALREADY_BUILT: throw new ArgumentException(msg);  // Graph.cs:86 (Dictionary.Add)
                case RwrStatus.E_BADINDEX: throw new IndexOutOfRangeException(msg); // Model.cs:87
                case RwrStatus.E_OOM: throw new OutOfMemoryException(msg);
                default: throw new InvalidOperationException("librwr_b200 error " + rc + ": " + msg);
            }
        }
    }
}
