#!/usr/bin/env python
"""frontier_probe.py -- what the sparse prefix of a single-seed run (frontier.cu) costs and saves.

On the C2 graph (bench.py's generator and timed seeds), with CUDA events around Model.rerun:
  * a 20-iteration run with the frontier kernels and with RWR_NO_FRONTIER=1 (the dense path), replayed iteration graph
    as in bench.py;
  * the first two iterations: runs of 2 and 3 iterations (both replayed graphs), both ways.  d = t(3) - t(2) of the
    dense path is one dense iteration; t(2) of the sparse path minus (t(2) - 2 d) of the dense one is what the two sparse
    iterations cost together;
  * the per-iteration split, in a child process with RWR_NO_GRAPH=1 so that every length launches kernel by kernel:
    t(k) - t(k-1) for k = 1, 2, 3, both ways, with the push links (raw links of the frontier) of each iteration;
  * the budget sweep: the 20-iteration run with RWR_FRONTIER_BUDGET = E/4096 ... E/4;
  * the size floor: smaller graphs of the same generator, the 20-iteration run forced sparse (budget E/64) against dense.

    python profiles/microbench/frontier_probe.py [scale] [--fp32] [--floor]
"""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch                                                    # noqa: E402
import recommendersystems_b200 as rs                            # noqa: E402
from recommendersystems_b200.rwr import run_fixed               # noqa: E402
from bench import C_FLOAT, pick_seeds, scaled_spec              # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
scale = float(args[0]) if args else 1.0
prec = rs.FP32 if "fp32" in sys.argv else rs.FP64
split_child = "--split" in sys.argv
floor_only = "--floor" in sys.argv          # the size floor alone
REPS = 5
c = rs.widen_float(C_FLOAT)


def build(sc):
    spec = scaled_spec(sc)
    g = rs.Graph.synthetic(spec, stream=torch.cuda.current_stream().cuda_stream)
    g.buildGraph()
    raw_deg = g.degrees(raw=True)
    return g, raw_deg, [int(s) for s in pick_seeds(raw_deg, spec["n_users"], 26)[3:11]]


def set_env(dense=False, budget=None):
    os.environ.pop("RWR_NO_FRONTIER", None)
    os.environ.pop("RWR_FRONTIER_BUDGET", None)
    if dense:
        os.environ["RWR_NO_FRONTIER"] = "1"
    if budget is not None:
        os.environ["RWR_FRONTIER_BUDGET"] = str(budget)


def time_runs(g, n_iter, seed_list):
    """ms per run (median over REPS passes) for each seed, one Model object, warmed up (graph captured when graphable)"""
    m = run_fixed(g, [seed_list[0]], c, n_iter, prec)
    m.rerun([seed_list[0]], c, n_iter)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    res = []
    for s in seed_list:
        t = []
        for _ in range(REPS):
            torch.cuda.synchronize()
            e0.record()
            m.rerun([s], c, n_iter)
            e1.record()
            torch.cuda.synchronize()
            t.append(e0.elapsed_time(e1))
        res.append(float(np.median(t)))
    m.close()
    return res


def size_floor():
    print("\nsize floor: smaller graphs of the generator, 20-iteration run, replayed graph, median over the seeds, ms")
    for sc in (0.005, 0.02, 0.05, 0.1, 0.16, 0.3):
        gs, _, ss = build(sc * scale)
        e = gs.info().nnz
        set_env(dense=True)
        td = float(np.median(time_runs(gs, 20, ss)))
        set_env(budget=e // 64)
        tf = float(np.median(time_runs(gs, 20, ss)))
        print(f"  scale {sc * scale:<6g} E = {e:10d}: dense {td:.3f}  frontier (budget E/64) {tf:.3f}", flush=True)
        gs.close()
    set_env()


if floor_only:
    size_floor()
    sys.exit(0)

g, raw_deg, seeds = build(scale)
info = g.info()
E = info.nnz

if split_child:
    # kernel by kernel for every length (RWR_NO_GRAPH=1 is set by the parent)
    links = g.export_links()
    order = np.argsort(links["src"], kind="stable")
    dst_sorted = links["dst"][order]
    ptr = np.zeros(info.n_nodes + 1, np.int64)
    np.cumsum(np.bincount(links["src"], minlength=info.n_nodes), out=ptr[1:])
    del links, order

    def push_links(seed, k_max=3):
        """raw out-links of the frontier of iterations 1..k_max"""
        out, front = [], np.array([seed])
        act = np.zeros(info.n_nodes, bool)
        for _ in range(k_max):
            front = front[raw_deg[front] > 0]
            out.append(int(raw_deg[front].sum()))
            tg = np.concatenate([dst_sorted[ptr[f]:ptr[f + 1]] for f in front]) if len(front) else np.zeros(0, np.int64)
            act[tg] = True
            act[seed] = True
            front = np.flatnonzero(act)
        return out

    t = {}
    for dense in (False, True):
        set_env(dense=dense)
        t[dense] = [time_runs(g, k, seeds[:4]) for k in (1, 2, 3)]
    print("per iteration, kernel by kernel (RWR_NO_GRAPH=1), ms: t(k) - t(k-1) with the frontier kernels / dense;"
          " t(0) = set-up of the run, not subtracted from iteration 1")
    for i, s in enumerate(seeds[:4]):
        pl = push_links(s)
        row = []
        for k in range(3):
            f = t[False][k][i] - (t[False][k - 1][i] if k else 0.0)
            d = t[True][k][i] - (t[True][k - 1][i] if k else 0.0)
            row.append(f"it{k + 1}: {f:.3f} / {d:.3f} ({pl[k]} links)")
        print(f"{s:8d}  " + "   ".join(row), flush=True)
    sys.exit(0)

print(f"{torch.cuda.get_device_name()}  n={info.n_nodes} E={E}  precision={'fp32' if prec == rs.FP32 else 'fp64'}", flush=True)
try:
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
except OSError:
    pass

set_env(dense=True)
dense20 = time_runs(g, 20, seeds)
set_env()
sparse20 = time_runs(g, 20, seeds)
print("\n20-iteration run, replayed graph, ms (median of %d)" % REPS)
print(" seed      dense   frontier   saved")
for s, d, f in zip(seeds, dense20, sparse20):
    print(f"{s:8d} {d:9.3f} {f:9.3f} {d - f:8.3f}")
print(f"  median {np.median(dense20):9.3f} {np.median(sparse20):9.3f} {np.median(dense20) - np.median(sparse20):8.3f}"
      f"  ({100 * (1 - np.median(sparse20) / np.median(dense20)):.1f} %)", flush=True)

print("\nfirst two iterations, replayed graph, ms: t(2), t(3) dense / frontier; d = dense t(3) - t(2);"
      " two sparse iterations = frontier t(2) - (dense t(2) - 2 d)")
tl = {}
for dense in (True, False):
    set_env(dense=dense)
    tl[dense] = [time_runs(g, k, seeds[:4]) for k in (2, 3)]
for i, s in enumerate(seeds[:4]):
    d2, d3, f2, f3 = tl[True][0][i], tl[True][1][i], tl[False][0][i], tl[False][1][i]
    d = d3 - d2
    print(f"{s:8d}  dense {d2:.3f} {d3:.3f}  frontier {f2:.3f} {f3:.3f}  one dense iteration {d:.3f}"
          f"  two sparse iterations {f2 - (d2 - 2 * d):.3f}", flush=True)

env = dict(os.environ, RWR_NO_GRAPH="1")
env.pop("RWR_NO_FRONTIER", None)
env.pop("RWR_FRONTIER_BUDGET", None)
print()
sys.stdout.flush()
subprocess.run([sys.executable, os.path.abspath(__file__), str(scale), "--split"] + (["--fp32"] if prec == rs.FP32 else []),
               env=env, check=True)

print("\nbudget sweep (RWR_FRONTIER_BUDGET), 20-iteration run, replayed graph, median over the seeds, ms")
for div in (4096, 1024, 256, 64, 16, 4):
    set_env(budget=E // div)
    t = time_runs(g, 20, seeds)
    print(f"  E/{div:<5d} = {E // div:10d} links: {np.median(t):.3f}", flush=True)
set_env()
g.close()
size_floor()
