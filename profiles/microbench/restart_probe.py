#!/usr/bin/env python
"""restart_probe.py -- what a restart-set run (rwr_run_fixed_restart) costs next to a seeded run.

On the C2 graph (bench.py's generator and timed seeds), 20-iteration runs in FP64 and FP32:
  * seeded   -- rwr_run_fixed of one seed with RWR_NO_FRONTIER=1: the dense path, like for like (a restart-set run never
                pushes from a frontier), as a fresh call and as a Model re-run; after the warm-up both replay the captured
                iteration graph (RWR_NO_GRAPH=1: both launch kernel by kernel);
  * set m    -- rwr_run_fixed_restart of m = 1, 16, 1 000 and 100 000 nodes (the hub, the timed seeds, then random nodes),
                weights 1/m, init RESTART.  Always kernel by kernel: restart-set runs have no iteration graph.
For each: `loop` = device time of the iteration loop (rwr_run_info.iterate_ms, CUDA events on the stream), `call` = host
clock around the whole call (set-up, upload, validation, result allocation; it ends in a device synchronise).  Median of
REPS calls after one warm-up call.  The card's name and power limit are read in the same process.  With RWR_NO_GRAPH=1 in
the environment (read once per process) the seeded runs launch kernel by kernel too: the difference to a plain run is what
the missing iteration graph costs a restart-set run.

    python profiles/microbench/restart_probe.py [scale]
    RWR_NO_GRAPH=1 python profiles/microbench/restart_probe.py [scale]
"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import recommendersystems_b200 as rs                                         # noqa: E402
from recommendersystems_b200.rwr import run_fixed, run_fixed_restart          # noqa: E402
from bench import C_FLOAT, pick_seeds, scaled_spec                            # noqa: E402

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
REPS = 7
N_ITER = 20
c = rs.widen_float(C_FLOAT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def timed(call):
    """(median loop ms, median call ms) over REPS calls after one warm-up"""
    call().close()
    loop, wall = [], []
    for _ in range(REPS):
        t0 = time.perf_counter()
        r = call()
        r.scores(0)[:1]                       # (scores() synchronises; the call itself already has)
        t1 = time.perf_counter()
        loop.append(r.info().iterate_ms)
        wall.append((t1 - t0) * 1e3)
        r.close()
    return float(np.median(loop)), float(np.median(wall))


def main():
    print(f"card: {card()}")
    print(f"RWR_NO_GRAPH={os.environ.get('RWR_NO_GRAPH', '')!r}: seeded runs " +
          ("kernel by kernel" if os.environ.get("RWR_NO_GRAPH") else "replay their captured iteration graph"))
    spec = scaled_spec(scale)
    g = rs.Graph.synthetic(spec)
    g.buildGraph()
    info = g.info()
    n = info.n_nodes
    raw_deg = g.degrees(raw=True)
    seeds = [int(s) for s in pick_seeds(raw_deg, spec["n_users"], 26)[3:11]]
    print(f"graph: C2 x {scale}: {n} nodes, {info.nnz} links, layout {info.layout}; {N_ITER} iterations, median of {REPS} calls")
    rng = np.random.default_rng(7)
    hub = int(np.argmax(raw_deg))
    pool = list(dict.fromkeys([hub] + seeds + [int(x) for x in rng.choice(n, 120_000, replace=False)]))
    os.environ["RWR_NO_FRONTIER"] = "1"
    for prec, name in ((rs.FP64, "FP64"), (rs.FP32, "FP32")):
        print(f"\n{name}                          loop ms   call ms   loop vs seeded")
        s = seeds[0]
        loop0, wall0 = timed(lambda: run_fixed(g, [s], c, N_ITER, prec))
        print(f"  seeded, fresh call          {loop0:8.3f}  {wall0:8.3f}")
        # a Model re-run replays the captured graph of the whole loop (bench.py's timed path)
        m = run_fixed(g, [s], c, N_ITER, prec)
        m.rerun([s], c, N_ITER)
        lr = []
        for _ in range(REPS):
            m.rerun([s], c, N_ITER)
            lr.append(m.info().iterate_ms)
        m.close()
        loopr = float(np.median(lr))
        print(f"  seeded, replayed graph      {loopr:8.3f}")
        for m_set in (1, 16, 1000, 100_000):
            nodes = pool[:m_set]
            w = np.full(m_set, 1.0 / m_set)
            loop, wall = timed(lambda: run_fixed_restart(g, nodes, w, c, N_ITER, rs.INIT_RESTART, 0, prec))
            print(f"  set of {m_set:6d} nodes        {loop:8.3f}  {wall:8.3f}   {100.0 * (loop / loop0 - 1.0):+6.2f} %")
    os.environ.pop("RWR_NO_FRONTIER")
    g.close()
    print(f"\ncard: {card()}")


if __name__ == "__main__":
    main()
