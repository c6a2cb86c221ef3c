#!/usr/bin/env python
"""resume_probe.py -- what continuing a result on the device (rwr_continue_fixed / rwr_continue_threshold / rwr_set_rank)
costs and saves, on the C2 graph (bench.py's generator and timed seeds), FP64, one seed:
  (a) run(20) against run(10) + continue_fixed(10): a continuation launches one init kernel (k_init_resume) and then its
      iterations kernel by kernel, without the replay of a captured iteration graph;
  (b) 20 deliverRanks() / updateRanks() pairs through the Python Model (host clock around the loop) -- run it once with this
      tree and once with the tree of the parent commit on PYTHONPATH (`--pairs-only`) to compare;
  (c) warm start: 1 000 users held out (fold 0 of 5), then a threshold run of 1e-9 * N from the constructor state against
      one from the ranks of the full graph (rwr_set_rank): iterations and loop milliseconds.
`loop` = rwr_run_info.iterate_ms (CUDA events on the stream), `call` = host clock around the call, which ends in a device
synchronise.  Median of REPS calls after one warm-up call.  The card's name and power limit are read in the same process.

    python profiles/microbench/resume_probe.py [--pairs-only]
"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.append(ROOT)
import recommendersystems_b200 as rs                                         # noqa: E402
from recommendersystems_b200.rwr import run_fixed                             # noqa: E402
from bench import C2_SPEC, C_FLOAT, pick_seeds                                # noqa: E402

REPS = 7
c = rs.widen_float(C_FLOAT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def median_ms(fn):
    fn()
    t = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t))


def graph(hold=None):
    g = rs.Graph.synthetic(C2_SPEC)
    if hold is not None:
        g.hold_out(hold, 5, 0)
    g.buildGraph()
    return g


def main():
    pairs_only = "--pairs-only" in sys.argv
    print(f"card: {card()}")
    print(f"package: {os.path.dirname(rs.__file__)}")
    g = graph()
    n = g.size()
    seed = int(pick_seeds(g.degrees(raw=True), C2_SPEC["n_users"], 1)[0])

    # (b) the step methods
    def pairs():
        m = rs.Model(g, c, seed)
        for _ in range(20):
            m.deliverRanks()
            m.updateRanks()
        return m.rank
    print(f"(b) 20 deliverRanks/updateRanks pairs, seed {seed}: {median_ms(pairs):.2f} ms (host clock, median of {REPS})")
    if pairs_only:
        return

    # (a) a continuation against one run
    r = run_fixed(g, [seed], c, 20)
    r.rerun([seed], c, 20)                             # the second run with this key captures the iteration graph
    loop20, loop10 = [], []

    def whole():
        r.rerun([seed], c, 20)
        loop20.append(r.info().iterate_ms)

    def halves():
        r.rerun([seed], c, 10)
        a = r.info().iterate_ms
        r.continue_fixed(10)
        loop10.append(a + r.info().iterate_ms)
    w = median_ms(whole)
    h = median_ms(halves)
    same = np.array_equal(r.scores(0).view(np.uint64), run_fixed(g, [seed], c, 20).scores(0).view(np.uint64))
    print(f"(a) run(20): call {w:.3f} ms, loop {np.median(loop20):.3f} ms | run(10) + continue_fixed(10): call {h:.3f} ms, "
          f"loop {np.median(loop10):.3f} ms | continuation launches {r.info().kernel_launches} | bit-identical: {same}")
    full = run_fixed(g, [seed], c, 30).scores(0)
    r.close()
    g.close()

    # (c) warm start after a hold-out of 1 000 users
    users = [u for u in range(1000, 2000) if u != seed]
    g2 = graph(users)
    thr = 1e-9 * n
    cold_it, cold_ms, warm_it, warm_ms = [], [], [], []
    for _ in range(REPS):
        rc, it = rs.rwr.run_threshold(g2, [seed], c, thr)
        cold_it.append(int(it[0]))
        cold_ms.append(rc.info().iterate_ms)
        rc.close()
        rw = run_fixed(g2, [seed], c, 0)
        rw.set_rank(0, full)
        warm_it.append(int(rw.continue_threshold(thr)[0]))
        warm_ms.append(rw.info().iterate_ms)
        rw.close()
    print(f"(c) threshold {thr:.3e} after a hold-out of {len(users)} users: from the constructor {cold_it[0]} iterations, "
          f"loop {np.median(cold_ms):.3f} ms | from the full graph's run(30) ranks {warm_it[0]} iterations, "
          f"loop {np.median(warm_ms):.3f} ms")
    g2.close()


if __name__ == "__main__":
    main()
