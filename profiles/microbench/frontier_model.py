#!/usr/bin/env python
"""frontier_model.py -- CPU MODEL (not a measurement).

How sparse are the first iterations of a single-seed run on the C2 graph?  Rebuilds the graph with the CPU oracle's
generator and the label order of graph.cu (wavefront_model.relabel), takes bench.py's timed seeds, and prints per
iteration k (x_k computed from x_{k-1}):
    frontier    nonzero entries of x_{k-1} (the sources that contribute anything)
    push_links  their out-links, as a fraction of all links (what a push from the frontier reads)
    act_rows    rows of W^T with at least one nonzero source, plus the seed (the rows a sparse iteration writes)
    pull_links  the in-links of those rows, as a fraction of the edge stream (what a pull restricted to them reads)
    stages% / tiles%  256-link stages / 4096-link tiles of the edge stream holding a link of an active row

    python profiles/microbench/frontier_model.py [scale]        (1.0 = C2, ~4 min and ~20 GB of host memory)
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for d in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "profiles", "microbench")):
    sys.path.insert(0, d)
import oracle as O                                      # noqa: E402
from wavefront_model import relabel                     # noqa: E402
from bench import pick_seeds, scaled_spec               # noqa: E402

scale = float(sys.argv[1]) if len(sys.argv) > 1 else 1.0
spec = scaled_spec(scale)
t0 = time.time()
g = O.synth_generate(spec)
n = len(g["node_id"]); src = g["src"].astype(np.int64); dst = g["dst"].astype(np.int64)
E = len(src)
print(f"n={n} E={E} ({time.time()-t0:.0f}s)", flush=True)
raw_deg = np.bincount(src, minlength=n)
new_of_old, n_hot, deg = relabel(n, src, dst)
# stream offsets per row (internal label), one padding link for rows without in-links
indeg_lab = np.bincount(new_of_old[dst], minlength=n)
ptr2 = np.zeros(n + 1, np.int64); np.cumsum(np.maximum(indeg_lab, 1), out=ptr2[1:])
Es = int(ptr2[-1])
n_st = -(-Es // 256)
seeds = pick_seeds(raw_deg, spec["n_users"], 26)[3:13]      # bench.py: warm-up 3, then the timed steps
for seed in seeds[:4]:
    nz = np.zeros(n, bool); nz[seed] = True
    print(f"seed {seed} (outdeg {raw_deg[seed]})")
    print(" k  frontier  push_links  act_rows  pull_links  stages%  tiles%")
    for k in range(1, 9):
        fmask = nz[src]
        push = int(fmask.sum())
        act = np.zeros(n, bool); act[dst[fmask]] = True; act[seed] = True
        rows = new_of_old[np.flatnonzero(act)]
        pull = int(np.maximum(indeg_lab[rows], 1).sum())
        d = np.zeros(n_st + 1, np.int64)
        np.add.at(d, ptr2[rows] // 256, 1); np.add.at(d, (ptr2[rows + 1] - 1) // 256 + 1, -1)
        st = np.cumsum(d)[:n_st] > 0
        ti = st[: (n_st // 16) * 16].reshape(-1, 16).any(1)
        print(f"{k:2d} {int(nz.sum()):9d} {push/E:10.4f} {act.sum():9d} {pull/Es:10.4f} {100*st.mean():7.2f} {100*ti.mean():7.2f}", flush=True)
        nz = act & (deg > 0)        # dangling rows (no out-links) keep their rank but gather nothing: inv = 0
        if pull / Es > 0.999:
            break
