"""TEST INFRASTRUCTURE ONLY -- the restart-set oracle of tests/test_restart_oracle.py and tests/test_gpu_restart.py.

`RestartOracle(flat)` builds the graph with the CPU oracle (oracle/liboracle.so: Graph.buildGraph, the seeded and uniform
models, the rankings) and adds what the reference does with a caller-written `Model.restart`: the iteration of
tests/restart_oracle.cpp (compiled on first use into a temporary directory) and the ranking of Recommender.cs:19-38 with the
LIKE targets of every listed node excluded."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import oracle as O

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
ITEM, LIKE = 2, 1


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        d = tempfile.mkdtemp(prefix="restart_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "librestart_oracle.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared",
                               "-o", so, os.path.join(_HERE, "restart_oracle.cpp")])
        L = C.CDLL(so)
        vp, i32, i64, f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double
        L.ro_run.argtypes = [i32, vp, vp, vp, f64, i32, i32, vp, vp, i32, i32, i32, f64, i32, i64, vp, vp]
        _LIB = L
    return _LIB


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


class RestartOracle:
    """The CPU oracle's graph (every OracleGraph member is available here) plus restart sets."""

    def __init__(self, flat):
        f = {k: np.asarray(flat[k]) for k in ("node_id", "node_type", "src", "dst", "etype", "w")}
        self.og = O.OracleGraph(f["node_id"].astype(np.int64), f["node_type"].astype(np.int32), f["src"].astype(np.int32),
                                f["dst"].astype(np.int32), f["etype"].astype(np.int32), f["w"].astype(np.float64))
        assert self.og.build() == 0
        self.n = self.og.n
        self.rp, self.col, self.val = (np.ascontiguousarray(a) for a in self.og.csr())
        self.rp = self.rp.astype(np.int64)
        self.col = self.col.astype(np.int32)
        self.val = self.val.astype(np.float64)
        self.src, self.dst, self.etype = (f[k].astype(np.int64) for k in ("src", "dst", "etype"))
        self.node_id, self.node_type = f["node_id"].astype(np.int64), f["node_type"]

    def __getattr__(self, name):
        return getattr(self.og, name)

    def run_restart(self, nodes, weights, init: int, damping: float, n_iter: int | None = None, threshold: float | None = None,
                    default_threshold: bool = False, literal: bool = False, max_iter: int = 0, init_node: int = 0):
        """A Model whose `restart` is `weights` at `nodes`, from the initial rank `init` (0: 1 everywhere, 1: N at init_node,
        2: fl(N * weight)) -> (rank[N], number of deliverRanks calls)."""
        nodes = np.ascontiguousarray(nodes, np.int32)
        weights = np.ascontiguousarray(weights, np.float64)
        rank = np.empty(max(self.n, 1), np.float64)
        iters = C.c_int64()
        if n_iter is not None:
            mode, ni, thr = 0, int(n_iter), 0.0
        elif default_threshold:
            mode, ni, thr = 2, 0, 0.0
        else:
            mode, ni, thr = 1, 0, float(threshold)
        rc = lib().ro_run(self.n, _p(self.rp), _p(self.col), _p(self.val), float(damping), int(init), int(init_node), _p(nodes),
                          _p(weights), len(nodes), mode, ni, thr, int(literal), int(max_iter), _p(rank), C.byref(iters))
        if rc < 0:
            raise ValueError("ro_run: bad argument")
        return rank[:self.n], iters.value

    def rank_scores_set(self, nodes, rank):
        """Recommender.cs:19-38 on `rank`, excluding the targets of the raw LIKE links of every listed node (a node without
        links adds nothing) -> (ids, scores) in (score desc, id desc) order, NaN below every number (Double.CompareTo)."""
        rank = np.asarray(rank, np.float64)
        listed = np.zeros(self.n, bool)
        listed[np.asarray(nodes, np.int64)] = True
        liked = np.zeros(self.n, bool)
        sel = listed[self.src] & (self.etype == LIKE)
        liked[self.dst[sel]] = True
        cand = np.flatnonzero((self.node_type == ITEM) & ~liked)
        sc = rank[cand]
        ids = self.node_id[cand]
        notnan = ~np.isnan(sc)
        order = np.lexsort((ids, np.where(notnan, sc, 0.0), notnan))[::-1]     # all keys descending; ids are distinct
        return ids[order].copy(), sc[order].copy()
